"""`jitter_correction_imagers` -- same signature as the reference's `jitter_correction/jitter_correction.py:14-174`.

Host file-walking driver (SURVEY.md section 8f rank 1): the list of frames is cut into overlapping sublists; every
frame of a sublist is co-aligned with the sublist's first frame -- which, from the second sublist on, is the
CORRECTED file the previous sublist wrote -- and written out with its corrected header. The frames of a sublist share
its reference, so they are searched by one `hdrshift/sequence.py::SequenceAlignment` call (Carrington grid by default,
like the reference, or helioprojective): the reference is read, uploaded and, in the Carrington frame, projected once
per sublist instead of once per frame; every cube, and so every file written, is the one of the per-frame `Alignment`.
Co-alignment of Carrington maps ("initial_carrington") stays one `Alignment` per frame. The chain between sublists is
sequential by construction: all files of a sublist are written before the next sublist reads its reference. The reference's "before the reference frame" loop (`:141-174`) can only ever see the single-element
sublist [0] (`idx_list[idx_list[0]::-1]` with `idx_list[0] == 0`) and would raise a NameError on anything longer;
it is kept as the no-op it is.
"""
from __future__ import annotations

import os
import shutil
import warnings

import numpy as np

from .._compat import timeutil
from ..hdrshift.alignment import Alignment
from ..hdrshift.sequence import SequenceAlignment
from ..utils import Util


def _hms(date_iso):
    """`Time(...).fits[11:19]` with ':' -> '_'"""
    return timeutil.from_seconds(timeutil.to_seconds(date_iso))[11:19].replace(":", "_")


def jitter_correction_imagers(
        list_files_input: list, path_files_output: str,
        lonlims=None, latlims=None, shape=None,
        lag_crval1: np.array = np.arange(-5, 5, 0.1),
        lag_crval2: np.array = np.arange(-5, 5, 0.1),
        lag_cdelt1: np.array = np.arange(0, 1, 1),
        lag_cdelt2: np.array = np.arange(0, 1, 1),
        lag_crota: np.array = np.arange(0, 1, 1),
        sublist_length: int = 10, overlap: int = 1,
        window_files_input: int = -1,
        method_carrington_reprojection: str = "fa",
        unit_lag: str = "arcsec",
        path_figures: str = None, plot_all_figures: bool = False,
        parallelism: bool = True, cpu_count: int = None,
        small_fov_value_max: float = None, small_fov_value_min: float = None,
        alignement_method="carrington"):
    """Same parameters as the reference. Returns the list of `AlignmentResults` in processing order (the reference
    returns None; the files written are the same)."""
    if overlap == 0:
        raise ValueError("number of overlapping images between sublists can not be equal to 0.")
    dates_files_input = []
    for path in list_files_input:
        with Util._fits().open(path) as hdul:
            dates_files_input.append(hdul[window_files_input].header["DATE-AVG"])
    parameter_alignment = {"lag_crval1": lag_crval1, "lag_crval2": lag_crval2, "lag_cdelt1": lag_cdelt1,
                           "lag_cdelt2": lag_cdelt2, "lag_crota": lag_crota}
    kwargs_carrington = {"lonlims": lonlims, "latlims": latlims, "shape": shape}
    idx_list = np.arange(len(list_files_input))
    list_after_ref = idx_list[idx_list[0]:] if len(idx_list) else idx_list
    sublists_after = [list_after_ref[n: n + sublist_length + overlap]
                      for n in range(0, len(list_after_ref), sublist_length)]
    all_results = []
    for ii, list_ in enumerate(sublists_after):
        index_ref = list_[0]
        path_reference = os.path.join(path_files_output, os.path.basename(list_files_input[index_ref]))
        if ii == 0:
            shutil.copyfile(list_files_input[index_ref], path_reference)
        frames = list_[1:]
        if alignement_method in ("carrington", "helioprojective") and len(frames):
            # every frame of the sublist against the one reference: one batched search, reference resident
            seq = SequenceAlignment(path_reference, [list_files_input[i] for i in frames],
                                    large_fov_window=window_files_input, small_fov_window=window_files_input,
                                    small_fov_value_max=small_fov_value_max, small_fov_value_min=small_fov_value_min,
                                    unit_lag=unit_lag, **parameter_alignment)
            if alignement_method == "carrington":
                batch = seq.align_using_carrington(reference_date=dates_files_input[index_ref],
                                                   method_carrington_reprojection=method_carrington_reprojection,
                                                   **kwargs_carrington)
            else:
                batch = seq.align_using_helioprojective()
            for index_to_align, results in zip(frames, batch):
                _plot_correlation(results, path_figures, _hms(dates_files_input[index_to_align]),
                                  _hms(dates_files_input[index_ref]))
                _write_corrected(results, list_files_input[index_to_align], window_files_input, path_files_output)
                all_results.append(results)
            continue
        for index_to_align in frames:
            results = _align_hrieuv_with_hrieuv(
                path_output_figures=path_figures, large_fov_fits_path=path_reference,
                large_fov_window=window_files_input, small_fov_path=list_files_input[index_to_align],
                window_to_align=window_files_input, date_to_align=_hms(dates_files_input[index_to_align]),
                parameter_alignment=parameter_alignment, cpu_count=cpu_count, do_plot_figure=plot_all_figures,
                method_carrington_reprojection=method_carrington_reprojection,
                reference_date=dates_files_input[index_ref], parallelism=parallelism,
                alignement_method=alignement_method, small_fov_value_max=small_fov_value_max,
                small_fov_value_min=small_fov_value_min, unit_lag=unit_lag, **kwargs_carrington)
            _write_corrected(results, list_files_input[index_to_align], window_files_input, path_files_output)
            all_results.append(results)
    return all_results


def _align_hrieuv_with_hrieuv(large_fov_fits_path: str, large_fov_window, small_fov_path: str,
                              parameter_alignment: dict, date_to_align, cpu_count=30, window_to_align=3,
                              do_plot_figure=False, parallelism=True, lonlims=None, latlims=None, shape=None,
                              unit_lag="arcsec", reference_date=None, small_fov_value_max=None,
                              small_fov_value_min=None, method_carrington_reprojection="fa",
                              alignement_method="carrington", path_output_figures: str = None, fov_limits=None):
    """`jitter_correction/jitter_correction.py:175-256`."""
    a = Alignment(large_fov_known_pointing=large_fov_fits_path, large_fov_window=large_fov_window,
                  small_fov_to_correct=small_fov_path, small_fov_window=window_to_align,
                  display_progress_bar=False, small_fov_value_max=small_fov_value_max,
                  small_fov_value_min=small_fov_value_min, parallelism=parallelism,
                  counts_cpu_max=cpu_count if cpu_count is not None else 40, unit_lag=unit_lag, **parameter_alignment)
    date_ref = _hms(reference_date)
    if alignement_method == "carrington":
        results = a.align_using_carrington(method="correlation", lonlims=lonlims, latlims=latlims, shape=shape,
                                           reference_date=reference_date,
                                           method_carrington_reprojection=method_carrington_reprojection)
    elif alignement_method == "initial_carrington":
        results = a.align_using_initial_carrington(method="correlation")
    elif alignement_method == "helioprojective":
        results = a.align_using_helioprojective(method="correlation", fov_limits=fov_limits)
    else:
        raise ValueError("alignement_method must be 'carrington', 'initial_carrington' or 'helioprojective'")
    _plot_correlation(results, path_output_figures, date_to_align, date_ref)
    return results


def _plot_correlation(results, path_output_figures, date_to_align, date_ref):
    if path_output_figures is not None:
        try:
            results.plot_correlation(
                path_save_figure=os.path.join(path_output_figures, f"correlation_{date_to_align}_{date_ref}.pdf"))
        except ImportError:
            warnings.warn("matplotlib is not installed: no correlation figure written")


def _write_corrected(results, path_input, window, path_files_output):
    results.write_corrected_fits(window_list_to_apply_shift=[window],
                                 path_to_l3_output=os.path.join(path_files_output, os.path.basename(path_input)))
