from .alignment import Alignment  # noqa: F401
from .AlignmentResults import AlignmentResults, LocalAlignmentResults  # noqa: F401
from .alignment_spice import AlignmentSpice  # noqa: F401
from .sequence import SequenceAlignment  # noqa: F401
