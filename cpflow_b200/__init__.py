"""cpflow_b200 — B200-native engine for cpflow's multi-start variational synthesis loop.

Public names follow the reference package (cpflow/__init__.py:5-10)."""
__version__ = '0.1.0'

from ._lib import CpflowError  # noqa: F401
from .engine import Loss, MultiLoss, Penalty, Program, clean_ancilla_isometry  # noqa: F401
from .ansatz import Ansatz  # noqa: F401
from .main import (AdaptiveOptions, BasicOptions, Decomposition, RegularizationOptions, Results,  # noqa: F401
                   StaticOptions, Synthesize, synthesize_many)
from .legacy import load_reference_results  # noqa: F401,E402
