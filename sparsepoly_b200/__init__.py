"""sparsepoly_b200 -- B200-native (sm_100a CUDA) solver backend behind sparsepoly's
sklearn-style API.  See DESIGN.md; the C ABI is declared in include/sparsepoly_b200.h."""
from .estimators import (
    SparseAllSubsetsClassifier,
    SparseAllSubsetsRegressor,
    SparseFactorizationMachineClassifier,
    SparseFactorizationMachineRegressor,
)
from .multi import fit_many
from .objective import objective

__all__ = [
    "fit_many",
    "objective",
    "SparseAllSubsetsClassifier",
    "SparseAllSubsetsRegressor",
    "SparseFactorizationMachineClassifier",
    "SparseFactorizationMachineRegressor",
]
__version__ = "0.1.0"
