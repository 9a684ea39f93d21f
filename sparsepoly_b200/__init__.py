"""sparsepoly_b200 -- B200-native (sm_100a CUDA) solver backend behind sparsepoly's
sklearn-style API.  See DESIGN.md; the C ABI is declared in include/sparsepoly_b200.h."""
from .estimators import (
    SparseAllSubsetsClassifier,
    SparseAllSubsetsRegressor,
    SparseFactorizationMachineClassifier,
    SparseFactorizationMachineRegressor,
)
from .multi import decision_function_many, fit_many, objective_many, predict_many, score_many
from .objective import objective

__all__ = [
    "decision_function_many",
    "fit_many",
    "objective_many",
    "predict_many",
    "score_many",
    "objective",
    "SparseAllSubsetsClassifier",
    "SparseAllSubsetsRegressor",
    "SparseFactorizationMachineClassifier",
    "SparseFactorizationMachineRegressor",
]
__version__ = "0.1.0"
