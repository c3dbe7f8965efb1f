"""directtrajopt.jl_b200 -- B200-native evaluator for DirectTrajOpt.jl's NLP-callback hot path.

The directory name carries a dot (it is the reference's name), so import it through the shim at the
repository root:  ``import dto_b200``  (which loads this package under that name).

Everything numerical happens in ``lib/libdto_b200.so`` (hand-written sm_100a CUDA behind the C ABI in
``include/dto_b200.h``); this package is the host-side mirror of the reference's Julia API for the
path: trajectory, integrators, objectives, constraints, problem and the MOI-style evaluator.
"""
from . import _lib
from ._lib import DtoError
from .components import (AbstractIntegrator, AbstractNonlinearConstraint, AbstractObjective, BilinearIntegrator,
                         CarrierGenerator, CompositeObjective, DerivativeIntegrator, IsoInfidelity, KnotFunction,
                         KnotPointObjective, LinearCost, LinearMap, LinearRegularizer, MinimumTimeObjective, NonlinearKnotPointConstraint,
                         NormMinus, NormSqMinus, NormSqPlus, NullObjective, QuadraticRegularizer, SqDist, SqDistMinus,
                         TerminalObjective, TimeDependentBilinearIntegrator, UnsupportedComponent,
                         GlobalObjective, GlobalKnotPointObjective, NonlinearGlobalConstraint, NonlinearGlobalKnotPointConstraint,
                         NormProduct, SplitSqDist, KnotHVP, ConstantLowRankHVP, CustomKnotHVP, knot_hvp)
from .evaluator import DirectTrajOptProblem, Evaluator
from .knot_program import KnotProgram
from .trajectory import KnotPoint, NamedTrajectory
from . import problem_templates

__all__ = [n for n in dir() if not n.startswith("_")]
