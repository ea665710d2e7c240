"""montgomery_b200 -- B200-native MSM engine behind montgomery's msm(scalars, points) API."""
from . import curves, inputs  # noqa: F401
from .api import MsmEngine, MsmError, MultiGpuMsm, PointSet, TwistedEdwards, Weierstrass, make_compute_msm  # noqa: F401
from .api import PT_NONCANONICAL, PT_NOT_IN_SUBGROUP, PT_OFF_CURVE, InvalidPointsError  # noqa: F401
