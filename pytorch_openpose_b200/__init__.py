"""B200-native OpenPose inference path: drop-in `Body` / `Hand` (reference: src/body.py, src/hand.py) over
hand-written sm_100a kernels in libopenpose_b200.so.  See DESIGN.md / INTEGRATION.md."""
from .body import Body            # noqa: F401
from .hand import Hand            # noqa: F401
from .batch_model import Batch_body, Batch_hand, BatchPoseEstimator      # noqa: F401
from . import util                # noqa: F401


def install_as_src():
    """Register this package under the reference's module names so that `from src.body import Body`,
    `from src.hand import Hand`, `from src import util, model` (srcmx/MotionEstimation.py:12-15,
    srcmx/Batch_model.py:30-33) resolve to the B200 implementation."""
    import sys
    import types
    from . import body, hand, util as _util, model
    pkg = types.ModuleType("src")
    pkg.__path__ = []
    pkg.body, pkg.hand, pkg.util, pkg.model = body, hand, _util, model
    sys.modules.update({"src": pkg, "src.body": body, "src.hand": hand, "src.util": _util, "src.model": model})
    return pkg


def install_as_batch_model():
    """`import Batch_model as BM; BM.Batch_body(path)` (srcmx/Batch_motion_Estimation.py:11,22,60) -> the B200 classes.
    Only the two estimators are provided; the reference module's video dataset helpers stay where they are."""
    import sys
    from . import batch_model
    sys.modules["Batch_model"] = batch_model
    return batch_model
