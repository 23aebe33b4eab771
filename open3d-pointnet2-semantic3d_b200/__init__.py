"""pn2_b200 -- Blackwell-native PointNet++ set-abstraction / feature-propagation engine.

Drop-in for the hot path of isl-org/Open3D-PointNet2-Semantic3D: the ``tf_ops`` op surface
(``tf_sampling``, ``tf_grouping``, ``tf_interpolate``), the ``util.pointnet_util`` /
``util.tf_util`` layers and ``model.get_model/get_loss``, all backed by hand-written sm_100a
CUDA kernels behind the C ABI of ``include/pn2_b200.h`` (``lib/libpn2_b200.so``).  PyTorch
tensors are only the device-memory container.  There is no CPU fallback.

The directory name contains hyphens, so import it through the repo-root shim::

    import pn2_b200
    from pn2_b200.tf_ops.tf_sampling import farthest_point_sample
"""
import sys

from . import _ffi  # noqa: F401


def install_reference_aliases(include_model=True):
    """Register the reference's absolute module names (``tf_ops.tf_sampling``, ``util.tf_util``,
    ``util.pointnet_util`` ...) so code written against the reference imports resolves here.
    ``include_model=False`` leaves ``model`` / ``predict`` alone: the caller imports the reference's own
    model.py (see compat/tensorflow.py)."""
    from . import tf_ops, util, model, predict
    from .tf_ops import tf_grouping, tf_interpolate, tf_sampling
    from .util import metric, pointnet_util, tf_util
    sys.modules.setdefault("tf_ops", tf_ops)
    sys.modules.setdefault("tf_ops.tf_sampling", tf_sampling)
    sys.modules.setdefault("tf_ops.tf_grouping", tf_grouping)
    sys.modules.setdefault("tf_ops.tf_interpolate", tf_interpolate)
    sys.modules.setdefault("util", util)
    sys.modules.setdefault("util.tf_util", tf_util)
    sys.modules.setdefault("util.pointnet_util", pointnet_util)
    sys.modules.setdefault("util.metric", metric)
    if include_model:
        sys.modules.setdefault("model", model)      # the reference's top-level `import model`
        sys.modules.setdefault("predict", predict)  # `from predict import Predictor`
    return model
