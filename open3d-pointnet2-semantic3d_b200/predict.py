"""Inference wrapper: the reference's ``Predictor`` (predict.py:15-105) on the sm_100a engine.

  Predictor(checkpoint, num_classes, hyper_params)
      .predict(batch_data)                  eval-mode forward + arg-max           predict.py:65-91
      .predict_scene(scene, num_samples)    the scene loop: boxes -> sparse labels predict.py:146-205
      .interpolate_labels(sparse_points, sparse_labels, dense_points, knn=3)      predict.py:93-105

``checkpoint`` is the ``variable name -> array`` dictionary of a TensorFlow checkpoint of this
network (the reference's scope names, see model.py), or the path of an ``.npz`` holding it; there is
no TF Saver here.  Everything runs on the GPU: the network through model.get_model, the dense-cloud
label transfer through tf_ops.tf_interpolate.interpolate_label_with_color (the reference does that
step on the host through an Open3D KD-tree).
"""
import numpy as np
import torch

from . import model
from ._ffi import F32
from .tf_ops.tf_interpolate import interpolate_label_with_color
from .util import tf_util


def _as_cuda(a, dtype, device):
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=dtype).contiguous()
    return torch.as_tensor(np.ascontiguousarray(a)).to(device=device, dtype=dtype).contiguous()


class Predictor:
    def __init__(self, checkpoint, num_classes, hyper_params, device="cuda"):
        self.num_classes, self.hyper_params = int(num_classes), hyper_params
        self.device = torch.device(device)
        self.store = tf_util.VariableStore(device=device, seed=0)
        if isinstance(checkpoint, str):
            with np.load(checkpoint) as z:
                checkpoint = {k: z[k] for k in z.files}
        if not checkpoint:
            raise ValueError("Predictor needs the checkpoint's variables (name -> array)")
        self.skipped = self.store.load_state_dict(checkpoint)  # optimizer slots etc. of a full TF checkpoint
        # a variable the checkpoint lacks must fail loudly, not be xavier-initialised during predict()
        self.store.strict = True

    def predict(self, batch_data):
        """batch_data (batch_size, num_point, 3 or 6) -> labels (batch_size, num_point), the arg-max
        of the eval-mode logits (moving-average BatchNorm, no dropout)."""
        x = _as_cuda(batch_data, torch.float32, self.device)
        if x.dim() != 3 or x.shape[2] != 3 + 3 * int(self.hyper_params["use_color"]):
            raise ValueError("batch_data must be (batch_size, num_point, %d)"
                             % (3 + 3 * int(self.hyper_params["use_color"])))
        tf_util.set_default_store(self.store)
        with torch.no_grad():
            pred, _ = model.get_model(x, False, self.num_classes, self.hyper_params)
            labels = torch.argmax(pred, dim=2)
        return labels.cpu().numpy()

    def interpolate_labels(self, sparse_points, sparse_labels, dense_points, knn=3):
        """Labels and colours of the full-resolution cloud from the labelled sparse cloud
        (k nearest neighbours vote, predict.py:93-105 feeds knn=3)."""
        sp = _as_cuda(sparse_points, torch.float32, self.device)
        sl = _as_cuda(sparse_labels, torch.int32, self.device)
        dp = _as_cuda(dense_points, torch.float32, self.device)
        labels, colors = interpolate_label_with_color(sp, sl, dp, int(knn))
        return labels.cpu().numpy(), colors.cpu().numpy()

    def predict_scene(self, scene, num_samples, batch_size=64, rng=np.random, seed=0, confusion=None):
        """The scene loop of predict.py:146-205: ``num_samples`` boxes cut from ``scene`` (a
        dataset.SemanticFileData) in ceil(num_samples / batch_size) batches, the last one shorter, batch i drawn
        by ``scene.sample_batch(..., rng=rng, seed=seed + i)`` without augmentation; each batch is predicted and,
        with ``confusion`` (a util.metric.ConfusionMatrix), its (gt, predicted) labels are counted in the same
        launch that takes the arg-max.  Returns (sparse_points (num_samples*num_point, 3) float64 in scene
        coordinates, sparse_labels (num_samples*num_point,) int64), copied to the host once at the end."""
        num_samples, batch_size = int(num_samples), int(batch_size)
        if num_samples <= 0 or batch_size <= 0:
            raise ValueError("num_samples and batch_size must be positive")
        if confusion is not None and confusion.num_classes != self.num_classes:
            raise ValueError("confusion has %d classes, the model %d" % (confusion.num_classes, self.num_classes))
        num_point = int(self.hyper_params["num_point"])
        use_color = int(self.hyper_params["use_color"])
        if scene.feat != 3 * use_color:
            raise ValueError("the scene has %d colour channels, the model expects %d" % (scene.feat, 3 * use_color))
        scratch = confusion
        if scratch is None:
            from .util.metric import ConfusionMatrix
            scratch = ConfusionMatrix(self.num_classes, device=self.device)
        points, labels = [], []
        tf_util.set_default_store(self.store)
        with torch.no_grad():
            for batch_index in range(-(-num_samples // batch_size)):
                current = min(batch_size, num_samples - batch_index * batch_size)
                data, gt, _, index, _ = scene.sample_batch(current, num_point, rng=rng, seed=seed + batch_index)
                pred, _ = model.get_model(data, False, self.num_classes, self.hyper_params)
                pd = torch.empty(gt.shape, dtype=torch.int32, device=self.device)
                scratch.increment_from_logits(pred.to(F32).contiguous(), gt, pred_out=pd)
                points.append(scene.points[index.reshape(-1).long()])
                labels.append(pd.reshape(-1))
        return torch.cat(points).cpu().numpy(), torch.cat(labels).long().cpu().numpy()
