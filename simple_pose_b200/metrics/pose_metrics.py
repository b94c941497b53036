"""Heatmap decoders: drop-ins for the reference's ``metrics/pose_metrics.py``.

``BasicKeyPointDecoder`` (:10-52) and ``GaussTaylorKeyPointDecoder`` (:55-107) keep their
constructor and call signatures; every call is one launch of the fused sm_100a kernel
``sp_decode_f32`` (argmax + 13-point blur + log + Taylor + affine), instead of ~60 ATen ops and
seven passes over the heatmaps. ``flip_call`` adds the flip-test average (not in the reference;
composed from its ``flip_joints`` / ``joint_pairs`` semantics, see SURVEY.md section 8a A6).
"""
import numpy as np
import torch

from .. import _abi
from ..commons.joint_utils import swap_permutation


# cv.getGaussianKernel(n, 0) returns these fixed tables for n <= 9 (OpenCV's small_gaussian_tab, extended to 9
# in 4.x), not the closed form
_OPENCV_FIXED_TAPS = {
    1: (1.0,),
    3: (0.25, 0.5, 0.25),
    5: (0.0625, 0.25, 0.375, 0.25, 0.0625),
    7: (0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125),
    9: (4.0 / 256, 13.0 / 256, 30.0 / 256, 51.0 / 256, 60.0 / 256, 51.0 / 256, 30.0 / 256, 13.0 / 256, 4.0 / 256),
}


def gaussian_kernel_1d(kernel_size):
    """``cv.getGaussianKernel(kernel_size, 0)`` (float64 column). OpenCV itself when importable
    (as the reference does, pose_metrics.py:57); otherwise its fixed tables for n <= 9 and its closed
    form above that (sigma = 0.3*((n-1)*0.5-1)+0.8, normalised exp(-x^2/(2 sigma^2))), which gives
    bit-identical float32 2-D weights for the reference's kernel_size = 11."""
    n = int(kernel_size)
    try:
        import cv2
        return cv2.getGaussianKernel(n, 0)
    except ImportError:
        if n in _OPENCV_FIXED_TAPS:
            return np.array(_OPENCV_FIXED_TAPS[n], dtype=np.float64).reshape(-1, 1)
        if n < 11 or n % 2 == 0:
            raise RuntimeError("kernel_size %d needs OpenCV (cv2 not importable)" % n)
        sigma = 0.3 * ((n - 1) * 0.5 - 1) + 0.8
        x = np.arange(n, dtype=np.float64) - (n - 1) * 0.5
        g = np.exp(-(x * x) / (2.0 * sigma * sigma))
        return (g / g.sum()).reshape(-1, 1)


def _decode(heat_map, heat_map_flip, perm, trans_inv, blur_w, ksize, mode, want_index=False):
    dev = _abi.require_cuda(heat_map, heat_map_flip, trans_inv)
    if heat_map.dim() != 4:
        raise ValueError("heat_map must be [B, K, H, W]")
    b, k, h, w = (int(s) for s in heat_map.shape)
    hm = _abi.dense(heat_map.detach(), torch.float32)
    hf = None
    if heat_map_flip is not None:
        if tuple(heat_map_flip.shape) != tuple(heat_map.shape):
            raise ValueError("heat_map_flip must have the shape of heat_map")
        hf = _abi.dense(heat_map_flip.detach(), torch.float32)
    ti = None
    if trans_inv is not None:
        if tuple(trans_inv.shape) != (b, 2, 3):
            raise ValueError("trans_inv must be [B, 2, 3]")
        ti = _abi.dense(trans_inv.detach(), torch.float32)
    coords = torch.empty((b, k, 2), dtype=torch.float32, device=dev)
    maxval = torch.empty((b, k, 1), dtype=torch.float32, device=dev)
    index = torch.empty((b, k), dtype=torch.int32, device=dev) if want_index else None
    stream = _abi.stream_ptr(dev)
    ws = _abi.scratch(dev, stream, 16, "decode")
    with torch.cuda.device(dev):
        _abi.check_ws(_abi.lib().sp_decode_ws_f32(hm.data_ptr(), _abi.ptr(hf), _abi.ptr(perm), _abi.ptr(ti),
                                                  _abi.ptr(blur_w), coords.data_ptr(), maxval.data_ptr(),
                                                  _abi.ptr(index), b, k, h, w, int(ksize), int(mode),
                                                  ws.data_ptr(), ws.numel() * 8, stream), dev, stream)
    if want_index:
        return coords, maxval, index
    return coords, maxval


class BasicKeyPointDecoder(object):
    @staticmethod
    def heat_map_to_axis(heat_map):
        """[B,K,H,W] -> (coords [B,K,2] (x, y) float32, max_val [B,K,1]); reference :11-24."""
        return _decode(heat_map, None, None, None, None, 0, _abi.SP_DECODE_ARGMAX)

    @staticmethod
    def heat_map_argmax(heat_map):
        """As ``heat_map_to_axis`` plus the flat int32 argmax [B,K] (first maximal index)."""
        return _decode(heat_map, None, None, None, None, 0, _abi.SP_DECODE_ARGMAX, want_index=True)

    @torch.no_grad()
    def __call__(self, heat_map, trans_inv):
        return _decode(heat_map, None, None, trans_inv, None, 0, _abi.SP_DECODE_BASIC)


class GaussTaylorKeyPointDecoder(BasicKeyPointDecoder):
    def __init__(self, kernel_size=11, num_joints=17):
        kernel = gaussian_kernel_1d(kernel_size)
        self.kernel_size = kernel_size
        self.num_joints = num_joints
        # float32(k k^T), as pose_metrics.py:60 (one copy; the kernel is depthwise-identical)
        self.blur_weights = torch.from_numpy(np.ascontiguousarray((kernel * kernel.T).astype(np.float32)))
        self._perm_cache = {}

    def _weights_on(self, device):
        if self.blur_weights.device != device:
            self.blur_weights = self.blur_weights.to(device)
        return self.blur_weights

    def _perm_on(self, device, num_joints, joint_pairs):
        key = (device, num_joints, None if joint_pairs is None else tuple(map(tuple, joint_pairs)))
        perm = self._perm_cache.get(key)
        if perm is None:
            perm = torch.tensor(swap_permutation(num_joints, joint_pairs), dtype=torch.int32, device=device)
            self._perm_cache[key] = perm
        return perm

    @torch.no_grad()
    def __call__(self, heat_map, trans_inv):
        """heat_map [B,K,H,W], trans_inv [B,2,3] -> (coords [B,K,2] image px, max_val [B,K,1])."""
        return _decode(heat_map, None, None, trans_inv, self._weights_on(heat_map.device),
                       self.kernel_size, _abi.SP_DECODE_GAUSS_TAYLOR)

    @torch.no_grad()
    def flip_call(self, heat_map, heat_map_flip, trans_inv, joint_pairs=None):
        """Flip-test decode: ``heat_map_flip`` is the network output for the mirrored image.
        Decodes 0.5*(heat_map + mirror_x(heat_map_flip)[:, swap(joint_pairs)]) without
        materialising the average."""
        dev = heat_map.device
        perm = self._perm_on(dev, int(heat_map.shape[1]), joint_pairs)
        return _decode(heat_map, heat_map_flip, perm, trans_inv, self._weights_on(dev),
                       self.kernel_size, _abi.SP_DECODE_GAUSS_TAYLOR)

    @torch.no_grad()
    def decode_with_index(self, heat_map, trans_inv=None, heat_map_flip=None, joint_pairs=None):
        """Same as ``__call__``/``flip_call`` but also returns the flat argmax (int32 [B,K]);
        ``trans_inv=None`` gives heatmap-space coordinates."""
        dev = heat_map.device
        perm = self._perm_on(dev, int(heat_map.shape[1]), joint_pairs) if heat_map_flip is not None else None
        return _decode(heat_map, heat_map_flip, perm, trans_inv, self._weights_on(dev),
                       self.kernel_size, _abi.SP_DECODE_GAUSS_TAYLOR, want_index=True)


class DarkPoseOriginalKeyPointDecoder(GaussTaylorKeyPointDecoder):
    """Drop-in for the reference's third decoder (``metrics/pose_metrics.py:110-169``), its NumPy/OpenCV
    per-joint loop: zero-padded ``cv.GaussianBlur`` (float64), rescale by ``origin_max / blurred_max``,
    ``log(max(., 1e-10))``, the same Taylor step, and -- the one semantic difference to
    ``GaussTaylorKeyPointDecoder`` -- no ``clamp(min=0)`` of the refined coordinates. Same kernel, mode
    ``SP_DECODE_DARK_ORIGINAL``; agrees with the reference class to ~1e-5 px (it blurs in float64, the
    kernel in float32). Unlike the reference it returns tensors on the input's device and does not
    overwrite ``heat_map`` with its blurred copy (the reference does, through the shared NumPy view)."""

    def __init__(self, kernel_size=11):
        super().__init__(kernel_size=kernel_size, num_joints=17)

    @torch.no_grad()
    def __call__(self, heat_map, trans_inv):
        return _decode(heat_map, None, None, trans_inv, self._weights_on(heat_map.device),
                       self.kernel_size, _abi.SP_DECODE_DARK_ORIGINAL)


def heatmap_acc_from_axes(pred_xy, label_xy, height, width, distance_thresh=0.5, norm_frac=10.):
    """HeatMapAcc epilogue on [B,K,2] argmax coordinates -> 0-d float32 tensor (no host sync)."""
    dev = _abi.require_cuda(pred_xy, label_xy)
    p = _abi.dense(pred_xy, torch.float32)
    l = _abi.dense(label_xy, torch.float32)
    b, k = int(p.shape[0]), int(p.shape[1])
    acc = torch.empty((), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _abi.check(_abi.lib().sp_heatmap_acc_f32(p.data_ptr(), l.data_ptr(), acc.data_ptr(), b, k, int(height),
                                                 int(width), float(distance_thresh), float(norm_frac),
                                                 _abi.stream_ptr(dev)))
    return acc


class HeatMapAcc(object):
    """Drop-in for the reference's ``HeatMapAcc`` (metrics/pose_metrics.py:212-245): two argmax
    launches + one tiny epilogue, no 17-iteration Python loop and no ``.item()`` syncs. When the
    loss is computed with ``EncodeJointsMSELoss(with_acc=True)`` even the two argmax passes
    disappear (they ride along with the loss kernel)."""

    def __init__(self, distance_thresh=0.5, norm_frac=10.):
        self.distance_thresh = distance_thresh
        self.norm_frac = norm_frac

    @torch.no_grad()
    def __call__(self, predicts, targets):
        preds, _ = BasicKeyPointDecoder.heat_map_to_axis(predicts)
        labels, _ = BasicKeyPointDecoder.heat_map_to_axis(targets)
        return heatmap_acc_from_axes(preds, labels, predicts.shape[-2], predicts.shape[-1],
                                     self.distance_thresh, self.norm_frac)


def person_rows(predicts, scores):
    """[B,K,2], [B,K,1] device tensors -> float32 [B, 3K+1] device table: (x, y, conf) * K, then the
    person score mean(conf) + max(conf) of ``kps_to_dict_``; one launch of ``sp_person_rows_f32``."""
    dev = _abi.require_cuda(predicts, scores)
    if predicts.dim() != 3 or predicts.shape[-1] != 2 or scores.numel() != predicts.shape[0] * predicts.shape[1]:
        raise ValueError("predicts must be [B, K, 2] and scores [B, K, 1]")
    n, k = int(predicts.shape[0]), int(predicts.shape[1])
    c = _abi.dense(predicts.detach(), torch.float32)
    m = _abi.dense(scores.detach(), torch.float32)
    rows = torch.empty((n, 3 * k + 1), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _abi.check(_abi.lib().sp_person_rows_f32(c.data_ptr(), m.data_ptr(), rows.data_ptr(), n, k, _abi.stream_ptr(dev)))
    return rows


def kps_to_dict_(predicts, scores, img_ids, set_in_list):
    """Reference :172-179 with ONE kernel and ONE device->host copy instead of a ``mean``/``max``/``cat``
    chain plus one ``.item()`` and one ``.tolist()`` (two device syncs) per person:
    score = mean + max of the joint peaks, keypoints = [x, y, score] * K."""
    rows_to_dicts(person_rows(predicts, scores), img_ids, set_in_list)


def rows_to_dicts(rows, img_ids, set_in_list):
    """``kps_to_dict_``'s dicts from its [N, 3K+1] rows (``person_rows`` or ``HeatmapHotPath.val_step``), one
    device->host copy for the whole table."""
    for row, img_id in zip(rows.cpu().tolist(), img_ids):
        set_in_list.append({"image_id": img_id, "score": float(row[-1]), "category_id": 1, "keypoints": row[:-1]})
