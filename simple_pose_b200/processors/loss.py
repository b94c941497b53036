"""Masked joints-MSE loss: drop-in for the expression every reference solver repeats
(``processors/dp_pose_hrnet_solver.py:86,106-107`` and, under ``torch.cuda.amp``, ``:111-120``)::

    loss = 0.5 * nn.MSELoss()(pred.mul(mask[[..., None, None]]), target.mul(mask[[..., None, None]]))
    loss.backward()                      # or scaler.scale(loss).backward()

``JointsMSELoss()(pred, target, mask)`` returns the same 0-d float32 tensor with autograd support.

* float32 ``pred``: forward and backward are ONE kernel (``sp_mse_fwd_bwd_f32``): the gradient w.r.t.
  ``pred`` is produced while the loss is being reduced; ``backward`` only rescales it when the upstream
  gradient is not 1, and that rescale kernel exits without touching memory when the factor is exactly 1.
* float16 / bfloat16 ``pred`` (autocast output): no conversion passes. Forward reads ``pred`` in its own
  dtype and reduces the loss in float32 (as autocast does: the fp16 * fp32 product promotes, ``mse_loss``
  is on autocast's float32 list); backward recomputes the difference and writes the gradient in ``pred``'s
  dtype, with the upstream gradient -- ``GradScaler``'s scale -- applied in float32 BEFORE the cast and read
  from device memory (no host sync). 14 bytes per element instead of 32 for convert / float32 kernel /
  rescale / convert back.
"""
import torch

from .. import _abi

_DTYPE_CODE = {torch.float32: _abi.SP_DTYPE_F32, torch.float16: _abi.SP_DTYPE_F16, torch.bfloat16: _abi.SP_DTYPE_BF16}


def _workspace(device, stream_id):
    """Zero-initialised reduction workspace per (device, stream); the kernel restores the zero state."""
    return _abi.scratch(device, stream_id, int(_abi.lib().sp_mse_workspace_bytes()), "mse")


def _pred_tensor(pred):
    """pred as a dense tensor the kernels read natively (float32 / float16 / bfloat16; anything else -> float32)."""
    p = pred.detach()
    if p.dtype not in _DTYPE_CODE:
        p = p.to(torch.float32)
    return p.contiguous()


def _check_shapes(pred, target, mask):
    if pred.dim() < 3:
        raise ValueError("pred must be [B, K, ...]")
    b, k = int(pred.shape[0]), int(pred.shape[1])
    hw = 1
    for s in pred.shape[2:]:
        hw *= int(s)
    if tuple(target.shape) != tuple(pred.shape) or tuple(mask.shape) != (b, k):
        raise ValueError("shape mismatch: pred %s target %s mask %s" % (tuple(pred.shape), tuple(target.shape), tuple(mask.shape)))
    return b, k, hw


def mse_forward_backward(pred, target, mask, need_grad=True, grad_scale=1.0, skip_masked=False, need_loss=True,
                         grad_scale_dev=None, want_acc=False, distance_thresh=0.5, norm_frac=10., axes_out=None):
    """(loss 0-d float32 or None, grad like pred or None); everything on pred's CUDA device.

    ``pred`` may be float32, float16 or bfloat16 (``grad`` has the same dtype); ``grad_scale_dev`` is an
    optional 0-d float32 device tensor multiplied into the gradient on the device; ``need_loss=False``
    is the backward-only call.

    ``want_acc=True`` (forward calls only) also computes ``HeatMapAcc(distance_thresh, norm_frac)(pred.mul(mask),
    target.mul(mask))`` in the same launch (``sp_mse_acc_fwd_bwd``) and returns ``(loss, grad, acc)``, acc a 0-d
    float32 device tensor; ``axes_out`` = optional ``(pred_xy, label_xy)`` dense float32 [B, K, 2] tensors that
    receive the two argmax coordinate tables."""
    dev = _abi.require_cuda(pred, target, mask, grad_scale_dev)
    b, k, hw = _check_shapes(pred, target, mask)
    if not need_loss and not need_grad:
        raise ValueError("nothing to compute")
    if want_acc and (not need_loss or pred.dim() != 4):
        raise ValueError("want_acc needs the forward call (need_loss=True) and pred [B, K, H, W]")
    p = _pred_tensor(pred)
    t = _abi.dense(target.detach(), torch.float32)
    m = _abi.dense(mask.detach(), torch.float32)
    s = None if grad_scale_dev is None else _abi.dense(grad_scale_dev.detach(), torch.float32)
    loss = torch.empty((), dtype=torch.float32, device=dev) if need_loss else None
    grad = torch.empty_like(p) if need_grad else None
    stream = _abi.stream_ptr(dev)
    flags = _abi.SP_MSE_SKIP_MASKED if skip_masked else 0
    if not want_acc:
        ws = _workspace(dev, stream)
        with torch.cuda.device(dev):
            _abi.check_ws(_abi.lib().sp_mse_fwd_bwd(p.data_ptr(), _DTYPE_CODE[p.dtype], t.data_ptr(), m.data_ptr(),
                                                    _abi.ptr(grad), _abi.ptr(loss), ws.data_ptr(), ws.numel() * 8, b, k, hw,
                                                    float(grad_scale), _abi.ptr(s), flags, stream), dev, stream)
        return loss, grad
    h, w = int(pred.shape[2]), int(pred.shape[3])
    pxy, lxy = axes_out if axes_out is not None else (None, None)
    for a in (pxy, lxy):
        if a is not None and (a.device != dev or a.dtype != torch.float32 or tuple(a.shape) != (b, k, 2)
                              or not a.is_contiguous()):
            raise ValueError("axes_out must be two contiguous float32 [B, K, 2] tensors on %s" % dev)
    acc = torch.empty((), dtype=torch.float32, device=dev)
    ws = _abi.scratch(dev, stream, int(_abi.lib().sp_mse_acc_workspace_bytes(b, k)), "mse_acc")
    with torch.cuda.device(dev):
        _abi.check_ws(_abi.lib().sp_mse_acc_fwd_bwd(p.data_ptr(), _DTYPE_CODE[p.dtype], t.data_ptr(), m.data_ptr(),
                                                    _abi.ptr(grad), loss.data_ptr(), acc.data_ptr(), _abi.ptr(pxy),
                                                    _abi.ptr(lxy), ws.data_ptr(), ws.numel() * 8, b, k, h, w,
                                                    float(grad_scale), _abi.ptr(s), float(distance_thresh),
                                                    float(norm_frac), flags, stream), dev, stream)
    return loss, grad, acc


def _scale_saved_grad(ctx, grad, grad_out):
    """backward of the single-kernel float32 path: the gradient was written in forward; apply the upstream
    gradient in place (the kernel reads it on the device and exits without traffic when it is exactly 1)."""
    if getattr(ctx, "consumed", False):
        raise RuntimeError(
            "simple_pose_b200: the float32 loss node writes d loss / d pred in its forward kernel and rescales that "
            "buffer in place in backward, so it can be differentiated once; for repeated backward passes through one "
            "graph (retain_graph=True) build the loss with defer_grad=True")
    ctx.consumed = True
    dev = grad.device
    g = _abi.dense(grad_out.detach().to(dev), torch.float32)
    with torch.cuda.device(dev):
        _abi.check(_abi.lib().sp_scale_inplace_f32(grad.data_ptr(), grad.numel(), g.data_ptr(), _abi.stream_ptr(dev)))
    return grad


class _MaskedMSE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, mask, skip_masked, defer_grad, grad_mode, acc_args):
        need = grad_mode and pred.requires_grad        # grad_mode: torch.is_grad_enabled() at the call site (it is off in here)
        deferred = need and (defer_grad or pred.dtype in (torch.float16, torch.bfloat16))
        if acc_args is None:
            loss, grad = mse_forward_backward(pred, target, mask, need_grad=need and not deferred, skip_masked=skip_masked)
        else:                                          # (holder, distance_thresh, norm_frac): HeatMapAcc in the same launch
            holder, thresh, frac = acc_args
            loss, grad, holder["acc"] = mse_forward_backward(pred, target, mask, need_grad=need and not deferred,
                                                             skip_masked=skip_masked, want_acc=True,
                                                             distance_thresh=thresh, norm_frac=frac)
        ctx.deferred, ctx.skip_masked, ctx.pred_dtype = deferred, skip_masked, pred.dtype
        if deferred:
            ctx.save_for_backward(pred, target, mask)
        else:
            ctx.save_for_backward(grad if need else None)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        none = (None,) * 6
        if ctx.deferred:
            pred, target, mask = ctx.saved_tensors
            _, grad = mse_forward_backward(pred, target, mask, need_grad=True, need_loss=False, skip_masked=ctx.skip_masked,
                                           grad_scale_dev=grad_out.detach().to(pred.device).reshape(()))
            return (grad.to(ctx.pred_dtype).view_as(pred),) + none
        (grad,) = ctx.saved_tensors
        if grad is None:
            return (None,) + none
        out = _scale_saved_grad(ctx, grad, grad_out)
        return (out if ctx.pred_dtype == torch.float32 else out.to(ctx.pred_dtype),) + none


class JointsMSELoss(torch.nn.Module):
    """``loss = JointsMSELoss()(pred [B,K,H,W], target [B,K,H,W], mask [B,K])``.

    ``skip_masked=True`` does not read pred/target of joints whose mask is 0 (saves their HBM
    traffic; differs from the reference only when those maps hold NaN/Inf, which the
    reference would propagate into the loss). ``defer_grad=True`` computes the gradient in backward
    instead of forward also for float32 predictions (float16 / bfloat16 always do): nothing the size of
    ``pred`` is kept between forward and backward and the node may be differentiated repeatedly.

    ``with_acc=True`` returns ``(loss, acc)``: ``acc`` is ``HeatMapAcc(distance_thresh, norm_frac)(pred.mul(mask),
    target.mul(mask))``, a 0-d float32 device tensor (no host sync), computed by the loss kernel while ``pred`` and
    ``target`` stream by -- no masked copies, no argmax launches. ``pred`` must be [B, K, H, W]::

        crit = JointsMSELoss(with_acc=True)
        loss, acc = crit(predicts, targets, mask)     # == 0.5 * MSELoss(...) and HeatMapAcc()(predicts*mask, targets*mask)
    """

    def __init__(self, skip_masked=False, defer_grad=False, with_acc=False, distance_thresh=0.5, norm_frac=10.):
        super().__init__()
        self.skip_masked = bool(skip_masked)
        self.defer_grad = bool(defer_grad)
        self.with_acc = bool(with_acc)
        self.distance_thresh, self.norm_frac = distance_thresh, norm_frac
        self.acc = None

    def forward(self, pred, target, mask):
        if not self.with_acc:
            return _MaskedMSE.apply(pred, target, mask, self.skip_masked, self.defer_grad, torch.is_grad_enabled(), None)
        holder = {}
        loss = _MaskedMSE.apply(pred, target, mask, self.skip_masked, self.defer_grad, torch.is_grad_enabled(),
                                (holder, self.distance_thresh, self.norm_frac))
        self.acc = holder["acc"]
        return loss, self.acc


def encode_mse_forward_backward(joints, pred, sigma=2.0, need_grad=True, want_targets=False, want_axes=False,
                                grad_scale=1.0, need_loss=True, grad_scale_dev=None):
    """Fused target encoding + masked MSE (+ HeatMapAcc argmaxes): one pass over ``pred``.

    joints [B,K,3] heatmap px, pred [B,K,H,W] float32 / float16 / bfloat16. Returns a dict with loss (0-d),
    weights [B,K], and optionally grad (pred's dtype), targets, pred_xy / label_xy [B,K,2]."""
    dev = _abi.require_cuda(joints, pred, grad_scale_dev)
    if pred.dim() != 4:
        raise ValueError("pred must be [B, K, H, W]")
    b, k, h, w = (int(s) for s in pred.shape)
    if tuple(joints.shape) != (b, k, 3):
        raise ValueError("joints must be [B, K, 3] matching pred")
    j = _abi.dense(joints.detach(), torch.float32)
    p = _pred_tensor(pred)
    s = None if grad_scale_dev is None else _abi.dense(grad_scale_dev.detach(), torch.float32)
    out = {"loss": torch.empty((), dtype=torch.float32, device=dev) if need_loss else None,
           "weights": torch.empty((b, k), dtype=torch.float32, device=dev),
           "grad": torch.empty_like(p) if need_grad else None,
           "targets": torch.empty((b, k, h, w), dtype=torch.float32, device=dev) if want_targets else None,
           "pred_xy": torch.empty((b, k, 2), dtype=torch.float32, device=dev) if want_axes else None,
           "label_xy": torch.empty((b, k, 2), dtype=torch.float32, device=dev) if want_axes else None}
    stream = _abi.stream_ptr(dev)
    ws = _workspace(dev, stream)
    if w % 4 != 0:
        # shapes the fused kernel does not take: same results from the encoder and the loss kernel, which takes the
        # HeatMapAcc argmaxes along when they are wanted
        from ..commons.transforms import encode_heat_maps
        tg, wt = encode_heat_maps(j, sigma, (w, h))
        if want_axes:
            loss, grad, _ = mse_forward_backward(p, tg, wt, need_grad=need_grad, grad_scale=grad_scale, grad_scale_dev=s,
                                                 want_acc=True, axes_out=(out["pred_xy"], out["label_xy"]))
            loss = loss if need_loss else None
        else:
            loss, grad = mse_forward_backward(p, tg, wt, need_grad=need_grad, grad_scale=grad_scale, need_loss=need_loss,
                                              grad_scale_dev=s)
        out.update(loss=loss, grad=grad, weights=wt, targets=tg if want_targets else None)
        return out
    with torch.cuda.device(dev):
        _abi.check_ws(_abi.lib().sp_encode_mse_fwd_bwd(
            j.data_ptr(), p.data_ptr(), _DTYPE_CODE[p.dtype], _abi.ptr(out["grad"]), _abi.ptr(out["targets"]),
            out["weights"].data_ptr(), _abi.ptr(out["loss"]), _abi.ptr(out["pred_xy"]), _abi.ptr(out["label_xy"]),
            ws.data_ptr(), ws.numel() * 8, b, k, h, w, float(sigma), float(grad_scale), _abi.ptr(s), stream), dev, stream)
    return out


class _EncodeMaskedMSE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, joints, sigma, want_targets, want_axes, holder, defer_grad, grad_mode):
        need = grad_mode and pred.requires_grad
        deferred = need and (defer_grad or pred.dtype in (torch.float16, torch.bfloat16))
        out = encode_mse_forward_backward(joints, pred, sigma, need_grad=need and not deferred, want_targets=want_targets,
                                          want_axes=want_axes)
        holder.update(out)
        ctx.deferred, ctx.sigma, ctx.pred_dtype = deferred, sigma, pred.dtype
        if deferred:
            ctx.save_for_backward(pred, joints)
        else:
            ctx.save_for_backward(out["grad"] if need else None)
        return out["loss"]

    @staticmethod
    def backward(ctx, grad_out):
        none = (None,) * 7
        if ctx.deferred:
            pred, joints = ctx.saved_tensors
            out = encode_mse_forward_backward(joints, pred, ctx.sigma, need_grad=True, need_loss=False,
                                              grad_scale_dev=grad_out.detach().to(pred.device).reshape(()))
            return (out["grad"].to(ctx.pred_dtype).view_as(pred),) + none
        (grad,) = ctx.saved_tensors
        if grad is None:
            return (None,) + none
        out = _scale_saved_grad(ctx, grad, grad_out)
        return (out if ctx.pred_dtype == torch.float32 else out.to(ctx.pred_dtype),) + none


class EncodeJointsMSELoss(torch.nn.Module):
    """Training-step half of the path in one kernel (SURVEY section 8f ranks 1-2): takes the heatmap-pixel
    joints the loader already has (``transforms.py:218``) instead of pre-rendered targets.

        crit = EncodeJointsMSELoss(sigma=2.0, with_acc=True)
        loss, acc = crit(pred, joints)          # == reference loss and HeatMapAcc()(pred*mask, target*mask)
        loss.backward()                          # or scaler.scale(loss).backward() with a float16 pred
        crit.weights                             # the [B,K] mask the reference's loader would have shipped
    """

    def __init__(self, sigma=2.0, with_acc=False, keep_targets=False, distance_thresh=0.5, norm_frac=10., defer_grad=False):
        super().__init__()
        self.sigma, self.with_acc, self.keep_targets = float(sigma), bool(with_acc), bool(keep_targets)
        self.distance_thresh, self.norm_frac = distance_thresh, norm_frac
        self.defer_grad = bool(defer_grad)
        self.weights = self.targets = self.acc = None

    def forward(self, pred, joints):
        holder = {}
        loss = _EncodeMaskedMSE.apply(pred, joints, self.sigma, self.keep_targets, self.with_acc, holder, self.defer_grad,
                                      torch.is_grad_enabled())
        self.weights, self.targets = holder["weights"], holder["targets"]
        if not self.with_acc:
            return loss
        from ..metrics.pose_metrics import heatmap_acc_from_axes
        self.acc = heatmap_acc_from_axes(holder["pred_xy"], holder["label_xy"], pred.shape[-2], pred.shape[-1],
                                         self.distance_thresh, self.norm_frac)
        return loss, self.acc
