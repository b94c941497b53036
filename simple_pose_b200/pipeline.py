"""The hot path as one object: encode -> masked-MSE fwd/bwd -> decode over a batch of persons.

This is the call a training/eval loop makes per batch once the backbone has produced
``pred``; it is what ``bench.py`` times and what ``eval_shard.py`` runs per rank. Outputs are
pre-allocated once (the library itself never allocates device memory).
"""
import torch

from . import _abi
from .metrics.pose_metrics import GaussTaylorKeyPointDecoder

ALGO_BYTES = {
    # algorithmic bytes per person (SURVEY.md section 8d), K joints, H x W float32 maps
    "encode": lambda k, h, w: k * h * w * 4 + k * 4 + k * 12,
    "loss": lambda k, h, w: 3 * k * h * w * 4 + k * 4,
    "decode": lambda k, h, w: k * h * w * 4 + 24 + k * 12,
    "flip_decode": lambda k, h, w: 2 * k * h * w * 4 + 24 + k * 12,
    # fused encode + loss fwd/bwd + HeatMapAcc argmaxes: read pred, write grad (+ joints, weights, axes)
    "train_fused": lambda k, h, w: 2 * k * h * w * 4 + k * 12 + k * 4 + k * 16,
    # one-launch step (sp_step_f32): read pred once, write targets and grad (+ joints, weights, affine, keypoints)
    "step": lambda k, h, w: 3 * k * h * w * 4 + k * 12 + k * 4 + 24 + k * 12,
}


class HeatmapHotPath(object):
    """Pre-allocated buffers + raw ABI calls for one batch shape on one device."""

    def __init__(self, batch, joints=17, height=64, width=48, sigma=2.0, device=None, kernel_size=11,
                 coords=None, maxval=None):
        self.device = torch.device(device) if device is not None else _abi.default_device()
        self.batch, self.k, self.h, self.w = int(batch), int(joints), int(height), int(width)
        self.sigma = float(sigma)
        dev = self.device
        self.targets = torch.empty((self.batch, self.k, self.h, self.w), dtype=torch.float32, device=dev)
        self.weights = torch.empty((self.batch, self.k), dtype=torch.float32, device=dev)
        self.grad = torch.empty_like(self.targets)
        self.loss = torch.empty((), dtype=torch.float32, device=dev)
        # decoder outputs may be views into a larger buffer (e.g. the all-gather send buffer)
        self.coords = coords if coords is not None else torch.empty((self.batch, self.k, 2), dtype=torch.float32, device=dev)
        self.maxval = maxval if maxval is not None else torch.empty((self.batch, self.k, 1), dtype=torch.float32, device=dev)
        assert self.coords.is_contiguous() and self.maxval.is_contiguous()
        self.decoder = GaussTaylorKeyPointDecoder(kernel_size, joints)
        self.blur_w = self.decoder._weights_on(dev)
        self.ksize = int(kernel_size)
        self.pred_xy = self.label_xy = None
        self.rows = self.acc = self.vws = None       # val_step's outputs and workspace, allocated at its first call
        self._lib = _abi.lib()
        # reduction / work-counter scratch of THIS object (zeroed once; the kernels restore the zero state). Per object
        # rather than per stream: a captured CUDA graph bakes these pointers in and may be replayed on any stream while
        # other callers use the per-stream scratch of the wrappers; one object must not run on two streams at once.
        self.ws = torch.zeros((int(self._lib.sp_mse_workspace_bytes()) + 7) // 8, dtype=torch.int64, device=dev)
        self.dws = torch.zeros(2, dtype=torch.int64, device=dev)

    def _checked(self, t, shape, name, dtype=torch.float32):
        """The raw-pointer calls below read ``t`` as a dense tensor of exactly this shape and dtype on
        this object's device: anything else would be an out-of-bounds read, so it raises instead."""
        if not isinstance(t, torch.Tensor) or t.device != self.device:
            raise RuntimeError("%s must be a tensor on %s (there is no CPU path)" % (name, self.device))
        if t.dtype != dtype or tuple(t.shape) != tuple(shape) or not t.is_contiguous():
            raise ValueError("%s must be a contiguous %s tensor of shape %s, got %s %s%s" % (
                name, dtype, tuple(shape), t.dtype, tuple(t.shape), "" if t.is_contiguous() else " (non-contiguous)"))
        return t

    def _maps(self, t, name):
        return self._checked(t, (self.batch, self.k, self.h, self.w), name)

    # each method enqueues exactly one kernel on the current stream of self.device
    def encode(self, joints):
        self._checked(joints, (self.batch, self.k, 3), "joints")
        with torch.cuda.device(self.device):
            _abi.check(self._lib.sp_encode_f32(joints.data_ptr(), self.targets.data_ptr(), self.weights.data_ptr(),
                                               self.batch, self.k, self.h, self.w, self.sigma,
                                               _abi.stream_ptr(self.device)))

    def loss_fwd_bwd(self, pred):
        self._maps(pred, "pred")
        with torch.cuda.device(self.device):
            stream = _abi.stream_ptr(self.device)
            ws = self.ws
            _abi.check_ws(self._lib.sp_mse_fwd_bwd_f32(pred.data_ptr(), self.targets.data_ptr(), self.weights.data_ptr(),
                                                       self.grad.data_ptr(), self.loss.data_ptr(), ws.data_ptr(),
                                                       ws.numel() * 8, self.batch, self.k, self.h * self.w, 1.0, 0, stream),
                          self.device, stream, self)

    def train_fused(self, joints, pred, with_acc=True):
        """encode + loss fwd/bwd (+ HeatMapAcc argmaxes) in one launch; targets never materialised."""
        if with_acc and self.pred_xy is None:
            self.pred_xy = torch.empty((self.batch, self.k, 2), dtype=torch.float32, device=self.device)
            self.label_xy = torch.empty_like(self.pred_xy)
        self._checked(joints, (self.batch, self.k, 3), "joints")
        self._maps(pred, "pred")
        with torch.cuda.device(self.device):
            stream = _abi.stream_ptr(self.device)
            ws = self.ws
            _abi.check_ws(self._lib.sp_encode_mse_fwd_bwd_f32(
                joints.data_ptr(), pred.data_ptr(), self.grad.data_ptr(), None, self.weights.data_ptr(),
                self.loss.data_ptr(), _abi.ptr(self.pred_xy) if with_acc else None,
                _abi.ptr(self.label_xy) if with_acc else None, ws.data_ptr(), ws.numel() * 8,
                self.batch, self.k, self.h, self.w, self.sigma, 1.0, stream), self.device, stream, self)

    def decode(self, pred, trans_inv, pred_flip=None, perm=None):
        self._maps(pred, "pred")
        if trans_inv is not None:
            self._checked(trans_inv, (self.batch, 2, 3), "trans_inv")
        if pred_flip is not None:
            self._maps(pred_flip, "pred_flip")
            self._checked(perm, (self.k,), "perm", torch.int32)
        with torch.cuda.device(self.device):
            stream = _abi.stream_ptr(self.device)
            ws = self.dws
            _abi.check_ws(self._lib.sp_decode_ws_f32(pred.data_ptr(), _abi.ptr(pred_flip), _abi.ptr(perm),
                                                     _abi.ptr(trans_inv), self.blur_w.data_ptr(), self.coords.data_ptr(),
                                                     self.maxval.data_ptr(), None, self.batch, self.k, self.h, self.w,
                                                     self.ksize, _abi.SP_DECODE_GAUSS_TAYLOR, ws.data_ptr(), ws.numel() * 8,
                                                     stream), self.device, stream, self)

    def step_one_launch(self, joints, pred, trans_inv, want_targets=True, want_grad=True, with_acc=False, want_decode=True):
        """encode + loss fwd/bwd (+ HeatMapAcc argmaxes) + GaussTaylor decode of ``pred`` in ONE launch
        (``sp_step_f32``): every map is staged in shared memory once, pred is read from HBM once and the
        targets are written but not read back. Same outputs as ``step`` (loss up to summation order)."""
        self._checked(joints, (self.batch, self.k, 3), "joints")
        self._maps(pred, "pred")
        if trans_inv is not None:
            self._checked(trans_inv, (self.batch, 2, 3), "trans_inv")
        if with_acc and self.pred_xy is None:
            self.pred_xy = torch.empty((self.batch, self.k, 2), dtype=torch.float32, device=self.device)
            self.label_xy = torch.empty_like(self.pred_xy)
        with torch.cuda.device(self.device):
            stream = _abi.stream_ptr(self.device)
            ws = self.ws
            _abi.check_ws(self._lib.sp_step_f32(
                joints.data_ptr(), pred.data_ptr(), _abi.ptr(trans_inv), self.blur_w.data_ptr(),
                self.targets.data_ptr() if want_targets else None, self.weights.data_ptr(),
                self.grad.data_ptr() if want_grad else None, self.loss.data_ptr(),
                self.coords.data_ptr() if want_decode else None, self.maxval.data_ptr() if want_decode else None,
                _abi.ptr(self.pred_xy) if with_acc else None,
                _abi.ptr(self.label_xy) if with_acc else None, ws.data_ptr(), ws.numel() * 8,
                self.batch, self.k, self.h, self.w, self.sigma, self.ksize, 1.0, stream), self.device, stream, self)
        return self.loss, self.coords, self.maxval

    def one_launch_supported(self):
        """``sp_step_f32`` takes W % 4 == 0, the reference's 11 x 11 blur and maps that fit in shared memory."""
        per_warp = 1536 + 8 * (((self.w + 1) & ~1) + ((self.h + 1) & ~1)) + 4 * self.h * self.w
        return self.w % 4 == 0 and self.ksize == 11 and per_warp <= 226 * 1024 - 2048

    VAL_DECODERS = {"gauss_taylor": _abi.SP_DECODE_GAUSS_TAYLOR, "basic": _abi.SP_DECODE_BASIC}

    @staticmethod
    def val_one_launch_supported(height, width, kernel_size, decoder):
        """``sp_val_step_f32`` takes W % 4 == 0 and maps that fit in shared memory, and for the GaussTaylor decoder
        the reference's 11 x 11 blur (the Basic decoder has no blur)."""
        per_warp = 1536 + 8 * (((width + 1) & ~1) + ((height + 1) & ~1)) + 4 * height * width
        blur_ok = decoder == "basic" or kernel_size == 11
        return width % 4 == 0 and blur_ok and per_warp <= 226 * 1024 - 2048

    def val_step(self, joints, pred, trans_inv, decoder="gauss_taylor"):
        """The body of every solver's ``val()`` on one batch of predicted heatmaps (no gradient): the loss, the
        ``HeatMapAcc`` value, the solver's decoder (``"gauss_taylor"``: the HRNet solver; ``"basic"``: the ResNet
        solvers) and the ``kps_to_dict_`` rows. One launch (``sp_val_step_f32``) where the shape allows, otherwise
        the stand-alone kernels with the same results (the loss up to its float64 summation order). Returns
        ``(loss, acc, rows)``, this object's buffers: 0-d loss and acc, ``rows`` [B, 3K+1] float32 on the device
        (``metrics.coco_eval.evaluate_person_rows`` takes them as they are, ``metrics.pose_metrics.rows_to_dicts``
        turns them into ``kps_to_dict_``'s dicts). ``coords`` / ``maxval`` hold the decoder's output as well."""
        if decoder not in self.VAL_DECODERS:
            raise ValueError("decoder must be one of %s, got %r" % (sorted(self.VAL_DECODERS), decoder))
        mode = self.VAL_DECODERS[decoder]
        self._checked(joints, (self.batch, self.k, 3), "joints")
        self._maps(pred, "pred")
        if trans_inv is not None:
            self._checked(trans_inv, (self.batch, 2, 3), "trans_inv")
        dev = self.device
        if self.pred_xy is None:
            self.pred_xy = torch.empty((self.batch, self.k, 2), dtype=torch.float32, device=dev)
            self.label_xy = torch.empty_like(self.pred_xy)
        if self.rows is None:
            self.rows = torch.empty((self.batch, 3 * self.k + 1), dtype=torch.float32, device=dev)
            self.acc = torch.empty((), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            stream = _abi.stream_ptr(dev)
            if self.val_one_launch_supported(self.h, self.w, self.ksize, decoder):
                ws = self._val_ws()
                _abi.check_ws(self._lib.sp_val_step_f32(
                    joints.data_ptr(), pred.data_ptr(), _abi.ptr(trans_inv), self.blur_w.data_ptr(), mode,
                    self.weights.data_ptr(), self.loss.data_ptr(), self.acc.data_ptr(), self.rows.data_ptr(),
                    self.coords.data_ptr(), self.maxval.data_ptr(), self.pred_xy.data_ptr(), self.label_xy.data_ptr(),
                    ws.data_ptr(), ws.numel() * 8, self.batch, self.k, self.h, self.w, self.sigma, self.ksize,
                    0.5, 10.0, stream), dev, stream, self)
                return self.loss, self.acc, self.rows
            self._val_composed(joints, pred, trans_inv, mode, stream)
        return self.loss, self.acc, self.rows

    def _val_ws(self):
        """``vws``: the workspace of ``val_step``, large enough for the one launch and for the composed loss kernel."""
        if self.vws is None:
            nbytes = max(int(self._lib.sp_val_step_workspace_bytes(self.batch, self.k)),
                         int(self._lib.sp_mse_acc_workspace_bytes(self.batch, self.k)))
            self.vws = torch.zeros((nbytes + 7) // 8, dtype=torch.int64, device=self.device)
        return self.vws

    def _val_composed(self, joints, pred, trans_inv, mode, stream):
        """``val_step`` as the stand-alone kernels: loss + HeatMapAcc, decoder, rows."""
        if self.w % 4 == 0:           # the fused loss kernel with its argmaxes, forward only, then the HeatMapAcc epilogue
            ws = self.ws
            _abi.check_ws(self._lib.sp_encode_mse_fwd_bwd_f32(
                joints.data_ptr(), pred.data_ptr(), None, None, self.weights.data_ptr(), self.loss.data_ptr(),
                self.pred_xy.data_ptr(), self.label_xy.data_ptr(), ws.data_ptr(), ws.numel() * 8,
                self.batch, self.k, self.h, self.w, self.sigma, 1.0, stream), self.device, stream, self)
            _abi.check(self._lib.sp_heatmap_acc_f32(self.pred_xy.data_ptr(), self.label_xy.data_ptr(), self.acc.data_ptr(),
                                                    self.batch, self.k, self.h, self.w, 0.5, 10.0, stream))
        else:                         # encode, then the forward loss with HeatMapAcc of the masked maps in the same pass
            self.encode(joints)
            ws = self._val_ws()
            _abi.check_ws(self._lib.sp_mse_acc_fwd_bwd(
                pred.data_ptr(), _abi.SP_DTYPE_F32, self.targets.data_ptr(), self.weights.data_ptr(), None,
                self.loss.data_ptr(), self.acc.data_ptr(), self.pred_xy.data_ptr(), self.label_xy.data_ptr(),
                ws.data_ptr(), ws.numel() * 8, self.batch, self.k, self.h, self.w, 1.0, None, 0.5, 10.0, 0, stream),
                self.device, stream, self)
        _abi.check_ws(self._lib.sp_decode_ws_f32(pred.data_ptr(), None, None, _abi.ptr(trans_inv), self.blur_w.data_ptr(),
                                                 self.coords.data_ptr(), self.maxval.data_ptr(), None, self.batch, self.k,
                                                 self.h, self.w, self.ksize, mode, self.dws.data_ptr(),
                                                 self.dws.numel() * 8, stream), self.device, stream, self)
        _abi.check(self._lib.sp_person_rows_f32(self.coords.data_ptr(), self.maxval.data_ptr(), self.rows.data_ptr(),
                                                self.batch, self.k, stream))

    def step(self, joints, pred, trans_inv, one_launch=None):
        """encode(joints), decode(pred), loss/grad(pred, targets, weights).

        ``one_launch`` (default: whenever the shape allows) runs the three as one kernel, ``sp_step_f32``.
        Otherwise 3 launches, in one of two orders. Large batches (targets do not fit in L2): encode,
        decode, loss -- the decode between the two kernels that touch ``targets`` measured 2.5 % faster
        than encode -> loss -> decode (1418 vs 1455 us for 8 x 1024 persons). Small batches (targets <=
        64 MB, e.g. the reference's batch 128 = 26.7 MB): decode, encode, loss -- the loss then finds the
        targets the encoder just wrote in the 126 MB L2 (scratch/l2_pairs.py). Same results either way."""
        if one_launch is None:
            one_launch = self.one_launch_supported()
        if one_launch:
            return self.step_one_launch(joints, pred, trans_inv)
        if self.targets.numel() * 4 <= (64 << 20):
            self.decode(pred, trans_inv)
            self.encode(joints)
            self.loss_fwd_bwd(pred)
        else:
            self.encode(joints)
            self.decode(pred, trans_inv)
            self.loss_fwd_bwd(pred)
        return self.loss, self.coords, self.maxval

    def capture(self, joints, pred, trans_inv, one_launch=None):
        """Capture ``step`` on these (static) input buffers into a CUDA graph and return ``replay``: a callable
        that re-runs the step with whatever the buffers hold at that moment, for the price of one graph launch
        instead of the Python -> ctypes -> launch path per kernel (the literal batch-128 configs are bound by
        exactly that). Outputs land in this object's buffers as usual."""
        return self._capture(lambda: self.step(joints, pred, trans_inv, one_launch))

    def capture_val(self, joints, pred, trans_inv, decoder="gauss_taylor"):
        """``capture`` for ``val_step``: the returned ``replay`` re-runs the validation step on whatever the input
        buffers hold; loss, acc and rows land in this object's buffers."""
        return self._capture(lambda: self.val_step(joints, pred, trans_inv, decoder))

    def _capture(self, run):
        stream = torch.cuda.Stream(self.device)
        stream.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(stream):
            for _ in range(2):                       # warm-up: workspace creation, attribute caches
                run()
        torch.cuda.current_stream(self.device).wait_stream(stream)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            run()
        self._graph = graph                          # keeps the captured buffers alive
        return graph.replay

    LAUNCHES_PER_STEP = 3          # the three stand-alone kernels (run_batches); step() via sp_step_f32 is 1


def run_batches(paths, inputs, after_decode=None):
    """One pass of the hot path over several batches: ``paths[i]`` is the ``HeatmapHotPath`` of batch i and
    ``inputs[i] = (joints, pred, trans_inv)``. Launches are grouped by kernel -- all decodes, then
    all encodes, then all losses -- because B200 pays ~5 us whenever two different kernels follow
    each other on a stream (8 x 1024 persons: 1367 us grouped, 1408 us interleaved, 1354 us = sum
    of the kernels timed alone; scratch/seq_step.py). ``after_decode`` is called once all decodes
    are enqueued (bench.py starts the NCCL all-gather of the keypoints there, so that it overlaps
    the encode and loss kernels). Same 3 launches per batch and the same results as ``step``."""
    for hp, (joints, pred, trans_inv) in zip(paths, inputs):
        hp.decode(pred, trans_inv)
    if after_decode is not None:
        after_decode()
    for hp, (joints, pred, trans_inv) in zip(paths, inputs):
        hp.encode(joints)
    for hp, (joints, pred, trans_inv) in zip(paths, inputs):
        hp.loss_fwd_bwd(pred)
