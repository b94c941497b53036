"""GPU: every entry point that takes a torch.max argmax or runs the HeatMapAcc epilogue (``sp_argmax.cuh``) against a
host reference, on maps built to sit where the kernels split a map.

The reference runs on the CPU and shares no code with the kernels: the masked products are ``float32(m * float(p))``
formed in float64 and rounded once (one product is exact in float64, so this is autocast's ``pred.mul(mask)`` for
float32, float16 and bfloat16 ``pred``); the argmax, its value and the ``heat_map_to_axis`` coordinates are
``torch.max(dim=-1)`` on the CPU (``O.argmax_index`` / ``O.argmax_coords``); HeatMapAcc is ``O.heat_map_acc`` and its
epilogue ``O.heat_map_acc_from_axes``. Everything is compared bit for bit -- the same NaN positions, the sign of zero
included. Coordinates the Gauss-Taylor step refines are left to the decoder tests (its step is ill-conditioned on these
noise maps); those it leaves at the argmax are compared bit for bit.

The catalogue puts equal maxima, NaN (quiet, sign-bit and payload patterns), infinities, all-zero maps of either sign,
subnormal maxima, products that overflow or become subnormal, and float32 neighbours that a 0.75 mask rounds to the
same product at the first and last element, on both sides of a quad (4 elements), of a 16-byte half-precision group (8),
of the 32-lane stride (128) and of the loss and fused-training chunk sizes the tuning overrides select, and across the
ranges of different CTAs. The HeatMapAcc lattice feeds every distinct (dx, dy) offset of a map size through the epilogue
with one joint per x-offset and one person per y-offset, so a single verdict that differs from torch.norm's changes
the returned accuracy."""
import contextlib
import functools
import os

import numpy as np
import pytest
import torch

from oracle import heatmap_oracle as O
from simple_pose_b200 import _abi
from test_heatmap_acc_norm_cpu import LATTICES, double_form, lattice_axis

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")

F32_NANS = (0x7FC00000, 0xFFC00000, 0x7FA12345, 0xFFF00001)        # quiet, sign-bit, payload (signalling), both
HALF_NANS = {torch.float16: (0x7E00, 0xFE00, 0x7C01, 0xFD55), torch.bfloat16: (0x7FC0, 0xFFC0, 0x7F81, 0xFFA5)}
MASKS = (1.0, 0.75, 2.0, 0.5, 0.0, -0.0, 1.0, 0.75)
SUB_MIN = np.float32(1.4e-45)                                         # smallest positive subnormal
ROUND_LO, ROUND_HI = np.float32(1.5) + np.float32(2 * 2.0 ** -23), np.float32(1.5) + np.float32(3 * 2.0 ** -23)
assert ROUND_LO < ROUND_HI and np.float32(0.75) * ROUND_LO == np.float32(0.75) * ROUND_HI


def eq(x, y):
    """Bit-equal up to NaN payloads: same NaN positions, identical other values (including the sign of zero)."""
    x, y = x.detach().cpu(), y.detach().cpu()
    if x.dtype != y.dtype or x.shape != y.shape:
        return False
    if not x.is_floating_point():
        return torch.equal(x, y)
    nx, ny = torch.isnan(x), torch.isnan(y)
    view = {torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}[x.dtype]
    return torch.equal(nx, ny) and torch.equal(x.masked_fill(nx, 0).view(view), y.masked_fill(ny, 0).view(view))


def diff(x, y):
    """Where two tensors differ (for assertion messages)."""
    x, y = x.detach().cpu(), y.detach().cpu()
    bad = (x != y) & ~(torch.isnan(x) & torch.isnan(y))
    idx = bad.nonzero()[:4].tolist()
    return "%d differ, first %s: got %s want %s" % (int(bad.sum()), idx, [x[tuple(i)].item() for i in idx],
                                                   [y[tuple(i)].item() for i in idx])


@contextlib.contextmanager
def tuning(env):
    os.environ.update(env)
    _abi.reload_tuning()
    try:
        yield
    finally:
        for key in env:
            del os.environ[key]
        _abi.reload_tuning()


# ------------------------------------------------------------------------------------------------ the catalogue
def boundaries(hw):
    """Flat positions where the kernels split a map: first / last element, quad, half-precision group, lane stride,
    the loss chunks (8, 48, 192 quads) and the fused-training chunks (64, 192 quads), the middle."""
    pos = {0, hw - 1, hw // 2 - 1, hw // 2}
    for edge in (4, 8, 128, 32, 192, 256, 768, 1536, 2304, 3072, 8192):
        pos.update((edge - 1, edge))
    return sorted(p for p in pos if 0 <= p < hw)


CASES = ("tie", "tie3", "nan_before", "nan_after", "all_nan", "two_nan", "two_pinf", "all_ninf", "ninf_nan", "zeros",
         "zeros_neg_first", "sub_max", "sub_tie", "neg_sub_vs_negzero", "overflow", "sub_product", "round_tie",
         "all_negative", "benign")
FINITE_CASES = ("tie", "tie3", "zeros", "zeros_neg_first", "sub_max", "sub_tie", "neg_sub_vs_negzero", "sub_product",
                "round_tie", "all_negative", "benign")


def special_map(case, hw, rng):
    """One map of the catalogue: float32 values, the mask it needs (None: any) and the positions it set to NaN."""
    pos = boundaries(hw)
    a, b, c = sorted(rng.choice(pos, size=3, replace=len(pos) < 3))
    if a == b:
        a, b = 0, hw - 1
    v = rng.uniform(0.0, 1.0, hw).astype(np.float32)
    mask, nan_at = None, []
    if case == "tie":
        v[a] = v[b] = 3.0
    elif case == "tie3":
        v[a] = v[b] = v[c] = np.float32(2.5)
        v[rng.integers(0, hw)] = np.float32(2.4999998)
    elif case == "nan_before":
        nan_at, v[b] = [a], 5.0
    elif case == "nan_after":
        v[a], nan_at = 5.0, [b]
    elif case == "all_nan":
        nan_at = list(range(hw))
    elif case == "two_nan":
        nan_at = [a, b]
    elif case == "two_pinf":
        v[a] = v[b] = np.inf
    elif case == "all_ninf":
        v[:] = -np.inf
    elif case == "ninf_nan":
        v[:] = -np.inf
        nan_at = [b]
    elif case in ("zeros", "zeros_neg_first"):
        v[:] = np.where(rng.uniform(size=hw) < 0.5, np.float32(-0.0), np.float32(0.0))
        v[0] = np.float32(-0.0) if case == "zeros_neg_first" else np.float32(0.0)
        mask = 1.0
    elif case == "sub_max":
        v[:] = np.where(rng.uniform(size=hw) < 0.5, np.float32(-1.0), np.float32(0.0))
        v[b] = SUB_MIN
        mask = 1.0
    elif case == "sub_tie":
        v[:] = SUB_MIN
        v[a] = v[b] = SUB_MIN * np.float32(3)
        mask = 1.0
    elif case == "neg_sub_vs_negzero":
        v[:] = -1.0
        v[a] = -SUB_MIN
        v[b] = np.float32(-0.0)
        mask = 1.0
    elif case == "overflow":
        v[a] = v[b] = np.float32(3e38)
        v[c] = np.float32(1e38)
        mask = 2.0
    elif case == "sub_product":
        v[:] = -v
        v[b] = np.float32(2e-38)                     # normal; times 0.5 a subnormal
        v[a] = np.float32(1e-38)
        mask = 0.5
    elif case == "round_tie":
        v[a], v[b] = ROUND_LO, ROUND_HI              # equal after the 0.75 mask: the earlier, smaller one wins
        mask = 0.75
    elif case == "all_negative":
        v[:] = -v - 1.0
        v[b] = -0.5
    return v, mask, nan_at


@functools.lru_cache(maxsize=6)
def catalogue(b, k, h, w, seed, dtype=torch.float32, cases=CASES):
    """[B,K,H,W] maps in ``dtype`` and a [B,K] float32 mask: map i is case ``cases[i % len]`` with mask
    ``MASKS[(i // len) % len(MASKS)]`` unless the case needs its own."""
    rng = np.random.default_rng(seed)
    n, hw = b * k, h * w
    vals = np.empty((n, hw), np.float32)
    mask = np.empty(n, np.float32)
    nans = []
    for i in range(n):
        v, m, nan_at = special_map(cases[i % len(cases)], hw, rng)
        vals[i] = v
        mask[i] = MASKS[(i // len(cases)) % len(MASKS)] if m is None else m
        nans += [(i, j) for j in nan_at]
    maps = torch.from_numpy(vals).to(dtype)
    if nans:
        rows, cols = torch.tensor(nans).T
        patterns = F32_NANS if dtype == torch.float32 else HALF_NANS[dtype]
        bits = torch.tensor([patterns[(r + c) % len(patterns)] for r, c in nans], dtype=torch.int64)
        view = maps.view(torch.int32 if dtype == torch.float32 else torch.int16)
        half = 1 << (8 * view.element_size() - 1)
        view[rows, cols] = ((bits + half) % (2 * half) - half).to(view.dtype)          # the patterns as signed integers
    return maps.reshape(b, k, h, w), torch.from_numpy(mask).reshape(b, k)


def masked(maps, mask):
    """float32(m * float(p)), formed in float64 and rounded once."""
    return (maps.double() * mask.double()[..., None, None]).float()


def reference(maps, mask=None):
    """(heat_map_to_axis coordinates [B,K,2], max values [B,K,1], flat argmax [B,K]) of the (masked) maps."""
    x = maps.float() if mask is None else masked(maps, mask)
    xy, peak = O.argmax_coords(x)
    return xy, peak, O.argmax_index(x)


def joints_for(mask, h, w, seed):
    """Joints well inside the map (never culled: the encoder's weights are the visibilities) with vis = mask."""
    g = torch.Generator().manual_seed(seed)
    b, k = mask.shape
    x = 2.0 + torch.rand(b, k, generator=g) * (w - 5)
    y = 2.0 + torch.rand(b, k, generator=g) * (h - 5)
    return torch.stack([x, y, mask], -1)


def encoder_labels(joints, h, w):
    t, wt = O.encode_batch(joints.numpy(), shape=(w, h))
    return O.argmax_coords(torch.from_numpy(t) * torch.from_numpy(wt)[..., None, None])[0]


# ------------------------------------------------------------------------------------------------ decoders
def decode(hm, mode, hf=None, tinv=None, ksize=11):
    from simple_pose_b200.metrics.pose_metrics import GaussTaylorKeyPointDecoder
    b, k, h, w = hm.shape
    dec = GaussTaylorKeyPointDecoder(num_joints=k)
    perm = dec._perm_on(DEV, k, None) if hf is not None else None
    coords = torch.empty(b, k, 2, device=DEV)
    maxval = torch.empty(b, k, 1, device=DEV)
    index = torch.empty(b, k, dtype=torch.int32, device=DEV)
    ws = torch.zeros(2, dtype=torch.int64, device=DEV)
    _abi.check(_abi.lib().sp_decode_ws_f32(hm.data_ptr(), _abi.ptr(hf), _abi.ptr(perm), _abi.ptr(tinv),
                                           dec._weights_on(DEV).data_ptr(), coords.data_ptr(), maxval.data_ptr(),
                                           index.data_ptr(), b, k, h, w, ksize, mode, ws.data_ptr(), 16,
                                           _abi.stream_ptr(DEV)))
    torch.cuda.synchronize()
    assert int(ws.abs().sum()) == 0
    return coords.cpu(), maxval.cpu(), index.cpu().long()


def assert_index_derived(got, want, xy):
    """Gauss-Taylor coordinates the reference leaves at the argmax (no Taylor step: a peak near the border, a maximum
    <= 0) equal the argmax coordinates bit for bit. Refined ones are the decoder tests' business: on these noise maps
    the step is ill-conditioned."""
    same = (want == xy).all(-1)
    assert eq(got[same], xy[same]), diff(got[same], xy[same])


DECODE_ENVS = [{}, {"SP_DECODE_FORCE_GENERIC": "1"}, {"SP_DECODE_WARPS": "1", "SP_DECODE_STAGES": "1"},
               {"SP_DECODE_WARPS": "3", "SP_DECODE_STAGES": "4"}, {"SP_DECODE_GRID_WIDE": "1", "SP_DECODE_STATIC_PCT": "40"}]


@pytest.mark.parametrize("env", DECODE_ENVS)
@pytest.mark.parametrize("b,hw", [(12, (64, 48)), (4, (96, 72)), (3, (9, 7)), (160, (64, 48))])
def test_decode_argmax_and_values(env, b, hw):
    """sp_decode_ws_f32 in every mode: the flat argmax and the max value bit for bit; ARGMAX and BASIC coordinates bit
    for bit, and the Gauss-Taylor coordinates the step leaves at the argmax."""
    h, w = hw
    hm, _ = catalogue(b, 17, h, w, seed=b + h)
    xy, peak, idx = reference(hm)
    ident = torch.tensor([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]).expand(b, 2, 3).contiguous()
    hm_d, ident_d = hm.to(DEV), ident.to(DEV)
    with tuning(env):
        got = {mode: decode(hm_d, mode, tinv=None if mode == _abi.SP_DECODE_ARGMAX else ident_d)
               for mode in (_abi.SP_DECODE_ARGMAX, _abi.SP_DECODE_BASIC, _abi.SP_DECODE_GAUSS_TAYLOR,
                            _abi.SP_DECODE_DARK_ORIGINAL)}
    for mode, (c, m, i) in got.items():
        assert torch.equal(i, idx), (mode, diff(i, idx))
        assert eq(m, peak), (mode, diff(m, peak))
    assert eq(got[_abi.SP_DECODE_ARGMAX][0], xy), diff(got[_abi.SP_DECODE_ARGMAX][0], xy)
    basic, _ = O.basic_decode(hm, ident)
    assert eq(got[_abi.SP_DECODE_BASIC][0], basic), diff(got[_abi.SP_DECODE_BASIC][0], basic)
    gt, _ = O.gauss_taylor_decode(hm, ident)
    assert_index_derived(got[_abi.SP_DECODE_GAUSS_TAYLOR][0], gt, xy)


@pytest.mark.parametrize("env", DECODE_ENVS[:2] + DECODE_ENVS[4:])
@pytest.mark.parametrize("b,hw", [(8, (64, 48)), (3, (96, 72))])
def test_flip_decode_argmax(env, b, hw):
    """Flip test: the argmax and value of the flip average (O.flip_average) bit for bit."""
    h, w = hw
    hm, _ = catalogue(b, 17, h, w, seed=3 * b)
    hf, _ = catalogue(b, 17, h, w, seed=3 * b + 1)
    avg = O.flip_average(hm, hf)
    xy, peak, idx = reference(avg)
    with tuning(env):
        c, m, i = decode(hm.to(DEV), _abi.SP_DECODE_GAUSS_TAYLOR, hf=hf.to(DEV))
    assert torch.equal(i, idx), diff(i, idx)
    assert eq(m, peak), diff(m, peak)
    assert_index_derived(c, O.gauss_taylor_decode(avg, None, return_heatmap_space=True)[0], xy)


@pytest.mark.parametrize("thresh,frac", [(0.5, 10.), (1.25, 8.), (0.25, 4.)])
@pytest.mark.parametrize("b,hw", [(20, (64, 48)), (6, (100, 100)), (4, (9, 7))])
def test_heatmap_acc(thresh, frac, b, hw):
    """HeatMapAcc(distance_thresh, norm_frac)(predicts, targets): two ARGMAX decodes and sp_heatmap_acc_f32."""
    from simple_pose_b200.metrics.pose_metrics import HeatMapAcc
    h, w = hw
    pred, _ = catalogue(b, 17, h, w, seed=5 * b)
    tgt, _ = catalogue(b, 17, h, w, seed=5 * b + 1, cases=CASES[::-1])
    got = HeatMapAcc(thresh, frac)(pred.to(DEV), tgt.to(DEV))
    want = O.heat_map_acc(pred, tgt, thresh, frac)
    assert eq(got, want), (got.item(), want.item())


# ------------------------------------------------------------------------------------------------ loss kernels
def check_loss_acc(pred, tgt, mask, grad=True, skip_masked=False, thresh=0.5, frac=10.):
    from simple_pose_b200.processors.loss import mse_forward_backward
    b, k, h, w = pred.shape
    pxy, lxy = (torch.full((b, k, 2), -7.0, device=DEV) for _ in range(2))
    _, _, acc = mse_forward_backward(pred.to(DEV), tgt.to(DEV), mask.to(DEV), need_grad=grad, skip_masked=skip_masked,
                                     want_acc=True, distance_thresh=thresh, norm_frac=frac, axes_out=(pxy, lxy))
    torch.cuda.synchronize()
    want_p, want_l = reference(pred, mask)[0], reference(tgt, mask)[0]
    assert eq(pxy, want_p), diff(pxy, want_p)
    assert eq(lxy, want_l), diff(lxy, want_l)
    want_acc = O.heat_map_acc_from_axes(want_p, want_l, h, w, thresh, frac)
    assert eq(acc, want_acc), (acc.item(), want_acc.item())


LOSS_ENVS = [{}, {"SP_LOSS_WARPS": "1"}, {"SP_LOSS_WARPS": "7", "SP_LOSS_RING": "1"}, {"SP_LOSS_CHUNK_QUADS": "8"},
             {"SP_LOSS_CHUNK_QUADS": "48", "SP_LOSS_WARPS": "16"}, {"SP_LOSS_CHUNK_QUADS": "2048"},
             {"SP_LOSS_FORCE_LDG": "1"}]


@pytest.mark.parametrize("env", LOSS_ENVS)
@pytest.mark.parametrize("b,hw", [(40, (64, 48)), (9, (96, 72)), (300, (64, 48))])
def test_mse_acc_float32(env, b, hw):
    """sp_mse_acc_fwd_bwd, float32: the ring kernel under every chunk / warp / ring split, and the plain-load kernel,
    with and without the gradient."""
    h, w = hw
    pred, mask = catalogue(b, 17, h, w, seed=b)
    tgt, _ = catalogue(b, 17, h, w, seed=b + 1, cases=CASES[::-1])
    with tuning(env):
        for grad in (True, False):
            check_loss_acc(pred, tgt, mask, grad)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("b,hw", [(40, (64, 48)), (24, (10, 6)), (12, (9, 7))])
def test_mse_acc_half_precision(dtype, b, hw):
    """float16 / bfloat16 predictions: the 16-byte group loads (HW % 8 == 0) and the scalar loads (HW % 8 != 0),
    sign-bit and payload NaN patterns of the narrow types included."""
    h, w = hw
    pred, mask = catalogue(b, 17, h, w, seed=2 * b, dtype=dtype)
    tgt, _ = catalogue(b, 17, h, w, seed=2 * b + 1, cases=CASES[::-1])
    for grad in (True, False):
        check_loss_acc(pred, tgt, mask, grad)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_mse_acc_skip_masked(dtype):
    """SP_MSE_SKIP_MASKED on finite inputs: masked-out maps are not read and give (0, 0), as their products would."""
    pred, mask = catalogue(60, 17, 64, 48, seed=8, dtype=dtype, cases=FINITE_CASES)
    tgt, _ = catalogue(60, 17, 64, 48, seed=9, cases=FINITE_CASES[::-1])
    check_loss_acc(pred, tgt, mask, grad=True, skip_masked=True)


# ------------------------------------------------------------------------------------------------ fused kernels
def check_pred_axes(pxy, lxy, weights, pred, mask, joints, h, w):
    want_p = reference(pred, mask)[0]
    assert eq(weights, mask), diff(weights, mask)
    assert eq(pxy, want_p), diff(pxy, want_p)
    want_l = encoder_labels(joints, h, w)
    assert eq(lxy, want_l), diff(lxy, want_l)
    return want_p, want_l


TRAIN_ENVS = [{}, {"SP_TRAIN_NO_TILE": "1"}, {"SP_TRAIN_FORCE_LDG": "1"}, {"SP_TRAIN_CHUNK_QUADS": "64", "SP_TRAIN_RING": "4"},
              {"SP_TRAIN_WARPS": "3", "SP_TRAIN_RING": "2"}, {"SP_TRAIN_NO_TILE": "1", "SP_TRAIN_RING": "3", "SP_TRAIN_WARPS": "5"}]


@pytest.mark.parametrize("env", TRAIN_ENVS)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("b,hw", [(40, (64, 48)), (6, (96, 72))])
def test_encode_mse_acc(env, dtype, b, hw):
    """sp_encode_mse_fwd_bwd(_f32): the period-tiled kernel, the TMA ring and the plain-load kernel; pred_xy against the
    reference, label_xy against the oracle encoder's targets, and EncodeJointsMSELoss's acc against the epilogue."""
    from simple_pose_b200.processors.loss import EncodeJointsMSELoss, encode_mse_forward_backward
    h, w = hw
    pred, mask = catalogue(b, 17, h, w, seed=7 * b, dtype=dtype)
    joints = joints_for(mask, h, w, seed=b)
    with tuning(env):
        for want_targets, grad in ((False, True), (True, True), (False, False)):
            out = encode_mse_forward_backward(joints.to(DEV), pred.to(DEV), need_grad=grad, want_targets=want_targets,
                                              want_axes=True)
            torch.cuda.synchronize()
            want_p, want_l = check_pred_axes(out["pred_xy"], out["label_xy"], out["weights"], pred, mask, joints, h, w)
        crit = EncodeJointsMSELoss(with_acc=True, distance_thresh=1.25, norm_frac=8.)
        with torch.no_grad():
            _, acc = crit(pred.to(DEV), joints.to(DEV))
    want = O.heat_map_acc_from_axes(want_p, want_l, h, w, 1.25, 8.)
    assert eq(acc, want), (acc.item(), want.item())


STEP_ENVS = [{}, {"SP_STEP_STATIC_PCT": "0"}, {"SP_STEP_STATIC_PCT": "100"}, {"SP_STEP_WARPS": "3", "SP_STEP_STATIC_PCT": "30"},
             {"SP_STEP_WARPS": "5"}]


def identity(b):
    return torch.tensor([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]).expand(b, 2, 3).contiguous()


@pytest.mark.parametrize("env", STEP_ENVS)
@pytest.mark.parametrize("b,hw", [(20, (64, 48)), (520, (64, 48)), (7, (96, 72))])
def test_step(env, b, hw):
    """sp_step_f32 with the HeatMapAcc argmaxes: decode max values and flat-argmax coordinates, pred_xy, label_xy."""
    from simple_pose_b200.pipeline import HeatmapHotPath
    h, w = hw
    pred, mask = catalogue(b, 17, h, w, seed=11 * b)
    joints = joints_for(mask, h, w, seed=b + 1)
    hp = HeatmapHotPath(b, 17, h, w, device=DEV)
    with tuning(env):
        hp.step_one_launch(joints.to(DEV), pred.to(DEV), identity(b).to(DEV), with_acc=True)
        torch.cuda.synchronize()
    xy, peak, _ = reference(pred)
    assert eq(hp.maxval, peak), diff(hp.maxval, peak)
    assert_index_derived(hp.coords.cpu(), O.gauss_taylor_decode(pred, identity(b))[0], xy)
    check_pred_axes(hp.pred_xy, hp.label_xy, hp.weights, pred, mask, joints, h, w)


def val_step(hp, joints, pred, tinv, decoder, thresh=0.5, frac=10.):
    """HeatmapHotPath.val_step's one launch with HeatMapAcc's two constructor arguments."""
    assert hp.val_one_launch_supported(hp.h, hp.w, hp.ksize, decoder)
    b, k = hp.batch, hp.k
    hp.pred_xy, hp.label_xy = torch.empty(b, k, 2, device=DEV), torch.empty(b, k, 2, device=DEV)
    hp.rows, hp.acc = torch.empty(b, 3 * k + 1, device=DEV), torch.empty((), device=DEV)
    ws = hp._val_ws()
    _abi.check(hp._lib.sp_val_step_f32(
        joints.data_ptr(), pred.data_ptr(), _abi.ptr(tinv), hp.blur_w.data_ptr(), hp.VAL_DECODERS[decoder],
        hp.weights.data_ptr(), hp.loss.data_ptr(), hp.acc.data_ptr(), hp.rows.data_ptr(), hp.coords.data_ptr(),
        hp.maxval.data_ptr(), hp.pred_xy.data_ptr(), hp.label_xy.data_ptr(), ws.data_ptr(), ws.numel() * 8, b, k,
        hp.h, hp.w, hp.sigma, hp.ksize, thresh, frac, _abi.stream_ptr(DEV)))
    torch.cuda.synchronize()


@pytest.mark.parametrize("env", STEP_ENVS[:1] + STEP_ENVS[3:])
@pytest.mark.parametrize("decoder", ["gauss_taylor", "basic"])
@pytest.mark.parametrize("b,hw", [(20, (64, 48)), (1100, (64, 48)), (5, (96, 72))])
def test_val_step(env, decoder, b, hw):
    """sp_val_step_f32, both decoders: acc, pred_xy, label_xy, max values and the conf column of the rows."""
    from simple_pose_b200.pipeline import HeatmapHotPath
    h, w = hw
    pred, mask = catalogue(b, 17, h, w, seed=13 * b)
    joints = joints_for(mask, h, w, seed=b + 2)
    hp = HeatmapHotPath(b, 17, h, w, device=DEV)
    with tuning(env):
        val_step(hp, joints.to(DEV), pred.to(DEV), identity(b).to(DEV), decoder)
    xy, peak, _ = reference(pred)
    assert eq(hp.maxval, peak), diff(hp.maxval, peak)
    assert eq(hp.rows[:, 2:3 * 17:3], peak[..., 0]), diff(hp.rows[:, 2:3 * 17:3], peak[..., 0])
    if decoder == "basic":
        want = O.basic_decode(pred, identity(b))[0]
        assert eq(hp.coords, want), diff(hp.coords, want)
    else:
        assert_index_derived(hp.coords.cpu(), O.gauss_taylor_decode(pred, identity(b))[0], xy)
    want_p, want_l = check_pred_axes(hp.pred_xy, hp.label_xy, hp.weights, pred, mask, joints, h, w)
    want = O.heat_map_acc_from_axes(want_p, want_l, h, w)
    assert eq(hp.acc, want), (hp.acc.item(), want.item())


# ------------------------------------------------------------------------------------------------ HeatMapAcc lattice
@pytest.mark.parametrize("h,w,thresh,frac", LATTICES)
def test_heatmap_acc_lattice(h, w, thresh, frac):
    """Every distinct (dx, dy) offset of an h x w map through sp_heatmap_acc_f32, one joint per x-offset and one person
    per y-offset, 32 x 32 at a time, plus a joint whose labels sit on x = 1, a person whose labels sit on y = 1 and a
    person whose predictions were zeroed (max <= 0): the accuracy equals the oracle epilogue's bits in every call."""
    from simple_pose_b200.metrics.pose_metrics import heatmap_acc_from_axes
    _, px, lx = lattice_axis(w, frac)
    _, py, ly = lattice_axis(h, frac)
    step = 32
    results = []
    for i in range(0, len(px), step):
        for j in range(0, len(py), step):
            xs_p, xs_l = px[i:i + step].float(), lx[i:i + step].float()
            ys_p, ys_l = py[j:j + step].float(), ly[j:j + step].float()
            k, b = len(xs_p) + 1, len(ys_p) + 2
            pred = torch.zeros(b, k, 2)
            label = torch.zeros(b, k, 2)
            pred[:len(ys_p), :k - 1, 0], pred[:len(ys_p), :k - 1, 1] = xs_p[None, :], ys_p[:, None]
            label[:len(ys_p), :k - 1, 0], label[:len(ys_p), :k - 1, 1] = xs_l[None, :], ys_l[:, None]
            label[:, k - 1] = torch.tensor([1.0, 5.0])          # x = 1: not counted
            pred[:, k - 1] = pred[:, 0]
            label[b - 2] = label[0]
            label[b - 2, :, 1] = 1.0                          # y = 1: not counted
            pred[b - 2] = pred[0]
            label[b - 1] = label[0]                           # zeroed predictions against valid labels
            got = heatmap_acc_from_axes(pred.to(DEV), label.to(DEV), h, w, thresh, frac)
            results.append((got, O.heat_map_acc_from_axes(pred, label, h, w, thresh, frac), i, j))
    torch.cuda.synchronize()
    bad = [(i, j, g.item(), r.item()) for g, r, i, j in results if not eq(g, r)]
    assert not bad, "%d of %d calls differ, first %s" % (len(bad), len(results), bad[:3])


# (H, W, distance_thresh, norm_frac, pred (x, y), label (x, y)): torch.norm and a double-precision sum put these pairs
# on different sides of the threshold
FLIPPING_PAIRS = [(100, 100, 0.5, 10., (0, 3), (3, 7)), (65, 52, 0.5, 10., (5, 0), (6, 3)),
                  (30, 40, 0.5, 4., (0, 4), (3, 7)), (96, 72, 1.25, 8., (0, 16), (9, 25))]


def planted(h, w, p, l, dtype, seed):
    """Two persons x 17 joints of smooth maps: joint 0 of person 0 peaks at p (prediction) and l (target); every other
    prediction peaks where its target does. Returns pred (dtype), targets, mask and joints."""
    g = torch.Generator().manual_seed(seed)
    b, k = 2, 17
    joints = torch.ones(b, k, 3)
    joints[..., 0] = torch.randint(2, w - 2, (b, k), generator=g).float()
    joints[..., 1] = torch.randint(2, h - 2, (b, k), generator=g).float()
    joints[0, 0, :2] = torch.tensor(l, dtype=torch.float32)
    t, wt = O.encode_batch(joints.numpy(), shape=(w, h))
    pj = joints.clone()
    pj[0, 0, :2] = torch.tensor(p, dtype=torch.float32)
    pred = torch.from_numpy(O.encode_batch(pj.numpy(), shape=(w, h))[0]) * 0.9 + 0.05 * torch.rand(b, k, h, w, generator=g)
    pred[0, 0, p[1], p[0]] = 2.0
    return pred.to(dtype), torch.from_numpy(t), torch.from_numpy(wt), joints


@pytest.mark.parametrize("h,w,thresh,frac,p,l", FLIPPING_PAIRS)
def test_planted_flipping_pair(h, w, thresh, frac, p, l):
    """One pair whose verdict torch.norm and the double-precision form disagree on, planted in real maps and run through
    every entry point that returns HeatMapAcc with the pair's settings: JointsMSELoss(with_acc=True) in float32, float16
    and bfloat16, EncodeJointsMSELoss, HeatMapAcc and the one-launch val_step. Each equals the oracle."""
    from simple_pose_b200.metrics.pose_metrics import HeatMapAcc
    from simple_pose_b200.pipeline import HeatmapHotPath
    from simple_pose_b200.processors.loss import EncodeJointsMSELoss, JointsMSELoss
    norm = torch.tensor([w, h], dtype=torch.float) / frac
    d = torch.tensor([p], dtype=torch.float) / norm - torch.tensor([l], dtype=torch.float) / norm
    assert bool(torch.norm(d, dim=-1)[0] < thresh) != bool(double_form(d)[0] < thresh)
    for dtype in (torch.float32, torch.float16, torch.bfloat16):
        pred, tgt, mask, joints = planted(h, w, p, l, dtype, seed=h + w)
        want = O.heat_map_acc(masked(pred, mask), masked(tgt, mask), thresh, frac)
        crit = JointsMSELoss(with_acc=True, distance_thresh=thresh, norm_frac=frac)
        with torch.no_grad():
            _, acc = crit(pred.to(DEV), tgt.to(DEV), mask.to(DEV))
        assert eq(acc, want), ("JointsMSELoss", dtype, acc.item(), want.item())
        if w % 4 == 0:
            ecrit = EncodeJointsMSELoss(with_acc=True, distance_thresh=thresh, norm_frac=frac)
            with torch.no_grad():
                _, acc = ecrit(pred.to(DEV), joints.to(DEV))
            assert eq(acc, want), ("EncodeJointsMSELoss", dtype, acc.item(), want.item())
    pred, tgt, mask, joints = planted(h, w, p, l, torch.float32, seed=h + w)
    want = O.heat_map_acc(pred, tgt, thresh, frac)
    acc = HeatMapAcc(thresh, frac)(pred.to(DEV), tgt.to(DEV))
    assert eq(acc, want), ("HeatMapAcc", acc.item(), want.item())
    hp = HeatmapHotPath(2, 17, h, w, device=DEV)
    for decoder in ("gauss_taylor", "basic"):
        val_step(hp, joints.to(DEV), pred.to(DEV), None, decoder, thresh, frac)
        assert eq(hp.acc, want), ("val_step", decoder, hp.acc.item(), want.item())
    if (thresh, frac) == (0.5, 10.):                        # HeatmapHotPath.val_step runs HeatMapAcc's defaults
        _, acc, _ = hp.val_step(joints.to(DEV), pred.to(DEV), None, "basic")
        assert eq(acc, want), ("HeatmapHotPath.val_step", acc.item(), want.item())
