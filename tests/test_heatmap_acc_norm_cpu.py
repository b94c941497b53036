"""CPU: the float32 distance HeatMapAcc's CUDA epilogue (``sp_arg::heatmap_acc_block``) computes is what the oracle's
``torch.norm(p / norm - t / norm, dim=-1)`` returns, on every distinct (dx, dy) offset of whole map lattices.

The kernel evaluates ``sqrtf(fmaf(dy, dy, dx * dx))``, every step correctly rounded in float32, because that is what
torch's CPU kernel returns for a pair of float32 values. Nothing in torch documents it, so this pins it: a torch
release that sums the squares another way (in double, or without the fused multiply-add) fails here, and the kernel
would have to follow. The lattices are the map sizes and HeatMapAcc settings at which the two forms disagree on a
verdict (the offsets land on the threshold), and the defaults at 64 x 48 and 96 x 72. ``lattice_axis`` also feeds the
GPU lattice test (tests/test_gpu_argmax_reference.py)."""
import numpy as np
import pytest
import torch

# (H, W, distance_thresh, norm_frac)
LATTICES = [(100, 100, 0.5, 10.), (65, 52, 0.5, 10.), (30, 40, 0.5, 4.), (96, 72, 1.25, 8.), (64, 48, 0.5, 10.),
            (96, 72, 0.5, 10.), (64, 48, 0.25, 10.), (48, 64, 1.0, 6.), (17, 17, 0.3, 5.)]


def lattice_axis(n, norm_frac):
    """Distinct float32 offsets p / norm - l / norm along an axis of n pixels (norm = float32(n) / norm_frac, as the
    oracle's ``tensor([W, H]) / norm_frac``) over every prediction p in [0, n) and label l in [2, n) (HeatMapAcc only
    counts labels with x > 1 and y > 1). Returns (offsets float32 [D], p int64 [D], l int64 [D]): one (p, l) pair that
    gives each offset."""
    norm = torch.tensor([float(n)], dtype=torch.float32) / norm_frac
    xs = torch.arange(n, dtype=torch.float32)
    d = (xs[:, None] / norm) - (xs[None, 2:] / norm)
    vals, first = np.unique(d.numpy().reshape(-1), return_index=True)
    p, l = np.divmod(first, n - 2)
    return torch.from_numpy(vals), torch.from_numpy(p), torch.from_numpy(l + 2)


def lattice_offsets(h, w, norm_frac):
    """Every distinct (dx, dy) offset of an h x w map, float32 [N, 2]."""
    dx, _, _ = lattice_axis(w, norm_frac)
    dy, _, _ = lattice_axis(h, norm_frac)
    return torch.stack(torch.broadcast_tensors(dx[:, None], dy[None, :]), -1).reshape(-1, 2).contiguous()


def fma_sqrt_f32(d):
    """sqrtf(fmaf(dy, dy, dx * dx)) with exactly one rounding per step. dx * dx is a float32 product; dy * dy + s is
    exact in float64 as an unevaluated sum hi + lo (both products have at most 48 significant bits; TwoSum gives the
    error of the float64 addition), and hi + lo is rounded to float32 once: rounding hi alone is correct unless hi is a
    float32 midpoint, where the sign of lo decides."""
    dx = d[:, 0].numpy().astype(np.float32)
    dy = d[:, 1].numpy().astype(np.float32)
    s = (dx * dx).astype(np.float64)                   # float32 product, then exact in float64
    y2 = dy.astype(np.float64) * dy.astype(np.float64)  # exact
    hi = y2 + s
    bb = hi - y2
    lo = (y2 - (hi - bb)) + (s - bb)                   # TwoSum: hi + lo == y2 + s exactly
    r = hi.astype(np.float32)                          # round to nearest even
    below = np.where(r.astype(np.float64) <= hi, r, np.nextafter(r, np.float32(-np.inf)))   # float32 neighbours of hi
    above = np.nextafter(below, np.float32(np.inf))
    mid = (below.astype(np.float64) + above.astype(np.float64)) / 2       # exact in float64
    r = np.where((hi == mid) & (lo > 0), above, np.where((hi == mid) & (lo < 0), below, r))
    return torch.from_numpy(np.sqrt(r.astype(np.float32)))


def double_form(d):
    """The distance the kernel computed before: float(sqrt(double(dx)^2 + double(dy)^2))."""
    dd = d.double()
    return torch.sqrt(dd[:, 0] * dd[:, 0] + dd[:, 1] * dd[:, 1]).float()


@pytest.mark.parametrize("h,w,thresh,frac", LATTICES)
def test_torch_norm_is_float32_sqrt_of_fma(h, w, thresh, frac):
    d = lattice_offsets(h, w, frac)
    want = fma_sqrt_f32(d)
    assert torch.equal(torch.norm(d, dim=-1), want)
    # the layouts the oracle and the GPU lattice test evaluate: [B, K, 2] tables
    for k in (1, 17, 64):
        n = d.shape[0] // k * k
        assert torch.equal(torch.norm(d[:n].reshape(-1, k, 2), dim=-1).reshape(-1), want[:n])
    assert torch.equal(torch.norm(d[:51].reshape(3, 17, 2), dim=-1).reshape(-1), want[:51])


def test_the_lattices_tell_the_two_forms_apart():
    """The double-precision form differs from torch.norm in the last bit on these lattices, and at 100 x 100 with the
    defaults some of those offsets straddle the threshold: a kernel that still summed in double would fail the GPU
    lattice test there."""
    d = lattice_offsets(64, 48, 10.)
    assert int((double_form(d) != torch.norm(d, dim=-1)).sum()) > 1000
    d = lattice_offsets(100, 100, 10.)
    t = torch.norm(d, dim=-1)
    assert int(((t < 0.5) != (double_form(d) < 0.5)).sum()) > 0


def test_fma_rounding_helper_rounds_once():
    """fma_sqrt_f32's squared sum against exact rational arithmetic on offsets whose float64 sum is inexact."""
    from fractions import Fraction
    d = lattice_offsets(65, 52, 10.)
    g = torch.Generator().manual_seed(0)
    pick = torch.randint(0, d.shape[0], (3000,), generator=g)
    sub = d[pick]
    got = fma_sqrt_f32(sub).numpy()
    for (dx, dy), r in zip(sub.numpy(), got):
        s = Fraction(float(np.float32(dx) * np.float32(dx))) + Fraction(float(dy)) ** 2
        lo = np.float32(float(s))
        cands = [np.nextafter(lo, np.float32(-np.inf)), lo, np.nextafter(lo, np.float32(np.inf))]
        best = min(cands, key=lambda c: (abs(Fraction(float(c)) - s), int(np.array(c).view(np.int32)) & 1))
        assert np.sqrt(best) == r
