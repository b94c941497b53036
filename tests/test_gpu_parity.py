"""GPU parity: the CUDA path (through the Python mirror -> ctypes -> C ABI) against
(1) the fixtures frozen from the reference and (2) the oracle on seeded inputs.

Gates (BASELINE.json north_star / SURVEY.md section 8d):
  argmax indices bit-exact; max_val bit-exact; refined coordinates <= 1e-4 px in heatmap
  space; image space <= 1e-4 px scaled by the affine magnification (plus 2 ulp at the
  coordinate magnitude); loss <= 1e-5 relative; grad <= 1e-5 relative (floor 1e-12);
  encoder targets <= 1 float32 ulp with < 1e-6 of elements differing at all (float64
  separable evaluation, one rounding); weights, NMS keep sets and pick order exact.
"""
import os
import warnings

import numpy as np
import pytest
import torch

from conftest import bits
from oracle import heatmap_oracle as O
from simple_pose_b200 import synth

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def api():
    from simple_pose_b200 import _abi
    from simple_pose_b200.commons import transforms
    from simple_pose_b200.datasets import naive_data
    from simple_pose_b200.metrics import pose_metrics
    from simple_pose_b200.processors import loss

    class NS:
        pass
    ns = NS()
    ns.abi, ns.transforms, ns.naive, ns.metrics, ns.loss = _abi, transforms, naive_data, pose_metrics, loss
    _abi.lib()
    return ns


def ulp_diff(a, b):
    ia = np.ascontiguousarray(a).view(np.int32).astype(np.int64)
    ib = np.ascontiguousarray(b).view(np.int32).astype(np.int64)
    return np.abs(ia - ib)


def assert_targets_match(got, want):
    d = ulp_diff(got, want)
    assert d.max() <= 1, "max ulp diff %d" % d.max()
    assert (d != 0).mean() < 1e-6, "fraction differing %.3g" % (d != 0).mean()


# ------------------------------------------------------------------------------------ encode
def test_encode_golden(api, golden):
    g = golden("encode")
    for tag, shape, sigma in (("a", (48, 64), 2.0), ("b", (72, 96), 2.0), ("e", (48, 64), 2.0), ("s", (48, 64), 1.5)):
        t, w = api.transforms.encode_heat_maps(torch.from_numpy(g["joints_" + tag]).to(DEV), sigma, shape)
        assert np.array_equal(w.cpu().numpy(), g["weights_" + tag]), tag
        assert_targets_match(t.cpu().numpy(), g["targets_" + tag])
        # the hand-built vectors are few enough to demand bit equality outright
        if tag == "e":
            assert np.array_equal(bits(t.cpu().numpy()), bits(g["targets_e"]))


@pytest.mark.parametrize("shape,persons", [((48, 64), 128), ((72, 96), 32), ((50, 30), 8), ((4, 4), 3), ((132, 20), 4),
                                           ((48, 63), 5), ((20, 7), 3), ((36, 33), 4)])      # odd H: per-warp factor slices stay 16-byte aligned
def test_encode_vs_oracle(api, shape, persons):
    w, h = shape
    joints = synth.joints(persons, height=h, width=w, seed=123)
    t, wt = api.transforms.encode_heat_maps(joints.to(DEV), 2.0, shape)
    rt, rw = O.encode_batch(joints.numpy(), 2.0, shape)
    assert np.array_equal(wt.cpu().numpy(), rw)
    assert_targets_match(t.cpu().numpy(), rt)
    assert 0 < (rw == 0).mean() < 1          # both cull branches exercised


@pytest.mark.parametrize("warps", ["2", "4", "8"])
def test_encode_cta_sizes_agree(api, warps):
    """Every CTA size of the encoder (SP_ENCODE_WARPS) writes the same bits, odd map counts included."""
    joints = synth.joints(37, seed=321).to(DEV)
    base_t, base_w = api.transforms.encode_heat_maps(joints)
    os.environ["SP_ENCODE_WARPS"] = warps
    api.abi.reload_tuning()
    try:
        t, w = api.transforms.encode_heat_maps(joints)
        t2, w2 = api.transforms.encode_heat_maps(joints[:, :, :], 2.0, (48, 64))
    finally:
        del os.environ["SP_ENCODE_WARPS"]
        api.abi.reload_tuning()
    assert torch.equal(t, base_t) and torch.equal(w, base_w) and torch.equal(t2, base_t) and torch.equal(w2, base_w)


@pytest.mark.parametrize("parts", ["1", "2", "3", "4", "64", "200"])
@pytest.mark.parametrize("shape", [(48, 64), (72, 96), (50, 30), (132, 20), (48, 63)])
def test_encode_row_parts_agree(api, parts, shape):
    """A map may be split into row ranges, one warp each (small launches do so by default): every split,
    including uneven ones and more parts than rows, writes the same bits as one warp per map."""
    w, h = shape
    joints = synth.joints(21, height=h, width=w, seed=654).to(DEV)
    os.environ["SP_ENCODE_PARTS"] = "1"
    api.abi.reload_tuning()
    try:
        base_t, base_w = api.transforms.encode_heat_maps(joints, 2.0, shape)
        os.environ["SP_ENCODE_PARTS"] = parts
        api.abi.reload_tuning()
        t, wt = api.transforms.encode_heat_maps(joints, 2.0, shape)
    finally:
        del os.environ["SP_ENCODE_PARTS"]
        api.abi.reload_tuning()
    auto_t, auto_w = api.transforms.encode_heat_maps(joints, 2.0, shape)
    assert torch.equal(t, base_t) and torch.equal(wt, base_w) and torch.equal(auto_t, base_t) and torch.equal(auto_w, base_w)


def test_encode_per_sample_signature_and_empty(api, golden):
    g = golden("encode")
    t, w = api.transforms.RefineSimpleTransform.get_heat_map(g["joints_e"][0], sigma=2.0, shape=(48, 64))
    assert isinstance(t, np.ndarray) and t.dtype == np.float32 and t.shape == (17, 64, 48)
    assert np.array_equal(bits(t), bits(g["targets_e"][0])) and np.array_equal(w, g["weights_e"][0])
    t0, w0 = api.transforms.encode_heat_maps(torch.zeros(0, 17, 3, device=DEV))
    assert t0.shape == (0, 17, 64, 48) and w0.shape == (0, 17)


def test_encode_denormals_kept(api):
    j = torch.tensor([[[3.0, 3.0, 1.0]]], device=DEV)
    t, _ = api.transforms.encode_heat_maps(j, 2.0, (48, 64))
    t = t.cpu().numpy()
    assert ((t > 0) & (t < 1.1754944e-38)).any()


# ------------------------------------------------------------------------------------ loss
def test_loss_golden(api, golden):
    g = golden("loss")
    pred = torch.from_numpy(g["pred"]).to(DEV).requires_grad_(True)
    loss = api.loss.JointsMSELoss()(pred, torch.from_numpy(g["target"]).to(DEV), torch.from_numpy(g["mask"]).to(DEV))
    assert loss.dim() == 0 and loss.dtype == torch.float32
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))
    got = pred.grad.cpu().numpy()
    assert np.allclose(got, g["grad"], rtol=1e-5, atol=1e-12)
    assert np.array_equal(bits(got), bits(g["grad"]))      # same operation order as ATen


@pytest.mark.parametrize("b,hw", [(128, (64, 48)), (16, (96, 72)), (5, (7, 9))])
def test_loss_vs_oracle(api, b, hw):
    h, w = hw
    joints = synth.joints(b, height=h, width=w, seed=5)
    tgt_np, msk_np = O.encode_batch(joints.numpy(), 2.0, (w, h))
    tgt, msk = torch.from_numpy(tgt_np), torch.from_numpy(msk_np)
    pred = synth.predictions_like(tgt, seed=6)
    ref_loss, ref_grad = O.masked_mse_loss_and_grad(pred, tgt, msk)
    p = pred.to(DEV).requires_grad_(True)
    loss = api.loss.JointsMSELoss()(p, tgt.to(DEV), msk.to(DEV))
    loss.backward()
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    assert torch.allclose(p.grad.cpu(), ref_grad, rtol=1e-5, atol=1e-12)
    # skip_masked variant: identical on finite inputs
    p2 = pred.to(DEV).requires_grad_(True)
    loss2 = api.loss.JointsMSELoss(skip_masked=True)(p2, tgt.to(DEV), msk.to(DEV))
    loss2.backward()
    assert loss2.item() == loss.item() and torch.equal(p2.grad, p.grad)


def test_loss_upstream_gradient_and_determinism(api):
    tgt = synth.heatmaps(8, seed=3).to(DEV)
    msk = (torch.rand(8, 17, device=DEV) > 0.2).float()
    pred = synth.predictions_like(tgt, seed=4)
    crit = api.loss.JointsMSELoss()
    p1 = pred.clone().requires_grad_(True)
    l1 = crit(p1, tgt, msk)
    l1.backward()
    p2 = pred.clone().requires_grad_(True)
    l2 = crit(p2, tgt, msk)
    (l2 * 1024.0).backward()                      # GradScaler-style upstream gradient
    assert l1.item() == l2.item()                 # deterministic reduction
    assert torch.equal(p2.grad, p1.grad * 1024.0)
    p3 = pred.clone()                             # no grad requested -> forward only
    assert crit(p3, tgt, msk).item() == l1.item()


def test_loss_is_linear_in_squared_scale(api):
    """Size-independent property at the full cfg-2 shape: scaling (pred - target) by 2 scales
    the loss by 4 and the gradient by 2 (powers of two are exact in float32)."""
    tgt = synth.heatmaps(128, seed=9).to(DEV)
    msk = torch.ones(128, 17, device=DEV)
    diff = 0.05 * torch.randn_like(tgt)
    crit = api.loss.JointsMSELoss()
    pa = (tgt + diff).requires_grad_(True)
    pb = (tgt + 2 * diff).requires_grad_(True)
    la, lb = crit(pa, tgt, msk), crit(pb, tgt, msk)
    la.backward()
    lb.backward()
    assert abs(lb.item() - 4 * la.item()) <= 2e-6 * lb.item()
    assert torch.allclose(pb.grad, 2 * pa.grad, rtol=2e-6, atol=1e-12)


# ------------------------------------------------------------------------------------ decode
def check_decode(api, hm, tinv, ref_img, ref_hsp, ref_max, ref_idx, dec=None):
    dec = dec or api.metrics.GaussTaylorKeyPointDecoder()
    hm_d = hm.to(DEV)
    keep = hm_d.clone()
    hsp, mx, idx = dec.decode_with_index(hm_d)
    assert torch.equal(hm_d, keep)                                   # input not modified
    assert np.array_equal(idx.cpu().numpy(), np.asarray(ref_idx, dtype=np.int32)), "argmax not bit-exact"
    assert np.array_equal(bits(mx.cpu().numpy()), bits(np.asarray(ref_max))), "max_val not bit-exact"
    err = np.abs(hsp.cpu().numpy().astype(np.float64) - np.asarray(ref_hsp, dtype=np.float64))
    assert np.nanmax(err) <= 1e-4, "heatmap-space error %.3g px" % np.nanmax(err)
    assert np.array_equal(np.isnan(hsp.cpu().numpy()), np.isnan(ref_hsp))
    if tinv is not None:
        img, mx2 = dec(hm_d, tinv.to(DEV))
        assert img.shape == (hm.shape[0], hm.shape[1], 2) and mx2.shape == (hm.shape[0], hm.shape[1], 1)
        mag = tinv[:, :, :2].abs().sum(-1).max(-1)[0].numpy()[:, None, None]     # px per heatmap px
        tol = 1e-4 * mag + 2 * np.spacing(np.abs(np.asarray(ref_img)).astype(np.float32))
        ierr = np.abs(img.cpu().numpy().astype(np.float64) - np.asarray(ref_img, dtype=np.float64))
        assert (ierr <= tol).all(), "image-space error %.3g" % ierr.max()
    return float(np.nanmax(err))


def test_decode_golden(api, golden):
    g = golden("decode")
    for tag in ("a", "b", "e"):
        check_decode(api, torch.from_numpy(g["hm_" + tag]), torch.from_numpy(g["tinv_" + tag]),
                     g["img_" + tag], g["hsp_" + tag], g["max_" + tag], g["idx_" + tag])


def test_blur_weights_are_the_reference_ones(api, golden):
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    assert np.array_equal(bits(dec.blur_weights.cpu().numpy()), bits(golden("blur_weights")["w11"]))


@pytest.mark.parametrize("b,hw,noise", [(128, (64, 48), 0.01), (64, (96, 72), 0.01), (32, (64, 48), 0.05),
                                        (8, (32, 24), 0.02), (6, (40, 50), 0.01), (4, (33, 31), 0.01)])
def test_decode_vs_oracle(api, b, hw, noise):
    h, w = hw
    hm = synth.heatmaps(b, height=h, width=w, seed=77, noise=noise)
    tinv = synth.inverse_affines(b, height=h, width=w, seed=77)[0]
    ref_img, ref_max = O.gauss_taylor_decode(hm, tinv)
    ref_hsp, _ = O.gauss_taylor_decode(hm, None, return_heatmap_space=True)
    check_decode(api, hm, tinv, ref_img.numpy(), ref_hsp.numpy(), ref_max.numpy(), O.argmax_index(hm).numpy())


@pytest.mark.parametrize("ksize", [3, 5, 7, 9, 13, 15])
@pytest.mark.parametrize("hw", [(64, 48), (40, 36)])
def test_decode_other_kernel_sizes(api, ksize, hw):
    """GaussTaylorKeyPointDecoder(kernel_size != 11): OpenCV's fixed Gaussian tables (n <= 9) and the closed
    form (n >= 13) through the run-time-ksize kernel path, against the restatement (itself pinned to the
    reference for these sizes by oracle/fuzz_vs_reference.py)."""
    h, w = hw
    hm = synth.heatmaps(24, height=h, width=w, seed=700 + ksize, noise=0.01)
    dec = api.metrics.GaussTaylorKeyPointDecoder(kernel_size=ksize)
    assert np.array_equal(bits(dec.blur_weights.cpu().numpy()), bits(O.blur_weights(ksize)))
    c, m, idx = dec.decode_with_index(hm.to(DEV))
    oc, om = O.gauss_taylor_decode(hm, None, ksize, return_heatmap_space=True)
    assert torch.equal(idx.cpu().long(), O.argmax_index(hm)) and torch.equal(m.cpu(), om)
    assert (c.cpu() - oc).abs().max().item() <= 1e-4


def test_decode_generic_path_matches_fast_path(api):
    hm = synth.heatmaps(16, seed=5).to(DEV)
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    a = dec.decode_with_index(hm)
    os.environ["SP_DECODE_FORCE_GENERIC"] = "1"
    api.abi.reload_tuning()
    try:
        b = dec.decode_with_index(hm)
    finally:
        del os.environ["SP_DECODE_FORCE_GENERIC"]
        api.abi.reload_tuning()
    assert torch.equal(a[2], b[2]) and torch.equal(a[1], b[1])
    assert (a[0] - b[0]).abs().max().item() <= 1e-5


@pytest.mark.parametrize("warps,stages", [(1, 1), (4, 2), (8, 2), (16, 1), (3, 4)])
def test_decode_ring_configurations(api, warps, stages):
    """Every warps x stages ring layout walks the same maps (phase/parity bookkeeping)."""
    hm = synth.heatmaps(40, seed=6)
    ref_hsp, ref_max = O.gauss_taylor_decode(hm, None, return_heatmap_space=True)
    os.environ["SP_DECODE_WARPS"], os.environ["SP_DECODE_STAGES"] = str(warps), str(stages)
    api.abi.reload_tuning()
    try:
        check_decode(api, hm, None, None, ref_hsp.numpy(), ref_max.numpy(), O.argmax_index(hm).numpy())
    finally:
        del os.environ["SP_DECODE_WARPS"], os.environ["SP_DECODE_STAGES"]
        api.abi.reload_tuning()


def test_argmax_special_values(api):
    """torch.max semantics: first index on ties, NaN wins (first NaN), +-Inf, -0.0 == +0.0."""
    hm = torch.zeros(1, 8, 64, 48)
    hm[0, 0, 5, 5] = float("nan")
    hm[0, 0, 9, 9] = 3.0
    hm[0, 1, 7, 7] = float("inf")
    hm[0, 1, 8, 8] = float("inf")
    hm[0, 2] = -float("inf")
    hm[0, 3] = float("nan")
    hm[0, 4] = -0.0
    hm[0, 4, 2, 3] = 0.0
    hm[0, 5, 63, 47] = 1e-30
    hm[0, 6] = -1.0
    hm[0, 6, 0, 1] = -0.0
    hm[0, 7, 10, 4:8] = 2.0
    ref_c, ref_m = O.argmax_coords(hm)
    ref_i = O.argmax_index(hm)
    c, m, i = api.metrics.BasicKeyPointDecoder.heat_map_argmax(hm.to(DEV))
    assert torch.equal(i.cpu().long(), ref_i)
    assert np.array_equal(bits(m.cpu().numpy()), bits(ref_m.numpy()))
    assert torch.equal(c.cpu(), ref_c)
    c2, m2 = api.metrics.BasicKeyPointDecoder.heat_map_to_axis(hm.to(DEV))
    assert torch.equal(c2, c) and c2.shape == (1, 8, 2) and m2.shape == (1, 8, 1)
    # the full decoder must agree with the reference on which joints are refined at all
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    hsp, mx, idx = dec.decode_with_index(hm.to(DEV))
    o_hsp, o_mx = O.gauss_taylor_decode(hm, None, return_heatmap_space=True)
    assert torch.equal(idx.cpu().long(), ref_i)
    ok = ~torch.isnan(o_hsp)
    assert torch.equal(torch.isnan(hsp.cpu()), ~ok)
    assert (hsp.cpu()[ok] - o_hsp[ok]).abs().max().item() <= 1e-4


def test_decode_clamp_path_mixed_stencils(api):
    """Maps whose blurred neighbourhood straddles the 1e-10 clamp take the exact slow path
    (whole-map blur max); results must still match the reference."""
    g = torch.Generator().manual_seed(3)
    hm = 0.02 * torch.randn(4, 17, 64, 48, generator=g)            # noise-dominated: mixed signs after blur
    yy, xx = torch.meshgrid(torch.arange(64.), torch.arange(48.), indexing="ij")
    for k in range(17):
        hm[0, k] = torch.exp(-((xx - 10 - k) ** 2 + (yy - 20 - k) ** 2) / 1.0) - 0.03 * (k + 1) / 17
    ref_hsp, ref_max = O.gauss_taylor_decode(hm, None, return_heatmap_space=True)
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    hsp, mx, idx = dec.decode_with_index(hm.to(DEV))
    assert torch.equal(idx.cpu().long(), O.argmax_index(hm))
    assert torch.equal(mx.cpu(), ref_max)
    # ill-conditioned joints amplify 1-ulp differences (SURVEY.md fact 5): the gate scales with
    # the size of the Taylor step the reference itself takes (1e-4 px per px of offset)
    base = O.argmax_coords(hm)[0]
    off = (ref_hsp - base).abs().max(-1)[0]
    tol = 1e-4 * torch.clamp(off, min=1.0)
    err = (hsp.cpu() - ref_hsp).abs().max(-1)[0]
    assert (err <= tol).all(), (err / tol).max().item()
    assert (off > 0).float().mean() > 0.4           # most joints are actually refined
    assert torch.isfinite(hsp).all()


def test_basic_decoder(api, golden):
    g, d = golden("next_rows"), golden("decode")
    hm = torch.from_numpy(d["hm_a"]).to(DEV)
    img, mx = api.metrics.BasicKeyPointDecoder()(hm, torch.from_numpy(d["tinv_a"]).to(DEV))
    assert np.array_equal(bits(mx.cpu().numpy()), bits(g["basic_max"]))
    assert np.abs(img.cpu().numpy() - g["basic_img"]).max() <= 1e-3
    hsp, _ = api.metrics.BasicKeyPointDecoder()(hm, synth.identity_affines(3).to(DEV))
    assert np.array_equal(hsp.cpu().numpy(), g["basic_hsp"])
    e, _ = api.metrics.BasicKeyPointDecoder()(torch.from_numpy(d["hm_e"]).to(DEV), synth.identity_affines(1).to(DEV))
    assert np.array_equal(e.cpu().numpy(), g["basic_edge_hsp"])


# ------------------------------------------------------------------------------------ flip test
def test_dark_original_decoder(api, golden):
    """Mode SP_DECODE_DARK_ORIGINAL against the reference's NumPy/OpenCV decoder (frozen outputs and the
    pinned restatement): argmax-level outputs exact, coordinates within 1e-4 px in heatmap space (the
    reference blurs in float64, the kernel in float32), negative Taylor results kept, input not modified."""
    g, d = golden("dark_original"), golden("decode")
    dec = api.metrics.DarkPoseOriginalKeyPointDecoder()
    for tag in ("a", "b", "e"):
        hm = torch.from_numpy(d["hm_" + tag]).to(DEV)
        keep = hm.clone()
        tinv = torch.from_numpy(d["tinv_" + tag]).to(DEV)
        c, m = dec(hm, tinv)
        mag = tinv[:, :, :2].abs().sum(-1).max().item()
        assert np.array_equal(bits(m.cpu().numpy()), bits(g["max_" + tag]))
        assert np.abs(c.cpu().numpy() - g["img_" + tag]).max() <= 1e-4 * mag + 1e-4
        assert torch.equal(hm, keep)
    eye = synth.identity_affines(1, device=DEV)
    c, m = dec(torch.from_numpy(g["hm_n"]).to(DEV), eye)
    got = c.cpu().numpy()
    assert (got < 0).any(axis=-1).all()
    assert np.abs(got - g["hsp_n"]).max() <= 2e-3          # float32 vs float64 blur with |offset| up to 23 px
    gt, _ = api.metrics.GaussTaylorKeyPointDecoder()(torch.from_numpy(g["hm_n"]).to(DEV), eye)
    assert gt.min().item() == 0.0
    # seeded maps against the restatement
    hm = synth.heatmaps(64, seed=35, noise=0.01)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        oc, om = O.dark_original_decode(hm, synth.identity_affines(64))
    c, m = dec(hm.to(DEV), synth.identity_affines(64, device=DEV))
    assert torch.equal(m.cpu(), om) and (c.cpu() - oc).abs().max().item() <= 1e-4


def test_flip_decode_golden(api, golden):
    g = golden("flip")
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    hm, hf = torch.from_numpy(g["hm"]).to(DEV), torch.from_numpy(g["hm_flip"]).to(DEV)
    keep_a, keep_b = hm.clone(), hf.clone()
    hsp, mx, idx = dec.decode_with_index(hm, None, hf)
    assert torch.equal(hm, keep_a) and torch.equal(hf, keep_b)
    assert np.array_equal(idx.cpu().numpy(), g["idx"])
    assert np.array_equal(bits(mx.cpu().numpy()), bits(g["max"]))
    assert np.abs(hsp.cpu().numpy() - g["hsp"]).max() <= 1e-4
    img, _ = dec.flip_call(hm, hf, torch.from_numpy(g["tinv"]).to(DEV), [[1, 2], [3, 4], [5, 6], [7, 8], [9, 10], [11, 12], [13, 14], [15, 16]])
    assert np.abs(img.cpu().numpy() - g["img"]).max() <= 1e-3


@pytest.mark.parametrize("b,hw", [(256, (64, 48)), (32, (96, 72)), (4, (20, 22))])
def test_flip_decode_vs_oracle_and_mirror_identity(api, b, hw):
    h, w = hw
    hm, hf = synth.flip_pair(b, height=h, width=w, seed=31)
    ref_hsp, ref_max = O.flip_decode(hm, hf, None, return_heatmap_space=True)
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    hsp, mx, idx = dec.decode_with_index(hm.to(DEV), None, hf.to(DEV))
    assert torch.equal(idx.cpu().long(), O.argmax_index(O.flip_average(hm, hf)))
    assert torch.equal(mx.cpu(), ref_max)
    assert (hsp.cpu() - ref_hsp).abs().max().item() <= 1e-4
    # property: if hm_flip is the exact mirrored/swapped copy of hm, flip decode == plain decode
    perm = O.swap_permutation(17)
    mirror = hm.flip(-1)[:, perm].contiguous()
    a = dec.decode_with_index(hm.to(DEV), None, mirror.to(DEV))
    p = dec.decode_with_index(hm.to(DEV))
    assert torch.equal(a[2], p[2]) and torch.equal(a[1], p[1]) and torch.equal(a[0], p[0])


# ------------------------------------------------------------------------------------ round trip
@pytest.mark.parametrize("hw", [(64, 48), (96, 72)])
def test_encode_decode_round_trip(api, hw):
    """Size-independent property: decoding an encoded target recovers the centre."""
    h, w = hw
    g = torch.Generator().manual_seed(1)
    mu = torch.rand(512, 17, 2, generator=g)
    mu[..., 0] = 3 + mu[..., 0] * (w - 7)
    mu[..., 1] = 3 + mu[..., 1] * (h - 7)
    joints = torch.cat([mu, torch.ones(512, 17, 1)], -1)
    t, wt = api.transforms.encode_heat_maps(joints.to(DEV), 2.0, (w, h))
    assert (wt == 1).all()
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    xy, mx = dec(t, synth.identity_affines(512).to(DEV))
    err = (xy.cpu() - mu).abs()
    # within 8 px of a border the zero-padded blur biases the estimate (reference: same 0.051 px)
    far = (mu[..., 0] > 8) & (mu[..., 0] < w - 9) & (mu[..., 1] > 8) & (mu[..., 1] < h - 9)
    assert err.max().item() < 0.06, err.max().item()
    assert err[far].max().item() < 1e-3, err[far].max().item()
    assert (mx > 0.77).all()


# ------------------------------------------------------------------------------------ OKS / NMS
def test_oks_golden(api, golden):
    g = golden("oks")
    keep, scores, rank = api.naive.rescore_and_nms(g["kps"], g["box_scores"], g["areas"], g["seg"])
    assert np.array_equal(keep.cpu().numpy(), g["keep"])
    assert np.allclose(scores.cpu().numpy(), g["scores"], rtol=1e-15, atol=0)
    lo, hi = int(g["seg"][0]), int(g["seg"][1])
    iou = api.naive.oks_iou(g["kps"][lo], g["kps"][lo:hi], g["areas"][lo], g["areas"][lo:hi])
    assert np.allclose(iou, g["iou0"], rtol=1e-14, atol=1e-300)
    iou_v = api.naive.oks_iou(g["kps"][lo], g["kps"][lo:hi], g["areas"][lo], g["areas"][lo:hi], in_vis_thresh=0.5)
    assert np.allclose(iou_v, g["iou0_vis"], rtol=1e-14, atol=1e-300)
    picks = []
    for s in range(len(g["seg"]) - 1):
        lo, hi = int(g["seg"][s]), int(g["seg"][s + 1])
        got = api.naive.oks_nms(g["kps"][lo:hi], g["scores"][lo:hi], g["areas"][lo:hi], 0.9)
        picks.extend(i + lo for i in got)
    assert picks == [int(i) for i in g["picks"]]


def test_oks_nms_vs_oracle_large(api):
    kps, box, area, seg = synth.nms_groups(400, mean_group=20.0, seed=8)
    keep, scores, rank = api.naive.rescore_and_nms(kps, box, area, seg)
    o_keep, o_scores, o_picks = O.rescore_and_nms(kps.numpy(), box.numpy(), area.numpy(), seg.numpy())
    assert np.array_equal(keep.cpu().numpy().astype(bool), o_keep)
    assert np.allclose(scores.cpu().numpy(), o_scores, rtol=1e-15, atol=0)
    assert 0.2 < o_keep.mean() < 0.95
    # pick order per image from (keep, rank)
    keep_np, rank_np = keep.cpu().numpy().astype(bool), rank.cpu().numpy()
    for s in range(0, 400, 37):
        lo, hi = int(seg[s]), int(seg[s + 1])
        kept = np.nonzero(keep_np[lo:hi])[0]
        order = [int(i) + lo for i in kept[np.argsort(rank_np[lo:hi][kept])]]
        assert order == o_picks[s]


@pytest.mark.parametrize("mean_group", [3.0, 30.0, 62.0, 90.0])
def test_oks_nms_pair_matrix_path_equals_greedy_loop(api, mean_group):
    """Images of up to 64 persons take the all-pairs bit-matrix path, larger ones the per-pick loop;
    SP_NMS_SERIAL=1 forces the loop everywhere. Keep sets, ranks and the oracle agree, with a score
    tie (visiting order = descending index) and segments of exactly 1, 2, 63, 64 and 65 persons."""
    kps, box, area, seg = synth.nms_groups(60, mean_group=mean_group, seed=int(mean_group))
    n = kps.shape[0]
    box[2] = box[1]                                             # a score tie inside the 2-person image (NumPy's argsort is
                                                                # only order-stable for such small inputs: insertion sort)
    cuts = sorted(set([0, 1, 3, 66, 130, 195] + [int(v) for v in seg.tolist() if v > 195] + [n]))
    cuts = [c for c in cuts if c <= n]
    seg2 = np.array(cuts, dtype=np.int32)
    keep, rank = api.naive.oks_nms_batched(kps, box, area, seg2, 0.9)
    os.environ["SP_NMS_SERIAL"] = "1"
    api.abi.reload_tuning()
    try:
        keep_s, rank_s = api.naive.oks_nms_batched(kps, box, area, seg2, 0.9)
    finally:
        del os.environ["SP_NMS_SERIAL"]
        api.abi.reload_tuning()
    assert torch.equal(keep, keep_s) and torch.equal(rank, rank_s)
    sizes = np.diff(seg2)
    assert sizes.min() <= 2 and (sizes == 63).any() and (sizes == 64).any() and (sizes == 65).any()
    keep_np = keep.cpu().numpy().astype(bool)
    for s_i in range(len(seg2) - 1):
        lo, hi = int(seg2[s_i]), int(seg2[s_i + 1])
        o = O.oks_greedy_nms(kps.numpy()[lo:hi], box.numpy()[lo:hi], area.numpy()[lo:hi], 0.9)
        assert sorted(int(i) + lo for i in o) == [int(i) for i in np.nonzero(keep_np)[0] if lo <= i < hi], s_i
    assert 0 < keep_np.sum() < n


@pytest.mark.parametrize("n", [9, 17, 33, 64, 80])
def test_oks_nms_score_ties_follow_the_documented_rule(api, n):
    """Equal scores are visited higher index first (what `argsort()[::-1]` gives over a stable sort); the
    reference leaves that order to NumPy's host-dependent SIMD sort (DESIGN.md section 4, OKS-NMS). The kernel's keep
    set and pick order equal the reference algorithm run on scores de-tied by that rule, in both kernel paths."""
    rng = np.random.RandomState(n)
    for trial in range(6):
        kps, _, area, _ = synth.nms_groups(1, mean_group=float(n), seed=1000 * n + trial)
        m = kps.shape[0]
        tied = rng.choice([0.2, 0.4, 0.6], size=m)
        want = [int(i) for i in O.oks_greedy_nms(kps.numpy(), O.detie_scores(tied), area.numpy(), 0.9)]
        assert api.naive.oks_nms(kps.numpy(), tied, area.numpy(), 0.9) == want
        assert len(want) < m                                   # duplicates with equal scores really compete


def test_oks_nms_decisions_at_the_threshold(api):
    """The kernel decides oks > thresh from a float32 evaluation when that is further than 1e-4 from the threshold and
    re-evaluates with the reference's float64 chain otherwise. Thresholds a relative 1e-12 either side of a pair's exact
    OKS value (the float64 chain itself agrees with NumPy to 1e-14: CUDA's and NumPy's exp may differ in the last bit)
    and a few 1e-5 either side must all give the float64 verdict (both entry points)."""
    kps, _, area, _ = synth.nms_groups(1, mean_group=60.0, seed=3, dup_frac=0.7, jitter=3.0)
    kps_np, area_np = kps.numpy(), area.numpy()
    tested = 0
    for j in range(1, kps_np.shape[0]):
        v = float(O.oks_similarity(kps_np[0], kps_np[j:j + 1], area_np[0], area_np[j:j + 1])[0])
        if not 0.05 < v < 0.9995:
            continue
        pair_k, pair_a = kps_np[[0, j]], area_np[[0, j]]
        for thr in (v * (1 - 1e-12), v * (1 + 1e-12), v + 5e-5, v - 5e-5, v + 2e-4, v - 2e-4):
            want = [int(i) for i in O.oks_greedy_nms(pair_k, np.array([0.9, 0.8]), pair_a, thr)]
            assert api.naive.oks_nms(pair_k, np.array([0.9, 0.8]), pair_a, thr) == want, (j, v, thr)
            tested += 1
        if tested >= 140:
            break
    assert tested >= 24
    # the fused rows kernel takes the same decisions on float32 keypoints
    from simple_pose_b200 import _abi
    k32 = kps.float()
    v = float(O.oks_similarity(k32[0].double().numpy(), k32[1:2].double().numpy(), area_np[0], area_np[1:2])[0])
    for thr in (v * (1 - 1e-12), v * (1 + 1e-12), v - 3e-5, v + 3e-5):
        rows = torch.zeros(2, 54, device=DEV)
        rows[:, :51] = k32[:2].reshape(2, 51).to(DEV)
        seg = torch.tensor([0, 2], dtype=torch.int32, device=DEV)
        bs = torch.tensor([0.9, 0.8], dtype=torch.float64, device=DEV)
        ar = torch.from_numpy(area_np[:2]).to(DEV)
        _abi.check(_abi.lib().sp_eval_rows_nms_f32(rows.data_ptr(), 54, bs.data_ptr(), ar.data_ptr(), None, seg.data_ptr(), None, None,
                                                   2, 1, 17, 2, -1.0, float(thr), _abi.stream_ptr(torch.device(DEV))))
        keep = (rows[:, 51] > 0.5).cpu().tolist()
        assert keep == [True, not (v > thr)], (v, thr)


def test_oks_nms_edge_cases(api):
    kps, box, area, seg = synth.nms_groups(3, mean_group=5.0, seed=2)
    # empty segment in the middle, single-person image, and one big image
    n = kps.shape[0]
    seg2 = np.array([0, 1, 1, n], dtype=np.int32)
    keep, rank = api.naive.oks_nms_batched(kps, box, area, seg2, 0.9)
    assert keep[0].item() == 1
    o = O.oks_greedy_nms(kps.numpy()[1:], box.numpy()[1:], area.numpy()[1:], 0.9)
    assert sorted(int(i) + 1 for i in o) == [int(i) for i in np.nonzero(keep.cpu().numpy())[0] if i >= 1]
    assert api.naive.oks_nms(np.zeros((0, 17, 3)), np.zeros(0), np.zeros(0), 0.9) == []
    # identical poses: only the best survives
    same = kps[:1].repeat(6, 1, 1)
    got = api.naive.oks_nms(same.numpy(), np.array([.1, .5, .3, .9, .2, .4]), np.full(6, 1e4), 0.9)
    assert got == [3]


def test_pack_and_end_to_end_eval_chain(api):
    """decode -> pack -> rescore -> NMS on the device equals the reference chain."""
    hm = synth.heatmaps(64, seed=12)
    tinv, area = synth.inverse_affines(64, seed=12)
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    c, m = dec(hm.to(DEV), tinv.to(DEV))
    kps = api.naive.pack_keypoints(c, m)
    assert kps.dtype == torch.float64 and kps.shape == (64, 17, 3)
    assert torch.equal(kps[..., :2].float(), c) and torch.equal(kps[..., 2:].float(), m)
    seg = np.arange(0, 65, 8, dtype=np.int32)
    box = torch.rand(64, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    keep, scores, _ = api.naive.rescore_and_nms(kps, box, area, seg)
    o_keep, o_scores, _ = O.rescore_and_nms(kps.cpu().numpy(), box.numpy(), area.numpy(), seg)
    assert np.array_equal(keep.cpu().numpy().astype(bool), o_keep)
    assert np.allclose(scores.cpu().numpy(), o_scores, rtol=1e-15, atol=0)


def test_pack_rows_equals_torch_composition(api):
    from simple_pose_b200.eval_shard import pack_results
    g = torch.Generator().manual_seed(3)
    for n, k in ((0, 17), (1, 17), (777, 17), (40, 5)):
        coords = torch.randn(n, k, 2, generator=g).to(DEV)
        conf = torch.rand(n, k, 1, generator=g).to(DEV)
        keep = (torch.rand(n, generator=g) < 0.5).to(torch.uint8).to(DEV)
        scores = torch.rand(n, generator=g, dtype=torch.float64).to(DEV)
        rows = pack_results(coords, conf, keep, scores)
        want = torch.cat([torch.cat([coords, conf], dim=-1).reshape(n, 3 * k), keep.float()[:, None], scores.float()[:, None]], dim=1)
        assert rows.shape == (n, 3 * k + 2) and torch.equal(rows, want)
    with pytest.raises(RuntimeError, match="no CPU path"):
        pack_results(coords.cpu(), conf.cpu(), keep.cpu(), scores.cpu())


@pytest.mark.parametrize("chunks", [1, 3])
@pytest.mark.parametrize("use_boxes,flip", [(True, False), (False, True)])
def test_sharded_evaluator_single_rank_fused_rows(api, chunks, use_boxes, flip):
    """ShardedPoseEvaluator (decoder writing the result rows, rescoring + NMS fused on the rows) against the
    stand-alone kernels and the oracle: keypoints and keep flags identical, the float64 score bit-exact."""
    from simple_pose_b200 import eval_shard
    es = synth.EvalSet(persons=900, mean_group=7.0, seed=31)
    n = es.persons
    hm = es.heatmaps(0, n, "cpu")
    hf = synth.heatmaps(n, seed=32) if flip else None
    ev = eval_shard.ShardedPoseEvaluator(chunks=chunks)
    ev.plan(es.seg)
    assert ev.my_persons() == (0, n)
    c_, s_, area_np, tinv_np = O.box_affines(es.boxes.tolist())
    if use_boxes:
        rows = ev.run(hm.to(DEV), None, es.box_scores, None, boxes=es.boxes.to(DEV), heat_map_flip=None if hf is None else hf.to(DEV))
    else:
        rows = ev.run(hm.to(DEV), torch.from_numpy(tinv_np).to(DEV), es.box_scores, torch.from_numpy(area_np).double(),
                      heat_map_flip=None if hf is None else hf.to(DEV))
    assert rows.shape == (n, 54) and rows.dtype == torch.float32
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    tinv = torch.from_numpy(tinv_np).to(DEV)
    xy, conf = dec.flip_call(hm.to(DEV), hf.to(DEV), tinv) if flip else dec(hm.to(DEV), tinv)
    kps = api.naive.pack_keypoints(xy, conf)
    keep, scores, _ = api.naive.rescore_and_nms(kps, es.box_scores, torch.from_numpy(area_np).double(), es.seg.astype(np.int32))
    assert torch.equal(eval_shard.row_keypoints(rows), torch.cat([xy, conf], -1))
    assert torch.equal(eval_shard.row_keep(rows), keep.bool())
    assert torch.equal(eval_shard.row_scores(rows), scores)
    o_keep, o_scores, _ = O.rescore_and_nms(kps.cpu().numpy(), es.box_scores.numpy(), area_np.astype(np.float64), es.seg.astype(np.int32))
    assert np.array_equal(eval_shard.row_keep(rows).cpu().numpy(), o_keep)
    assert np.allclose(eval_shard.row_scores(rows).cpu().numpy(), o_scores, rtol=1e-15, atol=0)
    if not flip:
        assert 0 < int(o_keep.sum()) < n - 50                   # the duplicate detections are really suppressed
    raw = ev.run(hm.to(DEV), tinv, es.box_scores, torch.from_numpy(area_np).double(),
                 heat_map_flip=None if hf is None else hf.to(DEV), compact=False)
    assert raw.buffer.shape[:2] == (chunks, 1) and raw.persons == n and eval_shard.rows_equal(raw.rows(), rows)
    with pytest.raises(ValueError):
        ev.run(hm[:-1].to(DEV), tinv[:-1], es.box_scores[:-1], torch.from_numpy(area_np[:-1]).double())


def test_sharded_evaluator_incremental_batches(api):
    """begin / add_batch / finish (the shape of the reference's eval loop, eval.py:133-149: heatmaps arrive batch by
    batch) returns the table of one run() over all heatmaps, with boxes or with ready-made affines."""
    from simple_pose_b200 import eval_shard
    es = synth.EvalSet(persons=700, mean_group=6.0, seed=41)
    n = es.persons
    hm = es.heatmaps(0, n, DEV)
    boxes = es.boxes.to(DEV)
    ev = eval_shard.ShardedPoseEvaluator(chunks=1)
    ev.plan(es.seg)
    want = ev.run(hm, None, es.box_scores, None, boxes=boxes)
    cuts = [0, 1, 130, 131, 400, n]
    ev.begin(DEV)
    for a, b in zip(cuts[:-1], cuts[1:]):
        ev.add_batch(a, hm[a:b], boxes=boxes[a:b])
    ev.add_batch(n, hm[:0], boxes=boxes[:0])                      # an empty last batch is a no-op
    got = ev.finish(es.box_scores)
    assert eval_shard.rows_equal(got, want)
    aff = api.naive.box_affines(boxes)
    ev.begin(DEV)
    for a, b in zip(cuts[:-1], cuts[1:]):
        ev.add_batch(a, hm[a:b], trans_inv=aff["trans_inv"][a:b])
    got2 = ev.finish(es.box_scores, areas=aff["area"].double())
    assert eval_shard.rows_equal(got2, want)
    with pytest.raises(ValueError):
        ev.add_batch(n - 3, hm[:5], boxes=boxes[:5])
    ev3 = eval_shard.ShardedPoseEvaluator(chunks=2)
    ev3.plan(es.seg)
    with pytest.raises(ValueError):
        ev3.begin(DEV)


def test_kps_to_dict_on_device(api):
    """A10 (metrics/pose_metrics.py:172-179) with CUDA tensors: one kernel + one D2H; keypoints are the
    decoder's floats exactly, the score mean(conf) + max(conf) agrees with the reference's float32 torch
    reductions to 1 ulp (its summation order is not defined across torch's CPU and CUDA kernels)."""
    hm = synth.heatmaps(33, seed=77)
    tinv, _ = synth.inverse_affines(33, seed=77)
    xy, conf = api.metrics.GaussTaylorKeyPointDecoder()(hm.to(DEV), tinv.to(DEV))
    got, want = [], []
    ids = list(range(500, 533))
    api.metrics.kps_to_dict_(xy, conf, ids, got)
    O.kps_to_dict(xy.cpu(), conf.cpu(), ids, want)
    assert len(got) == len(want) == 33
    for g, w in zip(got, want):
        assert g["image_id"] == w["image_id"] and g["category_id"] == 1
        assert g["keypoints"] == w["keypoints"]
        assert abs(g["score"] - w["score"]) <= 2.4e-7 * abs(w["score"])
    rows = api.metrics.person_rows(xy, conf)
    assert rows.shape == (33, 52) and torch.equal(rows[:, :51].reshape(33, 17, 3), torch.cat([xy, conf], -1))
    nan_conf = conf.clone()
    nan_conf[3, 5] = float("nan")
    assert torch.isnan(api.metrics.person_rows(xy, nan_conf)[3, -1]) and not torch.isnan(api.metrics.person_rows(xy, nan_conf)[4, -1])
    with pytest.raises(RuntimeError, match="no CPU path"):
        api.metrics.kps_to_dict_(xy.cpu(), conf.cpu(), ids, [])
    empty = []
    api.metrics.kps_to_dict_(xy[:0], conf[:0], [], empty)
    assert empty == []


def test_pipeline_rejects_what_it_cannot_read(api):
    """HeatmapHotPath hands raw pointers to the C ABI: wrong dtype / shape / layout / device must raise."""
    from simple_pose_b200.pipeline import HeatmapHotPath
    hp = HeatmapHotPath(4, 17, 64, 48, device=DEV)
    joints = synth.joints(4, seed=1).to(DEV)
    pred = synth.heatmaps(4, seed=1).to(DEV)
    tinv = synth.identity_affines(4, device=DEV)
    hp.step(joints, pred, tinv)
    for bad in (pred.half(), pred[:3], pred.permute(0, 1, 3, 2), pred.double()):
        with pytest.raises(ValueError):
            hp.loss_fwd_bwd(bad)
        with pytest.raises(ValueError):
            hp.decode(bad, tinv)
        with pytest.raises(ValueError):
            hp.train_fused(joints, bad)
    with pytest.raises(ValueError):
        hp.encode(joints.double())
    with pytest.raises(RuntimeError):
        hp.encode(joints.cpu())
    torch.cuda.synchronize()


def test_errors_are_loud(api):
    with pytest.raises(RuntimeError):
        api.metrics.GaussTaylorKeyPointDecoder()(torch.zeros(1, 17, 64, 48), torch.zeros(1, 2, 3))   # CPU tensors
    with pytest.raises(ValueError):
        api.metrics.GaussTaylorKeyPointDecoder()(torch.zeros(1, 17, 64, 48, device=DEV), torch.zeros(2, 2, 3, device=DEV))
    with pytest.raises(RuntimeError):
        api.abi.check(-4)


# ------------------------------------------------------------------------------------ section 8f rows
def test_basic_encoder_golden(api, golden):
    g = golden("next_rows")
    t, w = api.transforms.encode_heat_maps_basic(torch.from_numpy(g["joints_q"]).to(DEV), 2.0, (48, 64), 4)
    assert np.array_equal(bits(t.cpu().numpy()), bits(g["targets_q"]))
    assert np.array_equal(w.cpu().numpy(), g["weights_q"])
    t1, w1 = api.transforms.BasicSimpleTransform.get_heat_map(g["joints_q"][0], 2.0, (48, 64), 4)
    assert np.array_equal(bits(t1), bits(g["targets_q"][0])) and np.array_equal(w1, g["weights_q"][0])


@pytest.mark.parametrize("shape,stride,sigma", [((48, 64), 4, 2.0), ((72, 96), 4, 2.0), ((30, 22), 8, 1.5), ((48, 64), 4, 1.0)])
def test_basic_encoder_vs_oracle(api, shape, stride, sigma):
    w, h = shape
    joints = synth.joints(16, height=h * stride, width=w * stride, seed=61)
    joints[..., :2] += torch.tensor([-20.0, 30.0])           # push some centres off the map
    t, wt = api.transforms.encode_heat_maps_basic(joints.to(DEV), sigma, shape, stride)
    ref = [O.encode_person_basic(j, sigma, shape, stride) for j in joints.numpy()]
    assert np.array_equal(bits(t.cpu().numpy()), bits(np.stack([r[0] for r in ref])))
    assert np.array_equal(wt.cpu().numpy(), np.stack([r[1] for r in ref]))


def test_heat_map_acc_golden_and_oracle(api, golden):
    g, e = golden("next_rows"), golden("encode")
    tgt = torch.from_numpy(e["targets_a"])
    msk = torch.from_numpy(e["weights_a"])[..., None, None]
    acc = api.metrics.HeatMapAcc()((torch.from_numpy(g["acc_pred"]) * msk).to(DEV), (tgt * msk).to(DEV))
    assert acc.dim() == 0 and np.float32(acc.item()) == g["acc_value"]
    for seed, noise in ((1, 0.05), (2, 0.3), (3, 1.0)):
        j = synth.joints(64, seed=seed)
        t_np, w_np = O.encode_batch(j.numpy())
        t, m = torch.from_numpy(t_np), torch.from_numpy(w_np)[..., None, None]
        p = synth.predictions_like(t, seed=seed + 10, noise=noise)
        want = O.heat_map_acc(p * m, t * m)
        got = api.metrics.HeatMapAcc()((p * m).to(DEV), (t * m).to(DEV))
        assert np.float32(got.item()) == np.float32(float(want)), (seed, got.item(), float(want))
    # no valid joint at all -> 0
    z = torch.zeros(2, 17, 64, 48, device=DEV)
    assert api.metrics.HeatMapAcc()(z, z).item() == 0.0


@pytest.mark.parametrize("b,hw,noise", [(128, (64, 48), 0.05), (24, (96, 72), 0.3), (6, (16, 12), 0.5), (5, (10, 6), 0.2),
                                        (4, (31, 24), 0.2), (3, (63, 48), 0.1), (5, (9, 64), 0.2)])     # odd H
def test_fused_encode_loss_acc(api, b, hw, noise):
    """EncodeJointsMSELoss(pred, joints) == reference loss/grad on reference-encoded targets, and its
    accuracy == HeatMapAcc()(pred*mask, target*mask) (solver :106-107,123-124)."""
    h, w = hw
    joints = synth.joints(b, height=h, width=w, seed=71)
    t_np, w_np = O.encode_batch(joints.numpy(), 2.0, (w, h))
    tgt, msk = torch.from_numpy(t_np), torch.from_numpy(w_np)
    pred = synth.predictions_like(tgt, seed=72, noise=noise)
    ref_loss, ref_grad = O.masked_mse_loss_and_grad(pred, tgt, msk)
    ref_acc = O.heat_map_acc(pred * msk[..., None, None], tgt * msk[..., None, None])
    crit = api.loss.EncodeJointsMSELoss(sigma=2.0, with_acc=True, keep_targets=True)
    p = pred.to(DEV).requires_grad_(True)
    loss, acc = crit(p, joints.to(DEV))
    loss.backward()
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    assert torch.allclose(p.grad.cpu(), ref_grad, rtol=1e-5, atol=1e-12)
    assert np.float32(acc.item()) == np.float32(float(ref_acc))
    assert np.array_equal(crit.weights.cpu().numpy(), w_np)
    assert_targets_match(crit.targets.cpu().numpy(), t_np)
    # identical to the two separate kernels
    t2, w2 = api.transforms.encode_heat_maps(joints.to(DEV), 2.0, (w, h))
    p2 = pred.to(DEV).requires_grad_(True)
    l2 = api.loss.JointsMSELoss()(p2, t2, w2)
    l2.backward()
    assert torch.equal(p2.grad, p.grad) and torch.equal(t2, crit.targets)
    assert abs(l2.item() - loss.item()) <= 1e-6 * abs(l2.item())
    # plain variant (no acc, no targets kept), upstream gradient != 1
    crit2 = api.loss.EncodeJointsMSELoss()
    p3 = pred.to(DEV).requires_grad_(True)
    l3 = crit2(p3, joints.to(DEV))
    (l3 * 8.0).backward()
    assert l3.item() == loss.item() and torch.equal(p3.grad, p.grad * 8.0)


def test_fused_acc_special_predictions(api):
    """NaN / Inf / all-negative predicted maps go through the exact argmax fallback."""
    joints = synth.joints(4, seed=5)
    joints[..., 2] = 1.0
    joints[..., 0] = joints[..., 0].clamp(5, 40)
    joints[..., 1] = joints[..., 1].clamp(5, 55)
    t_np, w_np = O.encode_batch(joints.numpy())
    tgt, msk = torch.from_numpy(t_np), torch.from_numpy(w_np)
    pred = synth.predictions_like(tgt, seed=3, noise=0.1)
    pred[0, 0, 10, 10] = float("inf")
    pred[0, 1] = -1.0
    pred[1, 2, 3, 3] = float("nan")
    m = msk[..., None, None]
    want_p, _ = O.argmax_coords(pred * m)
    want_l, _ = O.argmax_coords(tgt * m)
    out = api.loss.encode_mse_forward_backward(joints.to(DEV), pred.to(DEV), need_grad=False, want_axes=True)
    assert torch.equal(out["pred_xy"].cpu(), want_p) and torch.equal(out["label_xy"].cpu(), want_l)


# ------------------------------------------------------------------------------------ box -> affine (eval-side caller)
def test_box_affines_golden_and_oracle(api, golden):
    """sp_box_affine_f64 == the reference's box_to_center_scale + get_affine_transform, bit for bit
    (float64 matrix included), on the frozen fixtures and on seeded boxes against the oracle."""
    g = golden("affine")
    for tag in ("a", "b"):
        inp, outp = [tuple(int(v) for v in r) for r in g["shapes_" + tag]]
        out = api.naive.box_affines(g["boxes_" + tag], inp, outp, want_f64=True)
        for key, name in (("center", "center_"), ("scale", "scale_"), ("area", "area_"), ("trans_inv", "tinv_"),
                          ("trans_inv_f64", "tinv64_"), ("trans_f64", "fwd64_")):
            assert np.array_equal(bits(out[key].cpu().numpy()), bits(g[name + tag])), (tag, key)
    for inp, outp in (((192, 256), (48, 64)), ((288, 384), (72, 96)), ((256, 256), (64, 64))):
        boxes = synth.detection_boxes(3000, seed=88, ratio_exact_every=32, ratio=inp[0] / inp[1])
        c, s, a, tinv = O.box_affines(boxes.tolist(), inp, outp)
        out = api.naive.box_affines(boxes.to(DEV), inp, outp)
        assert np.array_equal(bits(out["center"].cpu().numpy()), bits(c))
        assert np.array_equal(bits(out["scale"].cpu().numpy()), bits(s))
        assert np.array_equal(bits(out["area"].cpu().numpy()), bits(a))
        assert np.array_equal(bits(out["trans_inv"].cpu().numpy()), bits(tinv))
    assert api.naive.box_affines(np.zeros((0, 4)))["trans_inv"].shape == (0, 2, 3)
    # per-sample drop-ins of commons/joint_utils.py and the batched centre/scale form
    from simple_pose_b200.commons import joint_utils as ju
    boxes, inp, outp = g["boxes_a"], (192, 256), (48, 64)
    for i in (0, 1, 2, 3, 8, 17):
        x1, y1, x2, y2 = boxes[i].tolist()
        c, s = ju.box_to_center_scale(x1, y1, x2 - x1, y2 - y1, inp[0] / inp[1])
        assert c.dtype == np.float32 and s.dtype == np.float32
        assert np.array_equal(bits(c), bits(g["center_a"][i])) and np.array_equal(bits(s), bits(g["scale_a"][i]))
        fwd, inv = ju.get_affine_transform(c, s, 0, outp)
        assert np.array_equal(bits(fwd), bits(g["fwd64_a"][i])) and np.array_equal(bits(inv), bits(g["tinv64_a"][i]))
    fwd, inv = ju.get_affine_transforms(g["center_b"], g["scale_b"], (72, 96))
    assert np.array_equal(bits(fwd.cpu().numpy()), bits(g["fwd64_b"])) and np.array_equal(bits(inv.cpu().numpy()), bits(g["tinv64_b"]))
    with pytest.raises(NotImplementedError):
        ju.get_affine_transform(c, s, 0, outp, shift=np.array([0.1, 0.0], dtype=np.float32))


def test_boxes_to_keypoints_device_resident(api):
    """Eval chain without host round trips: boxes -> trans_inv/area (device) -> decode -> pack ->
    rescore + NMS, against the oracle fed with the reference-style per-box transforms."""
    n = 200
    boxes = synth.detection_boxes(n, seed=99)
    hm = synth.heatmaps(n, seed=99)
    c, s, a, tinv = O.box_affines(boxes.tolist())
    want_xy, want_conf = O.gauss_taylor_decode(hm, torch.from_numpy(tinv))
    aff = api.naive.box_affines(boxes.to(DEV))
    xy, conf = api.metrics.GaussTaylorKeyPointDecoder()(hm.to(DEV), aff["trans_inv"])
    mag = float(np.abs(tinv[:, 0, 0]).max())
    assert (xy.cpu() - want_xy).abs().max().item() <= 1e-4 * mag + 1e-3 and torch.equal(conf.cpu(), want_conf)
    seg = np.arange(0, n + 1, 10, dtype=np.int32)
    box_scores = torch.linspace(0.95, 0.05, n, dtype=torch.float64)
    kps = api.naive.pack_keypoints(xy, conf)
    keep, scores, _ = api.naive.rescore_and_nms(kps, box_scores, aff["area"].double(), seg)
    o_keep, o_scores, _ = O.rescore_and_nms(kps.cpu().numpy(), box_scores.numpy(), a.astype(np.float64), seg)
    assert np.array_equal(keep.cpu().numpy().astype(bool), o_keep)
    assert np.allclose(scores.cpu().numpy(), o_scores, rtol=1e-15, atol=0)


# ------------------------------------------------------------------------------------ BASELINE full sizes
def test_cfg4_full_size_decode_and_nms_vs_oracle(api):
    """BASELINE config 4: HRNet-W48 384x288 (96x72 maps) decode + OKS-NMS, batch 512 -- the
    oracle still finishes in about a second at this size, so compare directly."""
    hm = synth.heatmaps(512, height=96, width=72, seed=404)
    tinv, area = synth.inverse_affines(512, height=96, width=72, seed=404)
    ref_hsp, ref_max = O.gauss_taylor_decode(hm, None, return_heatmap_space=True)
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    hsp, mx, idx = dec.decode_with_index(hm.to(DEV))
    assert torch.equal(idx.cpu().long(), O.argmax_index(hm)) and torch.equal(mx.cpu(), ref_max)
    assert (hsp.cpu() - ref_hsp).abs().max().item() <= 1e-4
    img, conf = dec(hm.to(DEV), tinv.to(DEV))
    seg = np.concatenate([[0], np.cumsum(np.random.RandomState(0).randint(1, 40, size=64))])
    seg = np.unique(np.clip(seg, 0, 512)).astype(np.int32)
    if seg[-1] != 512:
        seg = np.append(seg, 512).astype(np.int32)
    box = torch.rand(512, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    kps = api.naive.pack_keypoints(img, conf)
    keep, scores, _ = api.naive.rescore_and_nms(kps, box, area, seg)
    o_keep, o_scores, _ = O.rescore_and_nms(kps.cpu().numpy(), box.numpy(), area.numpy(), seg)
    assert np.array_equal(keep.cpu().numpy().astype(bool), o_keep)
    assert np.allclose(scores.cpu().numpy(), o_scores, rtol=1e-15, atol=0)


def test_cfg5_coco_val_sized_job_properties(api):
    """BASELINE config 5: ~104k persons (21.7 GB of 64x48 maps, > 2^31 bytes). Too big for the
    oracle; checked through size-independent properties: (1) one launch == the same job in 8
    shards, bit for bit; (2) argmax / max agree with torch.max on the device; (3) a sample of
    persons agrees with the oracle; (4) encode -> decode round trip at full size."""
    free, _ = torch.cuda.mem_get_info()
    if free < 60e9:
        pytest.skip("needs ~50 GB of free device memory")
    P = 104_000
    hm = synth.heatmaps(P, seed=505, device=DEV)
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    hsp, mx, idx = dec.decode_with_index(hm)
    cuts = np.linspace(0, P, 9).astype(int)
    for a, b in zip(cuts[:-1], cuts[1:]):
        h2, m2, i2 = dec.decode_with_index(hm[a:b])
        assert torch.equal(h2, hsp[a:b]) and torch.equal(m2, mx[a:b]) and torch.equal(i2, idx[a:b])
    tmax, targ = hm.view(P, 17, -1).max(dim=-1)
    assert torch.equal(targ.int(), idx) and torch.equal(tmax[..., None], mx)
    pick = torch.randint(0, P, (96,), generator=torch.Generator().manual_seed(0))
    pick[0], pick[-1] = 0, P - 1
    ref_hsp, ref_max = O.gauss_taylor_decode(hm[pick.to(DEV)].cpu(), None, return_heatmap_space=True)
    assert (hsp[pick.to(DEV)].cpu() - ref_hsp).abs().max().item() <= 1e-4
    assert torch.isfinite(hsp).all()
    del hm, tmax, targ
    torch.cuda.empty_cache()
    g = torch.Generator(device=DEV).manual_seed(9)
    mu = torch.rand(P, 17, 2, generator=g, device=DEV)
    mu[..., 0] = 9 + mu[..., 0] * (48 - 19)
    mu[..., 1] = 9 + mu[..., 1] * (64 - 19)
    joints = torch.cat([mu, torch.ones(P, 17, 1, device=DEV)], -1)
    t, wt = api.transforms.encode_heat_maps(joints)
    xy, conf = dec(t, synth.identity_affines(P, device=DEV))
    assert (xy - mu).abs().max().item() < 1e-3 and (wt == 1).all() and (conf > 0.77).all()


@pytest.mark.parametrize("env", [{"SP_TRAIN_FORCE_LDG": "1"}, {"SP_TRAIN_WARPS": "3", "SP_TRAIN_RING": "2"},
                                 {"SP_TRAIN_RING": "1"}, {"SP_TRAIN_RING": "4", "SP_TRAIN_CHUNK_QUADS": "64"},
                                 {"SP_TRAIN_CHUNK_QUADS": "768", "SP_TRAIN_RING": "1"}, {"SP_TRAIN_WARPS": "1", "SP_TRAIN_RING": "8"},
                                 {"SP_TRAIN_NO_TILE": "1"}, {"SP_TRAIN_NO_TILE": "1", "SP_TRAIN_RING": "3", "SP_TRAIN_WARPS": "5"},
                                 {"SP_TRAIN_WARPS": "3"}, {"SP_TRAIN_WARPS": "7"}, {"SP_TRAIN_WARPS": "1"}, {"SP_NO_PDL": "1"}])
@pytest.mark.parametrize("hw", [(64, 48), (96, 72)])
def test_fused_kernel_variants_agree(api, env, hw):
    """The period-tiled kernel with full and partial CTAs, every chunk/ring/warp layout of the generic
    TMA ring and the plain-load variant give identical outputs (weights 0, 1 and odd values all present)."""
    h, w = hw
    joints = synth.joints(40, height=h, width=w, seed=81)
    joints[3, :, 2] = 2.0
    joints[5, :, 2] = 0.75
    joints[7, :, 2] = 0.25
    joints = joints.to(DEV)
    pred = synth.heatmaps(40, height=h, width=w, seed=82).to(DEV)
    pred[1, 2, 5, 7] = float("nan")
    pred[2, 3] = -1.0
    pred[2, 4] = float("-inf")
    pred[4, 0, h - 1, w - 1] = float("inf")
    base = api.loss.encode_mse_forward_backward(joints, pred, want_targets=True, want_axes=True)
    slim = api.loss.encode_mse_forward_backward(joints, pred, want_axes=True)
    bare = api.loss.encode_mse_forward_backward(joints, pred)
    os.environ.update(env)
    api.abi.reload_tuning()
    try:
        other = api.loss.encode_mse_forward_backward(joints, pred, want_targets=True, want_axes=True)
        other_slim = api.loss.encode_mse_forward_backward(joints, pred, want_axes=True)
        other_bare = api.loss.encode_mse_forward_backward(joints, pred)
    finally:
        for k in env:
            del os.environ[k]
            api.abi.reload_tuning()
    for key in ("grad", "targets", "weights", "pred_xy", "label_xy"):
        assert torch.equal(base[key].nan_to_num(nan=7.0), other[key].nan_to_num(nan=7.0)), key
        for alt in (slim, other_slim):      # period-tiled kernel (no targets requested)
            if alt[key] is not None:
                assert torch.equal(base[key].nan_to_num(nan=7.0), alt[key].nan_to_num(nan=7.0)), key
    for alt in (bare, other_bare):
        assert torch.equal(base["grad"].nan_to_num(nan=7.0), alt["grad"].nan_to_num(nan=7.0))
        assert torch.equal(base["weights"], alt["weights"])
    # the odd-weight / special-value maps against torch on the device
    m = base["weights"][..., None, None]
    tv, ti = (pred * m).flatten(2).max(dim=-1)
    want_xy = torch.stack([(ti % w).float(), (ti // w).float()], -1) * (tv > 0)[..., None]
    assert torch.equal(base["pred_xy"], want_xy)
    lv, li = (base["targets"] * m).flatten(2).max(dim=-1)
    want_l = torch.stack([(li % w).float(), (li // w).float()], -1) * (lv > 0)[..., None]
    assert torch.equal(base["label_xy"], want_l)


def test_fused_label_argmax_ties_and_outside_centres(api):
    """The analytic target argmax (3x3 block around the rounded centre) must reproduce torch.max's
    first-index rule on exact ties (half-integer centres), near ties, centres outside the map and
    non-unit weights."""
    g = torch.Generator().manual_seed(17)
    j = synth.joints(256, seed=91)
    j[:64, :, 0] = torch.randint(-7, 54, (64, 17), generator=g).float() + 0.5          # exact x ties
    j[32:96, :, 1] = torch.randint(-7, 70, (64, 17), generator=g).float() + 0.5        # exact y ties
    j[96:128, :, 0] = torch.randint(0, 47, (32, 17), generator=g).float() + 0.5 + 1e-6 * torch.randn(32, 17, generator=g)
    j[128:160, :, 2] = 2.0                                                               # weight 2 (COCO "visible")
    j[160:176, :, 2] = 0.75                                                              # odd weight
    t_np, w_np = O.encode_batch(j.numpy())
    m = torch.from_numpy(w_np)[..., None, None]
    want, _ = O.argmax_coords(torch.from_numpy(t_np) * m)
    pred = torch.zeros(256, 17, 64, 48, device=DEV)
    out = api.loss.encode_mse_forward_backward(j.to(DEV), pred, need_grad=False, want_axes=True)
    assert torch.equal(out["label_xy"].cpu(), want)
    os.environ["SP_TRAIN_FORCE_LDG"] = "1"
    api.abi.reload_tuning()
    try:
        out2 = api.loss.encode_mse_forward_backward(j.to(DEV), pred, need_grad=False, want_axes=True)
    finally:
        del os.environ["SP_TRAIN_FORCE_LDG"]
        api.abi.reload_tuning()
    assert torch.equal(out2["label_xy"].cpu(), want)
    # sigma outside the analytic range falls back to the tracked argmax
    t3 = np.stack([O.encode_person(x, 0.2, (48, 64))[0] for x in j.numpy()[:8]])
    w3 = np.stack([O.encode_person(x, 0.2, (48, 64))[1] for x in j.numpy()[:8]])
    want3, _ = O.argmax_coords(torch.from_numpy(t3) * torch.from_numpy(w3)[..., None, None])
    out3 = api.loss.encode_mse_forward_backward(j[:8].to(DEV), pred[:8], sigma=0.2, need_grad=False, want_axes=True)
    assert torch.equal(out3["label_xy"].cpu(), want3)


# --------------------------------------------------------------- kernel layouts and launch ordering
@pytest.mark.parametrize("env", [{"SP_LOSS_FORCE_LDG": "1"}, {"SP_LOSS_WARPS": "1", "SP_LOSS_RING": "1"},
                                 {"SP_LOSS_WARPS": "7", "SP_LOSS_RING": "4", "SP_LOSS_CHUNK_QUADS": "64"},
                                 {"SP_LOSS_WARPS": "32", "SP_LOSS_RING": "2", "SP_LOSS_CHUNK_QUADS": "96"},
                                 {"SP_LOSS_CHUNK_QUADS": "768", "SP_LOSS_RING": "8"},
                                 {"SP_LOSS_CHUNK_QUADS": "100"}, {"SP_NO_PDL": "1"}])
@pytest.mark.parametrize("b,hw", [(40, (64, 48)), (3, (96, 72)), (9, (20, 12))])
def test_loss_kernel_variants_agree(api, env, b, hw):
    """Every chunk/ring/warp layout of the TMA-ring loss kernel, the plain-load fallback and the
    non-PDL launch give bit-identical gradients and the same loss (float64 partial order aside)."""
    h, w = hw
    tgt = synth.heatmaps(b, height=h, width=w, seed=11).to(DEV)
    msk = (torch.rand(b, 17, generator=torch.Generator().manual_seed(12)) > 0.25).float().to(DEV)
    msk[0, 0] = 2.0                                                # non-unit weight
    pred = synth.predictions_like(tgt.cpu(), seed=13).to(DEV)
    base_loss, base_grad = api.loss.mse_forward_backward(pred, tgt, msk)
    fwd_only, none = api.loss.mse_forward_backward(pred, tgt, msk, need_grad=False)
    assert none is None and fwd_only.item() == base_loss.item()
    os.environ.update(env)
    api.abi.reload_tuning()
    try:
        loss, grad = api.loss.mse_forward_backward(pred, tgt, msk)
        loss_f, _ = api.loss.mse_forward_backward(pred, tgt, msk, need_grad=False)
    finally:
        for k in env:
            del os.environ[k]
            api.abi.reload_tuning()
    assert torch.equal(grad, base_grad)
    assert abs(loss.item() - base_loss.item()) <= 1e-6 * abs(base_loss.item())
    assert loss_f.item() == loss.item()
    ref_loss, ref_grad = O.masked_mse_loss_and_grad(pred.cpu(), tgt.cpu(), msk.cpu())
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    assert torch.allclose(grad.cpu(), ref_grad, rtol=1e-5, atol=1e-12)


def test_back_to_back_dependent_launches(api):
    """Programmatic dependent launch: every kernel may be scheduled while its predecessor drains, so
    the chain encode -> loss (reads the targets just written, RAW) -> decode (reads the gradient
    just written) -> encode (overwrites the targets the loss was reading, WAR), issued 40 times
    without any host synchronisation, must give exactly what the stream-ordered launches give."""
    from simple_pose_b200.pipeline import HeatmapHotPath
    n, rounds = 96, 40
    hp = HeatmapHotPath(n, 17, 64, 48, device=torch.device(DEV))
    joints = [synth.joints(n, seed=200 + i).to(DEV) for i in range(4)]
    pred = [synth.heatmaps(n, seed=300 + i).to(DEV) for i in range(4)]
    ident = synth.identity_affines(n, device=DEV)
    losses = torch.zeros(rounds, device=DEV)
    coords = torch.zeros(rounds, n, 17, 2, device=DEV)

    def chain(sync):
        losses.zero_()
        coords.zero_()
        for r in range(rounds):
            hp.encode(joints[r % 4])
            hp.loss_fwd_bwd(pred[r % 4])
            hp.decode(hp.targets, ident)             # decodes what the encoder of this round wrote
            losses[r].copy_(hp.loss)
            coords[r].copy_(hp.coords)
            hp.train_fused(joints[(r + 1) % 4], pred[r % 4])    # same loss buffer, different value
            if sync:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        return losses.clone(), coords.clone()

    os.environ["SP_NO_PDL"] = "1"
    api.abi.reload_tuning()
    try:
        want_l, want_c = chain(sync=True)
    finally:
        del os.environ["SP_NO_PDL"]
        api.abi.reload_tuning()
    for _ in range(3):
        got_l, got_c = chain(sync=False)
        assert torch.equal(got_l, want_l) and torch.equal(got_c, want_c)
    assert len(set(want_l.tolist())) >= 4            # the four input sets really differ


@pytest.mark.parametrize("b,k", [(1, 1), (1, 17), (3, 17), (9, 16), (149, 1), (31, 5)])
def test_decode_work_distribution_covers_every_map(api, b, k):
    """CTAs own contiguous map ranges and their warps claim maps dynamically: every output slot is
    written exactly once for map counts below, at and above the CTA / warp counts."""
    hm = synth.heatmaps(b, joints=k, seed=21).to(DEV)
    dec = api.metrics.GaussTaylorKeyPointDecoder(num_joints=k)
    got = dec.decode_with_index(hm)
    os.environ["SP_DECODE_FORCE_GENERIC"] = "1"
    api.abi.reload_tuning()
    try:
        want = dec.decode_with_index(hm)
    finally:
        del os.environ["SP_DECODE_FORCE_GENERIC"]
        api.abi.reload_tuning()
    assert torch.equal(got[2], want[2]) and torch.equal(got[1], want[1])
    assert (got[0] - want[0]).abs().max().item() <= 1e-5
    assert torch.equal(got[2].long().cpu(), O.argmax_index(hm.cpu()))


@pytest.mark.parametrize("b,hw,flip", [(300, (64, 48), False), (64, (96, 72), True), (2, (64, 48), True), (700, (32, 24), False)])
def test_decode_grid_wide_dealing_equals_equal_ranges(api, b, hw, flip):
    """sp_decode_ws_f32 (maps dealt grid-wide from the workspace counter, what the Python API calls) and
    sp_decode_f32 (equal per-CTA ranges) return identical bits; the workspace is back at zero after
    every call, also after many back-to-back launches on one stream."""
    h, w = hw
    hm = synth.heatmaps(b, height=h, width=w, seed=91).to(DEV)
    hf = synth.heatmaps(b, height=h, width=w, seed=92).to(DEV) if flip else None
    tinv = synth.inverse_affines(b, height=h, width=w, seed=91)[0].to(DEV)
    dec = api.metrics.GaussTaylorKeyPointDecoder()
    run = (lambda: dec.flip_call(hm, hf, tinv)) if flip else (lambda: dec(hm, tinv))
    os.environ["SP_DECODE_GRID_WIDE"] = "1"              # by default only large launches and items >= 40 KB are dealt grid-wide
    api.abi.reload_tuning()
    try:
        got = [run() for _ in range(6)]
        for pct in ("0", "40", "85", "100", "300"):        # static interleaved share of a warp's maps, the rest claimed dynamically
            os.environ["SP_DECODE_STATIC_PCT"] = pct
            api.abi.reload_tuning()
            got.append(run())
        del os.environ["SP_DECODE_STATIC_PCT"]
        os.environ["SP_DECODE_GRID_WIDE"] = "0"
        api.abi.reload_tuning()
        want = run()
    finally:
        os.environ.pop("SP_DECODE_STATIC_PCT", None)
        del os.environ["SP_DECODE_GRID_WIDE"]
        api.abi.reload_tuning()
    got.append(run())                                    # the default policy
    for c, m in got:
        assert torch.equal(c, want[0]) and torch.equal(m, want[1])
    ws = api.abi.scratch(torch.device(DEV), api.abi.stream_ptr(torch.device(DEV)), 16, "decode")
    torch.cuda.synchronize()
    assert int(ws.abs().sum().item()) == 0
    lib = api.abi.lib()
    assert lib.sp_decode_ws_f32(hm.data_ptr(), None, None, None, dec._weights_on(hm.device).data_ptr(), got[0][0].data_ptr(),
                                got[0][1].data_ptr(), None, b, 17, h, w, 11, 0, None, 16, None) == -1
    assert lib.sp_decode_ws_f32(hm.data_ptr(), None, None, None, dec._weights_on(hm.device).data_ptr(), got[0][0].data_ptr(),
                                got[0][1].data_ptr(), None, b, 17, h, w, 11, 0, ws.data_ptr(), 8, None) == -3


# ------------------------------------------------------------------------------------ train-side caller of the encoder
def _oracle_train_geometry(smp, inp, outp, n=None):
    n = smp["boxes"].shape[0] if n is None else n
    return [O.train_sample_geometry(smp["boxes"][i].tolist(), int(smp["img_w"][i]), np.asarray(smp["joints"][i]),
                                    float(smp["scale_ratio"][i]), float(smp["rot"][i]), bool(smp["flip"][i]),
                                    input_shape=inp, output_shape=outp) for i in range(n)]


def _assert_joints_close(got, want):
    """float32 joints: at most 1 ulp apart and all but a vanishing fraction identical (the float64 dot
    is FMA-ordered on both sides; a last-bit float64 difference flips a float32 rounding ~1e-8 of the time)."""
    d = ulp_diff(got, want)
    assert d.max() <= 1 and (d != 0).mean() < 1e-4, (d.max(), (d != 0).mean())


def test_train_geometry_golden(api, golden):
    """sp_train_geometry_f32 + sp_encode_f32 against the frozen products of the reference's own
    RefineSimpleTransform.__call__ (scripted draws): trans_inv float64 bit-identical (rot = 0) or within
    the sin/cos last-bit allowance, input-pixel joints, masks, heat maps."""
    g = golden("train_geom")
    for tag in ("a", "b"):
        inp, outp = [tuple(int(v) for v in r) for r in g["shapes_" + tag]]
        args = (g["boxes_" + tag], g["joints_" + tag], g["img_w_" + tag], g["scale_ratio_" + tag], g["rot_" + tag],
                g["flip_" + tag].astype(np.uint8))
        geo = api.transforms.train_geometry(*args, input_shape=inp, output_shape=outp, want_input=True)
        tinv = geo["trans_inv_f64"].cpu().numpy()
        same = np.array([np.array_equal(bits(tinv[i]), bits(g["tinv64_" + tag][i])) for i in range(tinv.shape[0])])
        assert same[g["rot_" + tag] == 0].all()
        assert same.mean() >= 0.9 and np.allclose(tinv, g["tinv64_" + tag], rtol=1e-6, atol=1e-6)
        assert np.array_equal(bits(geo["trans_inv"].cpu().numpy()[same]), bits(g["tinv64_" + tag].astype(np.float32)[same]))
        _assert_joints_close(geo["joints_input"].cpu().numpy()[same], g["joints_input_" + tag][same])
        heat_maps, masks, tinv32 = api.transforms.train_targets(*args, input_shape=inp, output_shape=outp)
        assert np.array_equal(masks.cpu().numpy()[same], g["mask_" + tag][same])
        assert torch.equal(tinv32, geo["trans_inv"])
        orc = _oracle_train_geometry({k: g[k + "_" + tag] for k in ("boxes", "img_w", "joints", "scale_ratio", "rot", "flip")},
                                     inp, outp, n=g["heat_map_" + tag].shape[0])
        for i, o in enumerate(orc):
            assert np.array_equal(bits(o["heat_map"]), bits(g["heat_map_" + tag][i]))         # the oracle is pinned ...
            if np.array_equal(bits(geo["joints_hm"][i].cpu().numpy()), bits(o["joints_hm"])):  # ... and so is the kernel
                assert_targets_match(heat_maps[i].cpu().numpy(), g["heat_map_" + tag][i])
            else:
                assert (not same[i]) or ulp_diff(geo["joints_hm"][i].cpu().numpy(), o["joints_hm"]).max() <= 1


@pytest.mark.parametrize("inp,outp", [((192, 256), (48, 64)), ((288, 384), (72, 96))])
def test_train_geometry_vs_oracle(api, inp, outp):
    n = 1500
    smp = synth.train_samples(n, seed=404)
    orc = _oracle_train_geometry(smp, inp, outp)
    geo = api.transforms.train_geometry(smp["boxes"], smp["joints"], smp["img_w"], smp["scale_ratio"], smp["rot"],
                                        smp["flip"], input_shape=inp, output_shape=outp, want_input=True)
    torch.cuda.synchronize()
    tinv = geo["trans_inv_f64"].cpu().numpy()
    fwd_in = geo["img_trans_f64"].cpu().numpy()
    same = np.array([np.array_equal(bits(tinv[i]), bits(orc[i]["trans_inv"])) and
                     np.array_equal(bits(fwd_in[i]), bits(orc[i]["img_trans"])) for i in range(n)])
    assert same.mean() >= 0.999, "persons with a non-identical float64 affine: %d of %d" % ((~same).sum(), n)
    assert np.allclose(tinv, np.stack([o["trans_inv"] for o in orc]), rtol=1e-6, atol=1e-6)
    for key in ("center", "scale"):
        assert np.array_equal(bits(geo[key].cpu().numpy()), bits(np.stack([o[key] for o in orc]))), key
    _assert_joints_close(geo["joints_hm"].cpu().numpy()[same], np.stack([o["joints_hm"] for o in orc])[same])
    _assert_joints_close(geo["joints_input"].cpu().numpy()[same], np.stack([o["joints_input"] for o in orc])[same])
    # the composed product the solvers consume: masks exact, maps as the encoder's gate
    heat_maps, masks, _ = api.transforms.train_targets(smp["boxes"][:96], smp["joints"][:96], smp["img_w"][:96],
                                                       smp["scale_ratio"][:96], smp["rot"][:96], smp["flip"][:96],
                                                       input_shape=inp, output_shape=outp)
    jh = geo["joints_hm"].cpu().numpy()
    for i in range(96):
        if np.array_equal(bits(jh[i]), bits(orc[i]["joints_hm"])):
            assert np.array_equal(masks[i].cpu().numpy(), orc[i]["mask"])
            assert_targets_match(heat_maps[i].cpu().numpy(), orc[i]["heat_map"])
    assert 0 < masks.sum().item() < masks.numel()


def test_train_targets_basic_transform(api):
    """BasicSimpleTransform.joint_targets (train_geometry -> input-pixel joints -> quantised encoder) vs the
    pinned restatement of the reference's BasicSimpleTransform.__call__."""
    n = 200
    smp = synth.train_samples(n, seed=707)
    tr = api.transforms.BasicSimpleTransform(joint_pairs=[list(p) for p in O.COCO_JOINT_PAIRS])
    hm, mk, tinv = tr.joint_targets(smp["boxes"], smp["joints"], smp["img_w"], smp["scale_ratio"], smp["rot"], smp["flip"])
    geo = api.transforms.train_geometry(smp["boxes"], smp["joints"], smp["img_w"], smp["scale_ratio"], smp["rot"], smp["flip"],
                                        want_input=True)
    checked = 0
    for i in range(n):
        o = O.train_sample_geometry(smp["boxes"][i].tolist(), int(smp["img_w"][i]), smp["joints"][i].numpy(),
                                    float(smp["scale_ratio"][i]), float(smp["rot"][i]), bool(smp["flip"][i]), basic=True)
        if np.array_equal(bits(geo["joints_input"][i].cpu().numpy()), bits(o["joints_input"])):
            assert np.array_equal(bits(hm[i].cpu().numpy()), bits(o["heat_map"])) and np.array_equal(mk[i].cpu().numpy(), o["mask"]), i
            assert np.array_equal(bits(tinv[i].cpu().numpy()), bits(o["trans_inv"].astype(np.float32)))
            checked += 1
    assert checked >= n - 2


def test_train_geometry_drop_ins_and_edges(api):
    """Per-sample drop-ins of commons/joint_utils.py (flip_joints, affine_transform_batch,
    get_affine_transform with a rotation) and the degenerate batches."""
    from simple_pose_b200.commons import joint_utils as ju
    smp = synth.train_samples(12, seed=505)
    pairs = [list(p) for p in O.COCO_JOINT_PAIRS]
    for i in range(12):
        j = smp["joints"][i].numpy()
        w = int(smp["img_w"][i])
        img = np.arange(2 * w * 3, dtype=np.uint8).reshape(2, w, 3)
        fimg, fj = ju.flip_joints(img, j, pairs)
        assert np.array_equal(fimg, img[:, ::-1]) and np.array_equal(bits(fj), bits(O.flip_joints_only(j, w)))
        o = O.train_sample_geometry(smp["boxes"][i].tolist(), w, j, float(smp["scale_ratio"][i]), float(smp["rot"][i]), False)
        fwd, inv = ju.get_affine_transform(o["center"], o["scale"], float(smp["rot"][i]), (48, 64))
        assert np.allclose(fwd, o["joint_trans"], rtol=1e-12, atol=1e-12) and np.allclose(inv, o["trans_inv"], rtol=1e-12, atol=1e-12)
        aj = ju.affine_transform_batch(j, o["joint_trans"])
        assert aj.dtype == np.float32
        _assert_joints_close(aj, O.affine_joints(j, o["joint_trans"]))
    # no flip / no rotation / no scale draw == the eval-side transform, bit for bit
    boxes = synth.detection_boxes(300, seed=606)
    j = synth.train_samples(300, seed=606)["joints"]
    geo = api.transforms.train_geometry(boxes, j)
    ref = api.naive.box_affines(boxes.to(DEV), want_f64=True)
    assert torch.equal(geo["trans_inv_f64"], ref["trans_inv_f64"]) and torch.equal(geo["center"], ref["center"])
    assert torch.equal(geo["scale"], ref["scale"])
    # invisible rows are never mapped; K = 1; empty batch
    j1 = torch.tensor([[[5.0, 6.0, 0.0]], [[5.0, 6.0, 1.0]]])
    g1 = api.transforms.train_geometry(boxes[:2], j1)
    assert g1["joints_hm"][0].cpu().tolist() == [[5.0, 6.0, 0.0]] and g1["joints_hm"][1, 0, 2].item() == 1.0
    assert g1["joints_hm"][1, 0, 0].item() != 5.0
    empty = api.transforms.train_geometry(np.zeros((0, 4)), np.zeros((0, 17, 3), dtype=np.float32))
    assert empty["joints_hm"].shape == (0, 17, 3) and empty["trans_inv"].shape == (0, 2, 3)
    with pytest.raises(ValueError):
        api.transforms.train_geometry(boxes[:2], j1, flip=[1, 0])
    lib = api.abi.lib()
    d = torch.zeros(64, device=DEV, dtype=torch.float64)
    f = torch.zeros(64, device=DEV)
    u8 = torch.ones(8, device=DEV, dtype=torch.uint8)
    assert lib.sp_train_geometry_f32(d.data_ptr(), None, f.data_ptr(), None, None, u8.data_ptr(), None, f.data_ptr(), None,
                                     None, None, None, None, None, 1, 1, 192, 256, 48, 64, 1.25, None) == -1
    assert lib.sp_transform_joints_f32(f.data_ptr(), None, None, None, None, f.data_ptr(), 1, 1, None) == -1


# ------------------------------------------------------------------------------------ entry points without a Python caller
def test_center_scale_affine_entry_point_and_device_info(api, golden):
    """sp_center_scale_affine_f64 (get_affine_transform with rot = 0 for given centre/scale pairs) is what a host that already
    holds centres and scales binds; the Python mirror goes through the rotation entry point, so this one is called directly:
    float64 matrices bit-identical to the reference fixtures, the float32 inverse = the float64 one rounded once.
    sp_device_info must describe the device the kernels were built for."""
    import ctypes
    g = golden("affine")
    lib = api.abi.lib()
    for tag, outp in (("a", (48, 64)), ("b", (72, 96))):
        c = torch.from_numpy(g["center_" + tag]).to(DEV).contiguous()
        s = torch.from_numpy(g["scale_" + tag]).to(DEV).contiguous()
        n = int(c.shape[0])
        inv32 = torch.empty((n, 2, 3), dtype=torch.float32, device=DEV)
        inv64 = torch.empty((n, 2, 3), dtype=torch.float64, device=DEV)
        fwd64 = torch.empty((n, 2, 3), dtype=torch.float64, device=DEV)
        with torch.cuda.device(DEV):
            api.abi.check(lib.sp_center_scale_affine_f64(c.data_ptr(), s.data_ptr(), inv32.data_ptr(), inv64.data_ptr(),
                                                        fwd64.data_ptr(), n, outp[0], outp[1], api.abi.stream_ptr(c.device)))
        torch.cuda.synchronize()
        assert np.array_equal(bits(fwd64.cpu().numpy()), bits(g["fwd64_" + tag])), tag
        assert np.array_equal(bits(inv64.cpu().numpy()), bits(g["tinv64_" + tag])), tag
        assert np.array_equal(bits(inv32.cpu().numpy()), bits(g["tinv_" + tag])), tag
        only = torch.empty((n, 2, 3), dtype=torch.float32, device=DEV)         # any subset of the outputs
        with torch.cuda.device(DEV):
            api.abi.check(lib.sp_center_scale_affine_f64(c.data_ptr(), s.data_ptr(), only.data_ptr(), None, None, n,
                                                        outp[0], outp[1], api.abi.stream_ptr(c.device)))
        assert torch.equal(only, inv32)
    assert lib.sp_center_scale_affine_f64(c.data_ptr(), s.data_ptr(), None, None, None, n, 48, 64, None) != 0      # no output asked for
    info = api.abi.device_info()
    props = torch.cuda.get_device_properties(0)
    assert info["sm_count"] == props.multi_processor_count and info["cc"] == (props.major, props.minor) == (10, 0)
    sm = ctypes.c_int()
    assert lib.sp_device_info(ctypes.byref(sm), None, None) == 0 and sm.value == info["sm_count"]      # outputs are optional
