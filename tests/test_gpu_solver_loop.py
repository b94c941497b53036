"""GPU: the mirrors substituted into a solver-shaped loop, and the autocast (float16 / bfloat16) loss path.

Replays the structure of the reference's ``processors/dp_pose_hrnet_solver.py`` -- ``train()`` :99-127 (plain and
``amp.autocast`` + ``GradScaler`` branches) and ``val()`` :150-161 (loss, ``HeatMapAcc``, decoder, ``kps_to_dict_``)
-- with a one-convolution stand-in for the backbone. Every quantity the loop produces from ``predicts`` is
compared with the oracle evaluated on exactly those predictions (copied to the host)."""
import os

import numpy as np
import pytest
import torch

from oracle import heatmap_oracle as O
from simple_pose_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def reference_loss_and_grad(pred, target, mask, scale=1.0):
    """The solvers' expression on host tensors (oracle restatement of dp_pose_hrnet_solver.py:106-107 / :111-120),
    differentiated by torch autograd; ``pred`` may be float16 / bfloat16."""
    return O.masked_mse_loss_and_grad_scaled(pred, target, mask, scale)


def half_ulp_distance(a, b):
    ia = a.contiguous().view(torch.int16).to(torch.int32)
    ib = b.contiguous().view(torch.int16).to(torch.int32)
    # sign-magnitude -> monotone integers
    ia = torch.where(ia < 0, -32768 - ia, ia)
    ib = torch.where(ib < 0, -32768 - ib, ib)
    return (ia - ib).abs()


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("b,hw,scale", [(32, (64, 48), 65536.0), (6, (96, 72), 1.0), (5, (10, 6), 128.0), (3, (9, 7), 8.0)])
def test_loss_native_half_precision_pred(dtype, b, hw, scale):
    """pred in the autocast dtype: loss within 1e-5 relative of the reference expression on the same half
    tensor, gradient in pred's dtype equal to autograd's (float32 arithmetic, scale applied before the cast)."""
    from simple_pose_b200.processors.loss import JointsMSELoss, mse_forward_backward
    h, w = hw
    tgt = synth.heatmaps(b, height=h, width=w, seed=41)
    msk = (torch.rand(b, 17, generator=torch.Generator().manual_seed(42)) > 0.25).float()
    msk[0, 0] = 2.0
    pred = synth.predictions_like(tgt, seed=43).to(dtype)
    ref_loss, ref_grad = reference_loss_and_grad(pred, tgt, msk, scale)
    assert ref_grad.dtype == dtype
    p = pred.to(DEV).requires_grad_(True)
    loss = JointsMSELoss()(p, tgt.to(DEV), msk.to(DEV))
    (loss * scale).backward()
    assert loss.dtype == torch.float32 and p.grad.dtype == dtype
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    d = half_ulp_distance(p.grad.cpu(), ref_grad)
    assert int(d.max()) <= 1 and float((d != 0).float().mean()) < 1e-3
    assert torch.isfinite(p.grad).all()
    if dtype == torch.float16 and scale > 1000:
        # the scale really is applied in float32 before the cast: the unscaled gradient underflows float16
        _, unscaled = reference_loss_and_grad(pred, tgt, msk, 1.0)
        assert float((unscaled == 0).float().mean()) > 0.5 > float((p.grad == 0).float().mean())
    # second backward through the same node (deferred gradient: nothing was consumed)
    p2 = pred.to(DEV).requires_grad_(True)
    l2 = JointsMSELoss()(p2, tgt.to(DEV), msk.to(DEV))
    (l2 * scale).backward(retain_graph=True)
    first = p2.grad.clone()
    p2.grad = None
    (l2 * scale).backward()
    assert torch.equal(p2.grad, first)
    # forward only under no_grad: no gradient buffer, same loss
    with torch.no_grad():
        l3 = JointsMSELoss()(p, tgt.to(DEV), msk.to(DEV))
    assert l3.item() == loss.item() and not l3.requires_grad
    # raw call: backward only
    none, g = mse_forward_backward(pred.to(DEV), tgt.to(DEV), msk.to(DEV), need_loss=False,
                                   grad_scale_dev=torch.tensor(scale, device=DEV))
    assert none is None and torch.equal(g, p.grad)


def test_round2_golden_fixtures(golden):
    """The CUDA path against outputs of the reference itself frozen in tests/golden/round2.npz: float16 / bfloat16 loss and
    gradient (the solvers' AMP expression), kps_to_dict_, NMS with tied scores de-tied by the documented rule."""
    from simple_pose_b200.datasets.naive_data import oks_nms
    from simple_pose_b200.metrics.pose_metrics import kps_to_dict_
    from simple_pose_b200.processors.loss import JointsMSELoss
    g = golden("round2")
    target, mask = torch.from_numpy(g["amp_target"]).to(DEV), torch.from_numpy(g["amp_mask"]).to(DEV)
    for name, dtype in (("f16", torch.float16), ("bf16", torch.bfloat16)):
        p = torch.from_numpy(g["amp_%s_pred_bits" % name]).view(dtype).to(DEV).requires_grad_(True)
        loss = JointsMSELoss()(p, target, mask)
        (loss * float(g["amp_%s_scale" % name])).backward()
        want_loss = float(g["amp_%s_loss" % name])
        assert abs(loss.item() - want_loss) <= 1e-5 * abs(want_loss)
        want = torch.from_numpy(g["amp_%s_grad_bits" % name]).view(dtype)
        d = half_ulp_distance(p.grad.cpu(), want)
        assert p.grad.dtype == dtype and int(d.max()) <= 1 and float((d != 0).float().mean()) < 1e-3
    out = []
    kps_to_dict_(torch.from_numpy(g["dict_coords"]).to(DEV), torch.from_numpy(g["dict_conf"]).to(DEV), g["dict_image_id"].tolist(), out)
    assert [r["keypoints"] for r in out] == g["dict_keypoints"].tolist()
    assert [r["image_id"] for r in out] == g["dict_image_id"].tolist()
    assert np.allclose([r["score"] for r in out], g["dict_score"], rtol=2.4e-7, atol=0)
    assert oks_nms(g["tie_kps"], g["tie_scores"], g["tie_area"], 0.9) == g["tie_keep"].tolist()


def test_float32_loss_node_is_single_use_unless_deferred():
    from simple_pose_b200.processors.loss import JointsMSELoss
    tgt = synth.heatmaps(4, seed=3).to(DEV)
    msk = torch.ones(4, 17, device=DEV)
    pred = synth.predictions_like(tgt, seed=4)
    p = pred.clone().requires_grad_(True)
    loss = JointsMSELoss()(p, tgt, msk)
    (loss * 4.0).backward(retain_graph=True)
    want = p.grad.clone()
    with pytest.raises(RuntimeError, match="defer_grad"):
        (loss * 4.0).backward()
    q = pred.clone().requires_grad_(True)
    l2 = JointsMSELoss(defer_grad=True)(q, tgt, msk)
    (l2 * 4.0).backward(retain_graph=True)
    (l2 * 4.0).backward()
    assert l2.item() == loss.item() and torch.equal(q.grad, 2 * want)      # accumulated twice, each exact
    # under no_grad nothing the size of pred is allocated or written
    with torch.no_grad():
        JointsMSELoss()(p, tgt, msk)                  # (the reduction workspace of this stream exists from here on)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    with torch.no_grad():
        l3 = JointsMSELoss()(p, tgt, msk)
    torch.cuda.synchronize()
    assert l3.item() == loss.item()
    assert torch.cuda.max_memory_allocated() - before < pred.numel() * 4 // 2      # no gradient-sized buffer


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_fused_encode_loss_native_half_precision_pred(dtype):
    from simple_pose_b200.processors.loss import EncodeJointsMSELoss
    b = 24
    joints = synth.joints(b, seed=51)
    t_np, w_np = O.encode_batch(joints.numpy())
    tgt, msk = torch.from_numpy(t_np), torch.from_numpy(w_np)
    pred = synth.predictions_like(tgt, seed=52).to(dtype)
    scale = 4096.0
    ref_loss, ref_grad = reference_loss_and_grad(pred, tgt, msk, scale)
    ref_acc = O.heat_map_acc(pred.float() * msk[..., None, None], tgt * msk[..., None, None])
    crit = EncodeJointsMSELoss(with_acc=True)
    p = pred.to(DEV).requires_grad_(True)
    loss, acc = crit(p, joints.to(DEV))
    (loss * scale).backward()
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    assert acc.item() == float(ref_acc)
    assert torch.equal(crit.weights.cpu(), msk)
    d = half_ulp_distance(p.grad.cpu(), ref_grad)
    assert p.grad.dtype == dtype and int(d.max()) <= 1 and float((d != 0).float().mean()) < 1e-3


class StandInBackbone(torch.nn.Module):
    """One 3x3 convolution + 4x average pooling: [B,3,256,192] -> [B,17,64,48] (the solvers' model slot)."""

    def __init__(self):
        super().__init__()
        self.conv = torch.nn.Conv2d(3, 17, 3, padding=1)
        self.pool = torch.nn.AvgPool2d(4)

    def forward(self, x):
        return self.pool(self.conv(x))


@pytest.mark.parametrize("amp", [False, True])
@pytest.mark.parametrize("fused_targets", [False, True])
def test_train_loop_of_the_hrnet_solver(amp, fused_targets):
    """dp_pose_hrnet_solver.py:99-127 with JointsMSELoss / EncodeJointsMSELoss and HeatMapAcc substituted."""
    from simple_pose_b200.commons.transforms import encode_heat_maps
    from simple_pose_b200.metrics.pose_metrics import HeatMapAcc
    from simple_pose_b200.processors.loss import EncodeJointsMSELoss, JointsMSELoss
    torch.manual_seed(0)
    model = StandInBackbone().to(DEV)
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler("cuda", init_scale=1024.0) if amp else None
    creterion = EncodeJointsMSELoss(with_acc=True) if fused_targets else JointsMSELoss()
    acc_func = HeatMapAcc()
    losses = []
    for it in range(3):
        input_img = torch.randn(8, 3, 256, 192, generator=torch.Generator().manual_seed(it)).to(DEV)
        joints = synth.joints(8, seed=100 + it).to(DEV)
        targets, mask = encode_heat_maps(joints)                  # what the loader ships (heat_maps, masks)
        captured = {}
        optimizer.zero_grad()
        with torch.autocast("cuda", enabled=amp):
            predicts = model(input_img)
            predicts.register_hook(lambda g: captured.__setitem__("grad", g))
            if fused_targets:
                loss, acc = creterion(predicts, joints)
            else:
                loss = creterion(predicts, targets, mask)
        if scaler is None:
            loss.backward()
            optimizer.step()
            scale = 1.0
        else:
            scale = float(scaler.get_scale())
            scaler.scale(loss).backward()
            scaler.step(optimizer)
            scaler.update()
        if not fused_targets:
            acc = acc_func(predicts.mul(mask[..., None, None]).detach(), targets.mul(mask[..., None, None]).detach())
        # ---- the oracle on exactly these predictions
        assert predicts.dtype == (torch.float16 if amp else torch.float32)
        p_host = predicts.detach().cpu()
        t_np, w_np = O.encode_batch(joints.cpu().numpy())
        tgt, msk = torch.from_numpy(t_np), torch.from_numpy(w_np)
        ref_loss, ref_grad = reference_loss_and_grad(p_host, tgt, msk, scale)
        assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
        ref_acc = O.heat_map_acc(p_host.float() * msk[..., None, None], tgt * msk[..., None, None])
        assert acc.item() == float(ref_acc)
        g = captured["grad"]
        assert g.dtype == predicts.dtype and g.shape == predicts.shape
        if amp:
            d = half_ulp_distance(g.cpu(), ref_grad)
            assert int(d.max()) <= 1 and float((d != 0).float().mean()) < 1e-3
        else:
            assert torch.allclose(g.cpu(), ref_grad, rtol=1e-5, atol=1e-12)
        assert all(torch.isfinite(q).all() for q in model.parameters())
        losses.append(loss.item())
    assert len(set(losses)) == 3                                   # the optimizer really stepped


def test_val_loop_of_the_hrnet_solver():
    """dp_pose_hrnet_solver.py:150-161: loss, HeatMapAcc, GaussTaylorKeyPointDecoder, kps_to_dict_ on CUDA tensors."""
    from simple_pose_b200.commons.transforms import encode_heat_maps
    from simple_pose_b200.metrics.pose_metrics import GaussTaylorKeyPointDecoder, HeatMapAcc, kps_to_dict_
    from simple_pose_b200.processors.loss import JointsMSELoss
    torch.manual_seed(1)
    model = StandInBackbone().to(DEV).eval()
    creterion, acc_func, decoder = JointsMSELoss(), HeatMapAcc(), GaussTaylorKeyPointDecoder()
    kps_dict_list, want_list = [], []
    with torch.no_grad():
        for it in range(2):
            input_img = torch.randn(6, 3, 256, 192, generator=torch.Generator().manual_seed(50 + it)).to(DEV)
            joints = synth.joints(6, seed=60 + it).to(DEV)
            targets, mask = encode_heat_maps(joints)
            tran_inv = synth.inverse_affines(6, seed=70 + it)[0].to(DEV)
            img_ids = list(range(10 * it, 10 * it + 6))
            # a trained network emits one clear peak per joint; the random stand-in alone gives flat noise whose Taylor
            # step is ill-conditioned (offsets of thousands of pixels), so its output rides on synthetic peaks
            predicts = 0.02 * model(input_img) + synth.heatmaps(6, seed=80 + it, noise=0.0).to(DEV)
            loss = creterion(predicts.clone(), targets, mask)
            acc = acc_func(predicts.mul(mask[..., None, None]), targets.mul(mask[..., None, None]))
            pred_kps, scores = decoder(predicts, tran_inv)
            kps_to_dict_(pred_kps, scores, img_ids, kps_dict_list)
            # ---- oracle on the same predictions
            p_host, t_host, m_host = predicts.cpu(), targets.cpu(), mask.cpu()
            ref_loss = O.masked_mse_loss(p_host, t_host, m_host)
            assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
            ref_acc = O.heat_map_acc(p_host * m_host[..., None, None], t_host * m_host[..., None, None])
            assert acc.item() == float(ref_acc)
            want_xy, want_conf = O.gauss_taylor_decode(p_host, tran_inv.cpu())
            mag = float(tran_inv[:, 0, 0].abs().max())
            assert (pred_kps.cpu() - want_xy).abs().max().item() <= 1e-4 * mag + 1e-3
            assert torch.equal(scores.cpu(), want_conf)
            O.kps_to_dict(pred_kps.cpu(), scores.cpu(), img_ids, want_list)
    assert len(kps_dict_list) == len(want_list) == 12
    for g, w in zip(kps_dict_list, want_list):
        assert g["image_id"] == w["image_id"] and g["category_id"] == 1 and g["keypoints"] == w["keypoints"]
        assert abs(g["score"] - w["score"]) <= 2.4e-7 * abs(w["score"])


# ------------------------------------------------------------------------------------ one-launch step (sp_step_f32)
def _separate_kernels(hp, joints, pred, tinv):
    hp.encode(joints)
    hp.loss_fwd_bwd(pred)
    hp.decode(pred, tinv)
    hp.train_fused(joints, pred, with_acc=True)          # pred_xy / label_xy of the stand-alone fused kernel
    torch.cuda.synchronize()
    return {k: getattr(hp, k).clone() for k in ("targets", "weights", "grad", "loss", "coords", "maxval", "pred_xy", "label_xy")}


@pytest.mark.parametrize("b,hw", [(128, (64, 48)), (20, (96, 72)), (9, (20, 12)), (1, (64, 48)), (300, (32, 24)), (7, (63, 48))])
def test_one_launch_step_equals_the_three_kernels(b, hw):
    """sp_step_f32 (decode + encode + loss fwd/bwd + HeatMapAcc argmaxes on one staged copy of each map) returns the
    bits of sp_encode_f32 / sp_mse_fwd_bwd_f32 / sp_decode_f32 / the fused training kernel; only the loss may differ
    in its float64 summation order. Includes odd masks, NaN / Inf predictions and all-negative maps."""
    from simple_pose_b200.pipeline import HeatmapHotPath
    h, w = hw
    joints = synth.joints(b, height=h, width=w, seed=7 * b).to(DEV)
    if b >= 9:
        joints[3, :, 2] = 0.75                           # odd mask values: the general arithmetic path
        joints[4, :5, 2] = 2.0
    pred = synth.heatmaps(b, height=h, width=w, seed=7 * b + 1, noise=0.02).to(DEV)
    if b >= 9:
        pred[1, 2, 3, 4] = float("nan")
        pred[2, 3] = -1.0
        pred[2, 4, h - 1, w - 1] = float("inf")
        pred[5, 6] = 0.0
    tinv = synth.inverse_affines(b, height=h, width=w, seed=7 * b)[0].to(DEV)
    sep = HeatmapHotPath(b, 17, h, w, device=DEV)
    want = _separate_kernels(sep, joints, pred, tinv)
    one = HeatmapHotPath(b, 17, h, w, device=DEV)
    assert one.one_launch_supported()
    for variant in ({"want_targets": True, "want_grad": True, "with_acc": True}, {"want_targets": True, "want_grad": True, "with_acc": False},
                    {"want_targets": False, "want_grad": True, "with_acc": False}, {"want_targets": False, "want_grad": False, "with_acc": True}):
        for t in (one.targets, one.grad, one.coords, one.maxval, one.weights):
            t.fill_(-7.0)
        one.step_one_launch(joints, pred, tinv, **variant)
        torch.cuda.synchronize()
        eq = lambda x, y: torch.equal(x.nan_to_num(nan=7.5), y.nan_to_num(nan=7.5))
        assert eq(one.coords, want["coords"]) and eq(one.maxval, want["maxval"]) and torch.equal(one.weights, want["weights"])
        if variant["want_targets"]:
            assert torch.equal(one.targets, want["targets"])
        else:
            assert (one.targets == -7.0).all()
        if variant["want_grad"]:
            assert eq(one.grad, want["grad"])
        else:
            assert (one.grad == -7.0).all()
        if variant["with_acc"]:
            assert torch.equal(one.pred_xy, want["pred_xy"]) and torch.equal(one.label_xy, want["label_xy"])
        lw, lg = float(want["loss"]), float(one.loss)
        assert (lw != lw and lg != lg) or abs(lg - lw) <= 1e-6 * abs(lw)
    # the default step() takes the one-launch path and the workspace is back at zero afterwards
    loss, coords, maxval = one.step(joints, pred, tinv)
    torch.cuda.synchronize()
    assert torch.equal(coords.nan_to_num(nan=7.5), want["coords"].nan_to_num(nan=7.5))
    assert int(one.ws[:2].abs().sum().item()) == 0 and int(one.dws.abs().sum().item()) == 0


@pytest.mark.parametrize("b,hw", [(520, (64, 48)), (200, (96, 72))])
@pytest.mark.parametrize("env", [{}, {"SP_STEP_STATIC_PCT": "0"}, {"SP_STEP_STATIC_PCT": "100"}, {"SP_STEP_WARPS": "3", "SP_STEP_STATIC_PCT": "30"},
                                 {"SP_STEP_WARPS": "5"}])
def test_one_launch_step_large_launch_layouts(b, hw, env):
    """Launches large enough for the few-warps configuration of sp_step_f32 with maps dealt grid-wide (every split
    between statically assigned and dynamically claimed maps): all write the bits of the stand-alone kernels, every
    map exactly once, and the work counter is back at zero."""
    from simple_pose_b200 import _abi
    from simple_pose_b200.pipeline import HeatmapHotPath
    h, w = hw
    joints = synth.joints(b, height=h, width=w, seed=b).to(DEV)
    joints[3, :, 2] = 0.75
    pred = synth.heatmaps(b, height=h, width=w, seed=b + 1, noise=0.02).to(DEV)
    pred[1, 2, 3, 4] = float("nan")
    pred[2, 3] = -1.0
    tinv = synth.inverse_affines(b, height=h, width=w, seed=b)[0].to(DEV)
    want = _separate_kernels(HeatmapHotPath(b, 17, h, w, device=DEV), joints, pred, tinv)
    one = HeatmapHotPath(b, 17, h, w, device=DEV)
    os.environ.update(env)
    _abi.reload_tuning()
    try:
        one.step_one_launch(joints, pred, tinv, with_acc=True)
        torch.cuda.synchronize()
    finally:
        for k in env:
            del os.environ[k]
        _abi.reload_tuning()
    eq = lambda x, y: torch.equal(x.nan_to_num(nan=7.5), y.nan_to_num(nan=7.5))
    for key in ("targets", "weights", "grad", "coords", "maxval", "pred_xy", "label_xy"):
        assert eq(getattr(one, key), want[key]), key
    assert int(one.ws[:2].abs().sum().item()) == 0


def test_one_launch_step_vs_oracle_and_graph_replay():
    """The captured step (one CUDA-graph launch) against the oracle, and replay after the inputs changed in place."""
    from simple_pose_b200.pipeline import HeatmapHotPath
    b = 48
    hp = HeatmapHotPath(b, 17, 64, 48, device=DEV)
    joints = torch.empty(b, 17, 3, device=DEV)
    pred = torch.empty(b, 17, 64, 48, device=DEV)
    tinv = torch.empty(b, 2, 3, device=DEV)
    joints.copy_(synth.joints(b, seed=1))
    pred.copy_(synth.heatmaps(b, seed=1))
    tinv.copy_(synth.inverse_affines(b, seed=1)[0])
    replay = hp.capture(joints, pred, tinv)
    for seed in (2, 3):
        j_host, p_host, t_host = synth.joints(b, seed=seed), synth.heatmaps(b, seed=seed, noise=0.02), synth.inverse_affines(b, seed=seed)[0]
        joints.copy_(j_host)
        pred.copy_(p_host)
        tinv.copy_(t_host)
        replay()
        torch.cuda.synchronize()
        t_np, w_np = O.encode_batch(j_host.numpy())
        ref_loss, ref_grad = O.masked_mse_loss_and_grad(p_host, torch.from_numpy(t_np), torch.from_numpy(w_np))
        want_xy, want_conf = O.gauss_taylor_decode(p_host, t_host)
        d = np.abs(hp.targets.cpu().numpy().view(np.int32).astype(np.int64) - t_np.view(np.int32).astype(np.int64))
        assert d.max() <= 1 and (d != 0).mean() < 1e-6
        assert np.array_equal(hp.weights.cpu().numpy(), w_np)
        assert abs(hp.loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
        assert torch.allclose(hp.grad.cpu(), ref_grad, rtol=1e-5, atol=1e-12)
        mag = float(t_host[:, 0, 0].abs().max())
        assert (hp.coords.cpu() - want_xy).abs().max().item() <= 1e-4 * mag + 1e-3
        assert torch.equal(hp.maxval.cpu(), want_conf)
