"""GPU: the one-launch validation step (``sp_val_step_f32``, ``HeatmapHotPath.val_step``) for both decoder families.

It must return the bits of the composition it replaces -- the fused loss kernel with its HeatMapAcc argmaxes,
``sp_decode_ws_f32`` in the same mode, ``sp_heatmap_acc_f32`` and ``sp_person_rows_f32`` -- with only the loss allowed
to differ in its float64 summation order; agree with the oracle; leave its workspace reusable (eager and replayed from a
CUDA graph); and run the validation loop of the ResNet solvers (``BasicKeyPointDecoder``) down to the same AP."""
import os

import numpy as np
import pytest
import torch

from oracle import heatmap_oracle as O
from simple_pose_b200 import _abi, synth

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
MODES = {"gauss_taylor": _abi.SP_DECODE_GAUSS_TAYLOR, "basic": _abi.SP_DECODE_BASIC}


def eq(x, y):
    """Bit-equal up to NaN payloads: same NaN positions, identical other values (including the sign of zero)."""
    nx, ny = torch.isnan(x), torch.isnan(y)
    return torch.equal(nx, ny) and torch.equal(x.masked_fill(nx, 0).view(torch.int32), y.masked_fill(ny, 0).view(torch.int32))


def inputs(b, k, h, w, seed, special=True):
    """Seeded joints, predictions and inverse affines, with the awkward maps the decoders and the loss treat specially."""
    joints = synth.joints(b, num_joints=k, height=h, width=w, seed=seed)
    pred = synth.heatmaps(b, joints=k, height=h, width=w, seed=seed + 1, noise=0.02)
    if special and b >= 2:
        p = lambda i: i % b
        pred[p(1), 2 % k, 3, 4] = float("nan")                   # NaN map: peak, score and acc axes propagate it
        pred[p(2), 3 % k] = -1.0                                 # all negative: no positive peak
        pred[p(3), 4 % k] = 0.0                                  # all zero
        joints[p(4), :, 2] = 0.0                                 # zero-weight joints
        joints[p(5), : max(1, k // 2), 2] = 0.75                 # odd mask values
        # peaks on the border cases: Basic shifts for 1 < x < W-1, GaussTaylor refines for 1 < x < W-2 only
        for j, (y, x) in enumerate(((h // 2, w - 2), (h // 2, w - 1), (h - 2, w // 2), (1, w // 2), (2, 2), (h - 3, w - 3))):
            q, jj = p(6 + j), (5 + j) % k
            pred[q, jj] = 0.01 * pred[q, jj]
            pred[q, jj, y, x] = 2.0
            pred[q, jj, y, max(x - 1, 0)] = 1.5
            pred[q, jj, max(y - 1, 0), x] = 1.2
    tinv = synth.inverse_affines(b, height=h, width=w, seed=seed)[0]
    return joints.to(DEV), pred.to(DEV), tinv.to(DEV)


def composed(hp, joints, pred, tinv, decoder):
    """The stand-alone kernels val_step replaces, on fresh buffers: fused loss + argmaxes (no gradient), the decoder,
    the HeatMapAcc epilogue and the kps_to_dict_ rows."""
    lib = _abi.lib()
    b, k, h, w = hp.batch, hp.k, hp.h, hp.w
    f = lambda *s: torch.empty(s, dtype=torch.float32, device=DEV)
    out = {"weights": f(b, k), "loss": f(), "acc": f(), "rows": f(b, 3 * k + 1), "coords": f(b, k, 2), "maxval": f(b, k, 1),
           "pred_xy": f(b, k, 2), "label_xy": f(b, k, 2)}
    ws = torch.zeros((int(lib.sp_mse_workspace_bytes()) + 7) // 8, dtype=torch.int64, device=DEV)
    dws = torch.zeros(2, dtype=torch.int64, device=DEV)
    stream = _abi.stream_ptr(DEV)
    _abi.check(lib.sp_encode_mse_fwd_bwd_f32(joints.data_ptr(), pred.data_ptr(), None, None, out["weights"].data_ptr(),
                                             out["loss"].data_ptr(), out["pred_xy"].data_ptr(), out["label_xy"].data_ptr(),
                                             ws.data_ptr(), ws.numel() * 8, b, k, h, w, hp.sigma, 1.0, stream))
    blur = hp.blur_w.data_ptr() if decoder == "gauss_taylor" else None
    _abi.check(lib.sp_decode_ws_f32(pred.data_ptr(), None, None, tinv.data_ptr(), blur, out["coords"].data_ptr(),
                                    out["maxval"].data_ptr(), None, b, k, h, w, 11 if decoder == "gauss_taylor" else 0,
                                    MODES[decoder], dws.data_ptr(), 16, stream))
    _abi.check(lib.sp_heatmap_acc_f32(out["pred_xy"].data_ptr(), out["label_xy"].data_ptr(), out["acc"].data_ptr(),
                                      b, k, h, w, 0.5, 10.0, stream))
    _abi.check(lib.sp_person_rows_f32(out["coords"].data_ptr(), out["maxval"].data_ptr(), out["rows"].data_ptr(), b, k, stream))
    torch.cuda.synchronize()
    return out


def assert_same(hp, want):
    for key in ("rows", "weights", "coords", "maxval", "pred_xy", "label_xy", "acc"):
        assert eq(getattr(hp, key), want[key]), key
    lw, lg = float(want["loss"]), float(hp.loss)
    assert (lw != lw and lg != lg) or abs(lg - lw) <= 1e-6 * abs(lw)


def workspace_is_zero(hp):
    """The reduction ticket, the work counter and every per-person arrival counter are back at zero."""
    arrivals = (int(_abi.lib().sp_mse_workspace_bytes()) + 15) // 16 * 16 // 8
    return int(hp.vws[:2].abs().sum()) == 0 and int(hp.vws[arrivals:arrivals + (hp.batch + 1) // 2].abs().sum()) == 0


@pytest.mark.parametrize("decoder", ["gauss_taylor", "basic"])
@pytest.mark.parametrize("b,k,hw", [(1, 17, (64, 48)), (2, 17, (96, 72)), (128, 17, (64, 48)), (128, 17, (96, 72)),
                                    (1024, 17, (64, 48)), (40, 14, (64, 48)), (300, 5, (96, 72))])
def test_val_step_equals_the_composed_kernels(decoder, b, k, hw):
    from simple_pose_b200.pipeline import HeatmapHotPath
    h, w = hw
    joints, pred, tinv = inputs(b, k, h, w, seed=11 * b + k)
    hp = HeatmapHotPath(b, k, h, w, device=DEV)
    assert hp.val_one_launch_supported(h, w, hp.ksize, decoder)
    want = composed(hp, joints, pred, tinv, decoder)
    loss, acc, rows = hp.val_step(joints, pred, tinv, decoder)
    torch.cuda.synchronize()
    assert loss is hp.loss and acc is hp.acc and rows is hp.rows and rows.shape == (b, 3 * k + 1) and rows.is_cuda
    assert_same(hp, want)
    assert workspace_is_zero(hp)


@pytest.mark.parametrize("decoder", ["gauss_taylor", "basic"])
@pytest.mark.parametrize("env", [{}, {"SP_STEP_STATIC_PCT": "0"}, {"SP_STEP_STATIC_PCT": "100"},
                                 {"SP_STEP_WARPS": "3", "SP_STEP_STATIC_PCT": "30"}, {"SP_STEP_WARPS": "5"}])
def test_val_step_grid_wide_layouts(decoder, env):
    """1100 persons: the few-warps layout with maps dealt grid-wide, under every split between static and claimed maps."""
    from simple_pose_b200.pipeline import HeatmapHotPath
    b, k, h, w = 1100, 17, 64, 48
    joints, pred, tinv = inputs(b, k, h, w, seed=5)
    hp = HeatmapHotPath(b, k, h, w, device=DEV)
    want = composed(hp, joints, pred, tinv, decoder)
    os.environ.update(env)
    _abi.reload_tuning()
    try:
        hp.val_step(joints, pred, tinv, decoder)
        torch.cuda.synchronize()
    finally:
        for key in env:
            del os.environ[key]
        _abi.reload_tuning()
    assert_same(hp, want)
    assert workspace_is_zero(hp)


@pytest.mark.parametrize("decoder", ["gauss_taylor", "basic"])
def test_val_step_repeated_calls_and_graph_replay(decoder):
    """The same workspace serves call after call, and a captured graph replays correctly after the inputs changed in
    place: the per-person counters and the work counter are returned to zero by every launch."""
    from simple_pose_b200.pipeline import HeatmapHotPath
    b, k, h, w = 128, 17, 64, 48
    hp = HeatmapHotPath(b, k, h, w, device=DEV)
    joints, pred, tinv = inputs(b, k, h, w, seed=1)
    want = composed(hp, joints, pred, tinv, decoder)
    for _ in range(3):
        hp.val_step(joints, pred, tinv, decoder)
        torch.cuda.synchronize()
        assert_same(hp, want)
        assert workspace_is_zero(hp)
    replay = hp.capture_val(joints, pred, tinv, decoder)
    for seed in (2, 3, 2):
        j2, p2, t2 = inputs(b, k, h, w, seed=seed)
        joints.copy_(j2)
        pred.copy_(p2)
        tinv.copy_(t2)
        replay()
        torch.cuda.synchronize()
        assert_same(hp, composed(hp, joints, pred, tinv, decoder))
        assert workspace_is_zero(hp)


@pytest.mark.parametrize("decoder", ["gauss_taylor", "basic"])
@pytest.mark.parametrize("b,hw", [(48, (64, 48)), (20, (96, 72))])
def test_val_step_against_the_oracle(decoder, b, hw):
    """Loss, HeatMapAcc, the decoder and kps_to_dict_ against the oracle, with the tolerances of the HRNet solver's
    validation loop test."""
    from simple_pose_b200.metrics.pose_metrics import rows_to_dicts
    from simple_pose_b200.pipeline import HeatmapHotPath
    h, w = hw
    joints, pred, tinv = inputs(b, 17, h, w, seed=21, special=False)
    hp = HeatmapHotPath(b, 17, h, w, device=DEV)
    loss, acc, rows = hp.val_step(joints, pred, tinv, decoder)
    got_dicts = []
    rows_to_dicts(rows, list(range(b)), got_dicts)
    p_host, t_inv = pred.cpu(), tinv.cpu()
    t_np, w_np = O.encode_batch(joints.cpu().numpy(), shape=(w, h))
    tgt, msk = torch.from_numpy(t_np), torch.from_numpy(w_np)
    ref_loss = O.masked_mse_loss(p_host, tgt, msk)
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    ref_acc = O.heat_map_acc(p_host * msk[..., None, None], tgt * msk[..., None, None])
    assert abs(acc.item() - float(ref_acc)) <= 1e-6
    want_xy, want_conf = (O.gauss_taylor_decode if decoder == "gauss_taylor" else O.basic_decode)(p_host, t_inv)
    mag = float(t_inv[:, 0, 0].abs().max())
    assert (hp.coords.cpu() - want_xy).abs().max().item() <= 1e-4 * mag + 1e-3
    assert torch.equal(hp.maxval.cpu(), want_conf)
    want_dicts = []
    O.kps_to_dict(hp.coords.cpu(), hp.maxval.cpu(), list(range(b)), want_dicts)
    assert len(got_dicts) == len(want_dicts) == b
    for g, wd in zip(got_dicts, want_dicts):
        assert g["image_id"] == wd["image_id"] and g["category_id"] == 1 and g["keypoints"] == wd["keypoints"]
        assert abs(g["score"] - wd["score"]) <= 2.4e-7 * abs(wd["score"])


class StandInBackbone(torch.nn.Module):
    """One 3x3 convolution + 4x average pooling: [B,3,256,192] -> [B,17,64,48] (the solvers' model slot)."""

    def __init__(self):
        super().__init__()
        self.conv = torch.nn.Conv2d(3, 17, 3, padding=1)
        self.pool = torch.nn.AvgPool2d(4)

    def forward(self, x):
        return self.pool(self.conv(x))


def test_val_loop_of_the_resnet_solvers():
    """The validation loop of dp_pose_resnet_solver / ddp_pose_resnet_solver (BasicKeyPointDecoder) as one val_step per
    batch, ending in COCO keypoint AP from the rows; the AP equals that of the composed kernels' rows, and loss and acc
    agree with the JointsMSELoss / HeatMapAcc drop-ins the solvers call."""
    from simple_pose_b200.commons.transforms import encode_heat_maps
    from simple_pose_b200.metrics import coco_eval as CE
    from simple_pose_b200.metrics.pose_metrics import BasicKeyPointDecoder, HeatMapAcc, person_rows
    from simple_pose_b200.pipeline import HeatmapHotPath
    from simple_pose_b200.processors.loss import JointsMSELoss
    torch.manual_seed(2)
    model = StandInBackbone().to(DEV).eval()
    b = 16
    hp = HeatmapHotPath(b, 17, 64, 48, device=DEV)
    creterion, acc_func, decoder = JointsMSELoss(), HeatMapAcc(), BasicKeyPointDecoder()
    val_rows, ref_rows = [], []
    with torch.no_grad():
        for it in range(2):
            input_img = torch.randn(b, 3, 256, 192, generator=torch.Generator().manual_seed(90 + it)).to(DEV)
            joints = synth.joints(b, seed=91 + it).to(DEV)
            tran_inv = synth.inverse_affines(b, seed=92 + it)[0].to(DEV)
            predicts = 0.02 * model(input_img) + synth.heatmaps(b, seed=93 + it, noise=0.0).to(DEV)
            loss, acc, rows = hp.val_step(joints, predicts, tran_inv, decoder="basic")
            val_rows.append(rows.clone())
            # the reference's lines on the same predictions
            targets, mask = encode_heat_maps(joints)
            ref_loss = creterion(predicts.clone(), targets, mask)
            ref_acc = acc_func(predicts.mul(mask[..., None, None]), targets.mul(mask[..., None, None]))
            assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
            assert abs(acc.item() - ref_acc.item()) <= 1e-6
            pred_kps, scores = decoder(predicts, tran_inv)
            ref_rows.append(person_rows(pred_kps, scores))
    got, want = torch.cat(val_rows), torch.cat(ref_rows)
    assert eq(got, want)
    # synthetic GT: two persons per image, each GT the decoded keypoints moved by a few pixels
    n = got.shape[0]

    class Persons(object):
        images, seg = n // 2, np.arange(0, n + 1, 2)
        boxes, leader = synth.detection_boxes(n, seed=94), torch.arange(n)

    ds, _ = synth.eval_set_ground_truth(Persons, got[:, :-1].reshape(n, 17, 3).cpu().numpy(), seed=95, jitter=1.5)
    gt = CE.CocoKeypointGT(ds, device=DEV)
    img_ids = np.repeat(np.arange(1, n // 2 + 1), 2)
    ap_val = CE.evaluate_person_rows(gt, got, img_ids).stats.cpu().numpy()
    ap_ref = CE.evaluate_person_rows(gt, want, img_ids).stats.cpu().numpy()
    assert np.array_equal(ap_val, ap_ref) and ap_val[0] > 0
