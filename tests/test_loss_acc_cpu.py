"""CPU: the loss + HeatMapAcc entry point (``sp_mse_acc_fwd_bwd``) rejects bad arguments before any CUDA call, its
workspace query, and ``JointsMSELoss(with_acc=True)``'s constructor, return contract and refusal of CPU tensors."""
import pytest
import torch

F32, F16, BF16 = 0, 1, 2


@pytest.fixture(scope="module")
def lib():
    from simple_pose_b200 import build, _abi
    build.build()
    return _abi.lib()


NAMES = ["pred", "dtype", "target", "mask", "grad", "loss", "acc", "pred_xy", "label_xy", "ws", "ws_bytes", "B", "K", "H",
         "W", "grad_scale", "grad_scale_dev", "thresh", "norm_frac", "flags", "stream"]


def acc_args(lib, B=1, K=17, H=64, W=48):
    return [16, F32, 16, 16, 16, 16, 16, None, None, 16, lib.sp_mse_acc_workspace_bytes(B, K), B, K, H, W, 1.0, None,
            0.5, 10.0, 0, None]


def with_(args, **kw):
    out = list(args)
    for k, v in kw.items():
        out[NAMES.index(k)] = v
    return out


def test_mse_acc_argument_errors(lib):
    ok = acc_args(lib)
    call = lambda a: lib.sp_mse_acc_fwd_bwd(*a)
    for dtype in (3, -1, 7):
        assert call(with_(ok, dtype=dtype)) == -1
    for name in ("pred", "target", "mask", "loss", "acc", "ws"):
        assert call(with_(ok, **{name: None})) == -1, name         # loss is required: backward-only stays sp_mse_fwd_bwd
    assert call(with_(ok, pred_xy=16)) == -1                        # pred_xy without label_xy
    assert call(with_(ok, label_xy=16)) == -1
    for name in ("B", "K", "H", "W"):
        assert call(with_(ok, **{name: 0})) == -1, name
        assert call(with_(ok, **{name: -3})) == -1, name
    assert call(with_(ok, norm_frac=0.0)) == -1 and call(with_(ok, norm_frac=-10.0)) == -1
    assert call(with_(ok, norm_frac=float("nan"))) == -1
    assert call(with_(acc_args(lib, K=4097), K=4097)) == -4         # the epilogue's per-joint counters live in shared memory
    assert call(with_(ok, H=65536, W=65536)) == -4                  # flat map index past int32
    assert call(with_(ok, B=1 << 16, K=1 << 16)) == -4              # B * K past int32
    assert call(with_(ok, ws_bytes=ok[10] - 1)) == -3               # workspace too small for B x K
    assert call(with_(acc_args(lib), B=2)) == -3
    assert call(with_(ok, ws=24)) == -2                             # misaligned workspace
    assert call(with_(ok, pred_xy=24, label_xy=16)) == -2           # misaligned axes
    assert call(with_(ok, pred_xy=16, label_xy=40)) == -2
    for dtype in (F16, BF16):                                       # the autocast dtypes go through the same checks
        assert call(with_(ok, dtype=dtype, loss=None)) == -1
        assert call(with_(ok, dtype=dtype, ws_bytes=8)) == -3


def test_mse_acc_workspace_bytes(lib):
    base = (lib.sp_mse_workspace_bytes() + 15) // 16 * 16
    for b, k in ((1, 17), (128, 17), (1024, 17), (3, 5), (7, 1)):
        got = lib.sp_mse_acc_workspace_bytes(b, k)
        assert got == base + 32 * b * k                              # keys (2 x 8 bytes) + room for the axes, per map
        assert got % 16 == 0
    for b, k in ((0, 17), (1, 0), (-1, 17), (1 << 16, 1 << 16)):
        assert lib.sp_mse_acc_workspace_bytes(b, k) == 0


def test_joints_mse_loss_with_acc_constructor():
    from simple_pose_b200.processors.loss import JointsMSELoss
    crit = JointsMSELoss()
    assert (crit.skip_masked, crit.defer_grad, crit.with_acc) == (False, False, False)
    assert (crit.distance_thresh, crit.norm_frac) == (0.5, 10.)
    crit = JointsMSELoss(True, True, with_acc=True, distance_thresh=0.25, norm_frac=5.)   # the old positional order holds
    assert (crit.skip_masked, crit.defer_grad, crit.with_acc) == (True, True, True)
    assert (crit.distance_thresh, crit.norm_frac, crit.acc) == (0.25, 5., None)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_joints_mse_loss_with_acc_refuses_cpu_tensors():
    from simple_pose_b200.processors.loss import JointsMSELoss, mse_forward_backward
    p, t, m = torch.zeros(2, 17, 8, 8), torch.zeros(2, 17, 8, 8), torch.ones(2, 17)
    for crit in (JointsMSELoss(with_acc=True), JointsMSELoss(with_acc=True, defer_grad=True)):
        with pytest.raises(RuntimeError, match="no CPU path"):
            crit(p, t, m)
        with pytest.raises(RuntimeError, match="no CPU path"):
            crit(p.half().requires_grad_(), t, m)
    with pytest.raises(RuntimeError, match="no CPU path"):
        mse_forward_backward(p, t, m, want_acc=True)


def test_mse_forward_backward_acc_contract_errors(monkeypatch):
    """Shape and call-kind errors are raised before the device is touched (the device check is stubbed out)."""
    from simple_pose_b200 import _abi
    from simple_pose_b200.processors import loss as L
    monkeypatch.setattr(_abi, "require_cuda", lambda *t: torch.device("cpu"))
    p, t, m = torch.zeros(2, 17, 8, 8), torch.zeros(2, 17, 8, 8), torch.ones(2, 17)
    with pytest.raises(ValueError, match="forward call"):
        L.mse_forward_backward(p, t, m, need_loss=False, want_acc=True)        # backward-only calls carry no acc
    with pytest.raises(ValueError, match="forward call"):
        L.mse_forward_backward(p.reshape(2, 17, 64), t.reshape(2, 17, 64), m, want_acc=True)   # acc needs (H, W)
    with pytest.raises(ValueError, match="shape mismatch"):
        L.mse_forward_backward(p, t[:, :5], m, want_acc=True)
    with pytest.raises(ValueError, match="shape mismatch"):
        L.JointsMSELoss(with_acc=True)(p, t, m[:1])
