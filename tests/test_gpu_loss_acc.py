"""GPU: the masked-MSE loss with HeatMapAcc in the same pass (``sp_mse_acc_fwd_bwd``, ``JointsMSELoss(with_acc=True)``).

It must return the bits of what the solvers compose today on the same ``predicts`` / ``targets`` / ``mask`` --
``JointsMSELoss()`` for the loss and the gradient, ``HeatMapAcc()(predicts.mul(mask), targets.mul(mask))`` for acc and
the two heat_map_to_axis tables -- however a map is split over lanes, warps and blocks; leave its workspace reusable
(eager and replayed from a CUDA graph); agree with the oracle; and cost one launch per float32 forward."""
import os

import pytest
import torch

from oracle import heatmap_oracle as O
from simple_pose_b200 import _abi, synth

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def eq(x, y):
    """Bit-equal up to NaN payloads: same NaN positions, identical other values (including the sign of zero)."""
    if x is None or y is None:
        return x is None and y is None
    x, y = x.detach(), y.detach()
    if x.dtype != y.dtype or x.shape != y.shape:
        return False
    nx, ny = torch.isnan(x), torch.isnan(y)
    view = {torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}[x.dtype]
    return torch.equal(nx, ny) and torch.equal(x.masked_fill(nx, 0).view(view), y.masked_fill(ny, 0).view(view))


def inputs(b, k, h, w, seed, special=True):
    """Seeded predictions, the loader's targets and mask, and -- with ``special`` -- the maps the argmax order is decided
    on: equal maxima in the first and last quarter of a map (different chunks, and different blocks' ranges for the maps
    that straddle two), peaks on a map's last element, NaN before and after the finite maximum, +-inf, all-negative,
    all-zero and all -inf maps, NaN / inf in masked-out maps, odd and zero mask values, NaN and ties in a target."""
    joints = synth.joints(b, num_joints=k, height=h, width=w, seed=seed)
    pred = synth.heatmaps(b, joints=k, height=h, width=w, seed=seed + 1, noise=0.02)
    from simple_pose_b200.commons.transforms import encode_heat_maps
    target, mask = encode_heat_maps(joints.to(DEV), 2.0, (w, h))
    target, mask = target.cpu(), mask.cpu()
    if special:
        n, hw = b * k, h * w
        g = torch.Generator().manual_seed(seed)
        flat = pred.view(n, hw)
        sel = torch.arange(0, n, 3)
        flat[sel, torch.randint(0, max(1, hw // 4), (len(sel),), generator=g)] = 3.0
        flat[sel, torch.randint(3 * hw // 4, hw, (len(sel),), generator=g)] = 3.0
        last = torch.arange(1, n, 3)
        flat[last, hw - 1] = 4.0
        p = lambda i: i % b
        mask[p(1), 2 % k] = mask[p(1), 3 % k] = 1.0
        pred[p(1), 2 % k, 3 % h, 4 % w] = float("nan")
        pred[p(1), 3 % k, 0, 1] = 5.0
        pred[p(1), 3 % k, h - 1, w - 1] = float("nan")            # NaN after the finite maximum: NaN wins
        pred[p(2), 3 % k] = -1.0
        pred[p(3), 4 % k] = 0.0
        mask[p(4)] = 0.0
        pred[p(4), 1 % k, 2 % h, 2 % w] = float("nan")           # masked out: 0 * NaN is NaN, no peak either way
        pred[p(4), 2 % k, 0, 0] = float("inf")
        mask[p(5), : max(1, k // 2)] = 0.75
        mask[p(5), k - 1] = 2.0
        mask[p(6), 5 % k] = mask[p(6), 6 % k] = mask[p(7), 7 % k] = 1.0
        pred[p(6), 5 % k, h // 2, w // 2] = float("inf")
        pred[p(6), 5 % k, h - 1, 0] = float("inf")                # the first of two +inf wins
        pred[p(6), 6 % k, 0, 0] = float("-inf")
        pred[p(7), 7 % k] = float("-inf")
        mask[p(8), 8 % k] = mask[p(8), 9 % k] = 1.0
        target[p(8), 8 % k, 1, 1] = float("nan")
        target[p(8), 9 % k] = 0.0
        target[p(8), 9 % k, 1, 1] = target[p(8), 9 % k, h - 2, w - 2] = 1.0
    return pred.to(DEV), target.to(DEV), mask.to(DEV)


def composed(pred, target, mask, grad=True, skip_masked=False):
    """What the solvers run today: JointsMSELoss() (+ backward), HeatMapAcc()(pred.mul(mask), target.mul(mask)), and
    the two heat_map_to_axis tables HeatMapAcc decodes."""
    from simple_pose_b200.metrics.pose_metrics import BasicKeyPointDecoder, HeatMapAcc
    from simple_pose_b200.processors.loss import JointsMSELoss
    m = mask[..., None, None]
    p = pred.detach().clone().requires_grad_(grad)
    loss = JointsMSELoss(skip_masked=skip_masked)(p, target, mask)
    if grad:
        loss.backward()
    pm, tm = pred.detach().mul(m), target.mul(m)
    out = {"loss": loss.detach(), "grad": p.grad if grad else None, "acc": HeatMapAcc()(pm, tm),
           "pred_xy": BasicKeyPointDecoder.heat_map_to_axis(pm)[0], "label_xy": BasicKeyPointDecoder.heat_map_to_axis(tm)[0]}
    torch.cuda.synchronize()
    return out


def one_pass(pred, target, mask, grad=True, skip_masked=False):
    """JointsMSELoss(with_acc=True) (+ backward), and the same launch through mse_forward_backward for the axes."""
    from simple_pose_b200.processors.loss import JointsMSELoss, mse_forward_backward
    p = pred.detach().clone().requires_grad_(grad)
    loss, acc = JointsMSELoss(skip_masked=skip_masked, with_acc=True)(p, target, mask)
    if grad:
        loss.backward()
    b, k = mask.shape
    pxy, lxy = (torch.full((b, k, 2), -7.0, device=DEV) for _ in range(2))
    loss2, _, acc2 = mse_forward_backward(pred, target, mask, need_grad=False, skip_masked=skip_masked, want_acc=True,
                                          axes_out=(pxy, lxy))
    torch.cuda.synchronize()
    assert eq(loss2, loss) and eq(acc2, acc)
    assert acc.shape == () and acc.dtype == torch.float32 and acc.is_cuda and not acc.requires_grad
    return {"loss": loss.detach(), "grad": p.grad if grad else None, "acc": acc, "pred_xy": pxy, "label_xy": lxy}


def assert_same(got, want):
    for key in ("loss", "grad", "acc", "pred_xy", "label_xy"):
        assert eq(got[key], want[key]), key


@pytest.mark.parametrize("grad", [True, False])
@pytest.mark.parametrize("b,k,hw", [(1, 17, (64, 48)), (2, 17, (96, 72)), (128, 17, (64, 48)), (1024, 17, (64, 48)),
                                    (40, 14, (64, 48)), (300, 5, (96, 72)), (3, 17, (9, 7)), (64, 17, (10, 6))])
def test_loss_acc_equals_the_composition(grad, b, k, hw):
    h, w = hw
    pred, target, mask = inputs(b, k, h, w, seed=7 * b + k)
    want = composed(pred, target, mask, grad)
    assert_same(one_pass(pred, target, mask, grad), want)


@pytest.mark.parametrize("env", [{}, {"SP_LOSS_WARPS": "1"}, {"SP_LOSS_WARPS": "7", "SP_LOSS_RING": "1"},
                                 {"SP_LOSS_CHUNK_QUADS": "8"}, {"SP_LOSS_CHUNK_QUADS": "48", "SP_LOSS_WARPS": "16"},
                                 {"SP_LOSS_CHUNK_QUADS": "2048"}, {"SP_LOSS_FORCE_LDG": "1"}])
@pytest.mark.parametrize("hw", [(64, 48), (96, 72)])
def test_loss_acc_under_the_tuning_overrides(env, hw):
    """Every way the loss kernels split a map -- chunk sizes from 32 elements to whole maps, 1 to 16 warps per block, the
    plain-load kernel -- gives the same bits."""
    h, w = hw
    pred, target, mask = inputs(300, 17, h, w, seed=3)
    os.environ.update(env)
    _abi.reload_tuning()
    try:
        want = composed(pred, target, mask, True)          # the loss kernel under the same split: the same summation order
        got = one_pass(pred, target, mask, True)
    finally:
        for key in env:
            del os.environ[key]
        _abi.reload_tuning()
    assert_same(got, want)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_loss_acc_skip_masked(dtype):
    """SP_MSE_SKIP_MASKED (finite inputs): masked-out maps are not read and give (0, 0), as their products would."""
    pred, target, mask = inputs(200, 17, 64, 48, seed=4, special=False)
    pred = pred.to(dtype)
    assert_same(one_pass(pred, target, mask, True, skip_masked=True), composed(pred, target, mask, True, skip_masked=True))


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("b,hw", [(128, (64, 48)), (33, (96, 72)), (6, (9, 7))])
def test_loss_acc_autocast_dtypes(dtype, b, hw):
    """pred in the autocast dtype: the products are float32 float(p) * m, as autocast's predicts.mul(mask); loss and
    gradient are the existing mixed-precision path's bits."""
    h, w = hw
    pred, target, mask = inputs(b, 17, h, w, seed=9 * b)
    pred = pred.to(dtype)
    for grad in (True, False):
        with torch.autocast("cuda", dtype=dtype):
            want = composed(pred, target, mask, grad)
            got = one_pass(pred, target, mask, grad)
        assert got["grad"] is None or got["grad"].dtype == dtype
        assert_same(got, want)


class StandInBackbone(torch.nn.Module):
    """One 3x3 convolution + 4x average pooling: [B,3,256,192] -> [B,17,64,48] (the solvers' model slot)."""

    def __init__(self):
        super().__init__()
        self.conv = torch.nn.Conv2d(3, 17, 3, padding=1)
        self.pool = torch.nn.AvgPool2d(4)

    def forward(self, x):
        return self.pool(self.conv(x))


@pytest.mark.parametrize("amp", [False, True])
def test_train_and_val_loops_of_the_hrnet_solver(amp):
    """dp_pose_hrnet_solver.py:99-127 with the two-line change (loss, acc = JointsMSELoss(with_acc=True)(...); no .mul,
    no acc_func), plain and AMP + GradScaler: loss, acc and d loss / d predicts equal the composition's bits on the same
    predictions; then the val() loop (:150-157) under no_grad."""
    from simple_pose_b200.commons.transforms import encode_heat_maps
    from simple_pose_b200.metrics.pose_metrics import HeatMapAcc
    from simple_pose_b200.processors.loss import JointsMSELoss
    torch.manual_seed(0)
    model = StandInBackbone().to(DEV)
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-3)
    scaler = torch.amp.GradScaler("cuda", init_scale=1024.0) if amp else None
    creterion, old_creterion, acc_func = JointsMSELoss(with_acc=True), JointsMSELoss(), HeatMapAcc()
    losses = []
    for it in range(3):
        input_img = torch.randn(8, 3, 256, 192, generator=torch.Generator().manual_seed(it)).to(DEV)
        targets, mask = encode_heat_maps(synth.joints(8, seed=100 + it).to(DEV))
        captured = {}
        optimizer.zero_grad()
        with torch.autocast("cuda", enabled=amp):
            predicts = model(input_img)
            old_loss = old_creterion(predicts, targets, mask)
            loss, acc = creterion(predicts, targets, mask)
        old_acc = acc_func(predicts.mul(mask[..., None, None]).detach(), targets.mul(mask[..., None, None]).detach())
        scale = (lambda l: scaler.scale(l)) if amp else (lambda l: l)
        (old_grad,) = torch.autograd.grad(scale(old_loss), predicts, retain_graph=True)
        predicts.register_hook(lambda g: captured.__setitem__("grad", g))
        scale(loss).backward()
        if amp:
            scaler.step(optimizer)
            scaler.update()
        else:
            optimizer.step()
        assert eq(loss, old_loss) and eq(acc, old_acc) and eq(captured["grad"], old_grad)
        assert captured["grad"].dtype == predicts.dtype == (torch.float16 if amp else torch.float32)
        losses.append(loss.item())
    assert len(set(losses)) == 3
    model.eval()
    with torch.no_grad():
        for it in range(2):
            input_img = torch.randn(16, 3, 256, 192, generator=torch.Generator().manual_seed(50 + it)).to(DEV)
            targets, mask = encode_heat_maps(synth.joints(16, seed=60 + it).to(DEV))
            with torch.autocast("cuda", enabled=amp):
                predicts = model(input_img)
                loss, acc = creterion(predicts, targets, mask)
                old_loss = old_creterion(predicts, targets, mask)
            old_acc = acc_func(predicts.mul(mask[..., None, None]), targets.mul(mask[..., None, None]))
            assert eq(loss, old_loss) and eq(acc, old_acc)


def test_repeated_calls_and_graph_replay():
    """One workspace serves call after call, and a captured graph replays correctly after the inputs changed in place:
    every launch returns the ticket and the argmax keys to zero."""
    lib = _abi.lib()
    b, k, h, w = 128, 17, 64, 48
    pred, target, mask = inputs(b, k, h, w, seed=1)
    f = lambda *s: torch.empty(s, dtype=torch.float32, device=DEV)
    out = {"loss": f(), "acc": f(), "grad": f(b, k, h, w), "pred_xy": f(b, k, 2), "label_xy": f(b, k, 2)}
    nbytes = int(lib.sp_mse_acc_workspace_bytes(b, k))
    ws = torch.zeros((nbytes + 7) // 8, dtype=torch.int64, device=DEV)
    keys = (int(lib.sp_mse_workspace_bytes()) + 15) // 16 * 16 // 8

    def run():
        _abi.check(lib.sp_mse_acc_fwd_bwd(pred.data_ptr(), _abi.SP_DTYPE_F32, target.data_ptr(), mask.data_ptr(),
                                          out["grad"].data_ptr(), out["loss"].data_ptr(), out["acc"].data_ptr(),
                                          out["pred_xy"].data_ptr(), out["label_xy"].data_ptr(), ws.data_ptr(), nbytes,
                                          b, k, h, w, 1.0, None, 0.5, 10.0, 0, _abi.stream_ptr(DEV)))

    def check():
        torch.cuda.synchronize()
        assert_same(out, composed(pred, target, mask, True))
        assert int(ws[:2].abs().sum()) == 0 and int(ws[keys:keys + 2 * b * k].abs().sum()) == 0

    for _ in range(3):
        run()
        check()
    stream = torch.cuda.Stream(DEV)
    stream.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(stream):
        run()
    torch.cuda.current_stream(DEV).wait_stream(stream)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        run()
    for seed in (2, 3, 2):
        p2, t2, m2 = inputs(b, k, h, w, seed=seed)
        pred.copy_(p2)
        target.copy_(t2)
        mask.copy_(m2)
        graph.replay()
        check()


@pytest.mark.parametrize("b,hw", [(48, (64, 48)), (20, (96, 72)), (9, (10, 6))])
def test_loss_acc_against_the_oracle(b, hw):
    h, w = hw
    pred, target, mask = inputs(b, 17, h, w, seed=21, special=False)
    got = one_pass(pred, target, mask, True)
    p, t, m = pred.cpu(), target.cpu(), mask.cpu()[..., None, None]
    ref_acc = O.heat_map_acc(p * m, t * m)
    assert got["acc"].item() == float(ref_acc)             # float32 values: equal as doubles iff equal as floats
    ref_loss = O.masked_mse_loss(p, t, mask.cpu())
    assert abs(got["loss"].item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())


def test_one_kernel_per_float32_forward_and_per_no_grad_call():
    from torch.profiler import ProfilerActivity, profile
    from simple_pose_b200.processors.loss import JointsMSELoss
    pred, target, mask = inputs(128, 17, 64, 48, seed=5, special=False)
    crit = JointsMSELoss(with_acc=True)
    p = pred.clone().requires_grad_()
    crit(p, target, mask)                                    # workspace allocation and module load outside the trace
    with torch.no_grad():
        crit(pred, target, mask)
    torch.cuda.synchronize()

    def kernels(fn):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]

    p = pred.clone().requires_grad_()
    names = kernels(lambda: crit(p, target, mask))         # loss + gradient + acc
    assert len(names) == 1 and "mse_ring_kernel" in names[0], names

    def val():
        with torch.no_grad():
            crit(pred, target, mask)
    names = kernels(val)                                     # loss + acc
    assert len(names) == 1 and "mse_ring_kernel" in names[0], names


def test_val_step_composed_path_for_odd_widths():
    """HeatmapHotPath.val_step at a width the one launch does not take (W % 4 != 0) runs the encoder and this entry point:
    its acc and axes equal those of the masked copies decoded by heat_map_to_axis."""
    from simple_pose_b200.commons.transforms import encode_heat_maps
    from simple_pose_b200.pipeline import HeatmapHotPath
    b, k, h, w = 24, 17, 63, 50
    joints = synth.joints(b, height=h, width=w, seed=8).to(DEV)
    pred = synth.heatmaps(b, height=h, width=w, seed=9, noise=0.02).to(DEV)
    tinv = synth.inverse_affines(b, height=h, width=w, seed=8)[0].to(DEV)
    hp = HeatmapHotPath(b, k, h, w, device=DEV)
    assert not hp.val_one_launch_supported(h, w, hp.ksize, "basic")
    loss, acc, rows = hp.val_step(joints, pred, tinv, "basic")
    torch.cuda.synchronize()
    targets, mask = encode_heat_maps(joints, 2.0, (w, h))
    want = composed(pred, targets, mask, grad=False)
    for key in ("loss", "acc", "pred_xy", "label_xy"):
        assert eq(getattr(hp, key), want[key]), key
