"""The loss and HeatMapAcc of one batch, as every solver computes them from the loader's targets and mask
(processors/dp_pose_hrnet_solver.py:106-107 + 123-124, :156-157), against the one-pass form:

  composed   loss = JointsMSELoss()(predicts, targets, mask)                      1 launch (float32: + gradient)
             acc = HeatMapAcc()(predicts.mul(mask), targets.mul(mask))           2 mul + 2 argmax + 1 epilogue launches
  one_pass   loss, acc = JointsMSELoss(with_acc=True)(predicts, targets, mask)   1 launch (sp_mse_acc_fwd_bwd)
  loss_only  the loss launch of `composed` alone: what the argmax costs the loss kernel at the same shape

float32 predicts run the training call (loss + gradient in the forward launch); float16 / bfloat16 predicts the forward
launch of the autocast branch (its backward launch does not change). Each path is timed eager (called from Python) and
replayed from a CUDA graph, with CUDA events around `--reps` batches, warmed up, median of `--rounds` rounds, the paths
alternating. One JSON line per (size, dtype) with the card name and power limit read in the same run.

Batch 128 at 64x48 is 26.7 MB per map tensor: pred, targets and the gradient fit in the 126 MB L2, so the batches rotate
over `--sets` distinct input sets (>= 8) and every batch reads its inputs from HBM. The larger sizes rotate over two.

    python profiles/bench_loss_acc.py [--check] [--reps 200] [--rounds 5] [--sets 8]

--check compares the two forms (loss, gradient and acc bit for bit) on every input set and exits non-zero if they differ.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

from simple_pose_b200 import synth  # noqa: E402
from simple_pose_b200.commons.transforms import encode_heat_maps  # noqa: E402
from simple_pose_b200.metrics.pose_metrics import HeatMapAcc  # noqa: E402
from simple_pose_b200.processors.loss import mse_forward_backward  # noqa: E402

SIZES = [(128, 64, 48), (1024, 64, 48), (512, 96, 72)]
DTYPES = {"float32": torch.float32, "float16": torch.float16, "bfloat16": torch.bfloat16}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as exc:      # the card name from torch at least
        return torch.cuda.get_device_name(0), "unknown (%s)" % type(exc).__name__


def time_us(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(reps):
        fn(i)
    end.record()
    end.synchronize()
    return start.elapsed_time(end) * 1000.0 / reps


def eq(x, y):
    if x is None or y is None:
        return x is None and y is None
    nx, ny = torch.isnan(x), torch.isnan(y)
    view = torch.int32 if x.dtype == torch.float32 else torch.int16
    return torch.equal(nx, ny) and torch.equal(x.masked_fill(nx, 0).view(view), y.masked_fill(ny, 0).view(view))


def run_size(b, h, w, dtype, args):
    dev = torch.device("cuda:0")
    grad = dtype == torch.float32
    sets = max(1, args.sets if b * 17 * h * w * 4 < (64 << 20) else 2)
    data = []
    for s in range(sets):
        targets, mask = encode_heat_maps(synth.joints(b, height=h, width=w, seed=s).to(dev), 2.0, (w, h))
        pred = synth.heatmaps(b, height=h, width=w, seed=100 + s, noise=0.02, device=dev).to(dtype)
        data.append((pred, targets, mask))
    acc_func = HeatMapAcc()
    res = {}

    def composed(i):
        p, t, m = data[i % sets]
        loss, g = mse_forward_backward(p, t, m, need_grad=grad)
        mm = m[..., None, None]
        res["composed"] = (loss, g, acc_func(p.mul(mm), t.mul(mm)))

    def one_pass(i):
        p, t, m = data[i % sets]
        res["one_pass"] = mse_forward_backward(p, t, m, need_grad=grad, want_acc=True)

    def loss_only(i):
        p, t, m = data[i % sets]
        res["loss_only"] = mse_forward_backward(p, t, m, need_grad=grad)

    paths = {"composed": composed, "one_pass": one_pass, "loss_only": loss_only}
    out = {"batch": b, "H": h, "W": w, "dtype": str(dtype).replace("torch.", ""), "grad": grad, "input_sets": sets,
           "reps": args.reps, "rounds": args.rounds, "launches_composed": 6, "launches_one_pass": 1}
    ok = True
    if args.check:
        for i in range(sets):
            composed(i)
            one_pass(i)
            torch.cuda.synchronize()
            if not all(eq(x, y) for x, y in zip(res["composed"], res["one_pass"])):
                ok = False
                out["mismatch_set"] = i
        out["check"] = "identical" if ok else "MISMATCH"
    # graphs: one captured batch per input set and path, replayed in rotation; warmed up on the capture stream so that
    # the per-stream workspaces exist before the capture
    stream = torch.cuda.Stream(dev)
    stream.wait_stream(torch.cuda.current_stream(dev))
    graphs, keep = {}, []
    with torch.cuda.stream(stream):
        for fn in paths.values():
            for i in range(sets):
                fn(i)
    torch.cuda.current_stream(dev).wait_stream(stream)
    torch.cuda.synchronize()
    for name, fn in paths.items():
        reps = []
        for i in range(sets):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                fn(i)
            keep.append(g)
            reps.append(g.replay)
        graphs[name] = (lambda r: (lambda i: r[i % sets]()))(reps)
    for mode, table in (("eager", paths), ("graph", graphs)):
        for fn in table.values():
            time_us(fn, args.warmup)
        samples = {k: [] for k in table}
        for _ in range(args.rounds):
            for name, fn in table.items():            # alternate the paths
                samples[name].append(time_us(fn, args.reps))
        for name, v in samples.items():
            out["%s_%s_us" % (name, mode)] = round(sorted(v)[len(v) // 2], 2)
    return out, ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--sets", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_loss_acc.py needs a CUDA device")
    name, power = card()
    all_ok = True
    for b, h, w in SIZES:
        for dtype in DTYPES.values():
            res, ok = run_size(b, h, w, dtype, args)
            all_ok &= ok
            res.update({"device": name, "power_limit": power})
            print(json.dumps(res), flush=True)
    if args.check and not all_ok:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
