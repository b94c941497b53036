"""One validation batch (the body of the solvers' val(): loss, HeatMapAcc, decoder, kps_to_dict_ rows) as one launch of
``sp_val_step_f32`` against the stand-alone kernels it replaces: 3 launches for the GaussTaylor decoder (the one-launch
step with HeatMapAcc argmaxes, the HeatMapAcc epilogue, the person rows) and 4 for the Basic decoder (the fused loss
kernel with its argmaxes, the Basic decode, the epilogue, the person rows). Each is timed eager (launched from Python)
and replayed from a CUDA graph, with CUDA events around `--reps` batches, warmed up, median of `--rounds` rounds,
the two paths alternating. Prints one JSON line per size with the card name and power limit read in the same run.

Batch 128 at 64x48 is 26.7 MB of heatmaps, which fits in the 126 MB L2, so the batches rotate over `--sets` distinct
input buffer sets (>= 8: 214 MB) and every batch reads its heatmaps from HBM.

    python profiles/bench_val_step.py [--check] [--reps 200] [--rounds 5] [--sets 8]

--check compares the outputs of the two paths (rows, weights, coords, maxval, acc bit for bit; the loss within 1e-6
relative, its float64 summation order differs) and exits non-zero if they differ.
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

from simple_pose_b200 import _abi, synth  # noqa: E402
from simple_pose_b200.pipeline import HeatmapHotPath  # noqa: E402

SIZES = [(128, 64, 48), (1024, 64, 48), (512, 96, 72)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as exc:      # the card name from torch at least
        return torch.cuda.get_device_name(0), "unknown (%s)" % type(exc).__name__


def composed(hp, joints, pred, tinv, decoder):
    """The launches val_step replaces (outputs in hp's buffers)."""
    lib, stream = hp._lib, _abi.stream_ptr(hp.device)
    if decoder == "gauss_taylor":            # 3 launches: one-launch step (no grad, no targets) with the argmaxes
        hp.step_one_launch(joints, pred, tinv, want_targets=False, want_grad=False, with_acc=True)
    else:                                    # 4 launches: fused loss with the argmaxes, then the Basic decode
        _abi.check(lib.sp_encode_mse_fwd_bwd_f32(joints.data_ptr(), pred.data_ptr(), None, None, hp.weights.data_ptr(),
                                                 hp.loss.data_ptr(), hp.pred_xy.data_ptr(), hp.label_xy.data_ptr(),
                                                 hp.ws.data_ptr(), hp.ws.numel() * 8, hp.batch, hp.k, hp.h, hp.w,
                                                 hp.sigma, 1.0, stream))
        _abi.check(lib.sp_decode_ws_f32(pred.data_ptr(), None, None, tinv.data_ptr(), None, hp.coords.data_ptr(),
                                        hp.maxval.data_ptr(), None, hp.batch, hp.k, hp.h, hp.w, 0, _abi.SP_DECODE_BASIC,
                                        hp.dws.data_ptr(), 16, stream))
    _abi.check(lib.sp_heatmap_acc_f32(hp.pred_xy.data_ptr(), hp.label_xy.data_ptr(), hp.acc.data_ptr(),
                                      hp.batch, hp.k, hp.h, hp.w, 0.5, 10.0, stream))
    _abi.check(lib.sp_person_rows_f32(hp.coords.data_ptr(), hp.maxval.data_ptr(), hp.rows.data_ptr(), hp.batch, hp.k, stream))


def time_us(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(reps):
        fn(i)
    end.record()
    end.synchronize()
    return start.elapsed_time(end) * 1000.0 / reps


def snapshot(hp):
    return {k: getattr(hp, k).clone() for k in ("rows", "weights", "coords", "maxval", "acc", "loss")}


def same(a, b):
    def eq(x, y):
        nx, ny = torch.isnan(x), torch.isnan(y)
        return torch.equal(nx, ny) and torch.equal(x.masked_fill(nx, 0).view(torch.int32), y.masked_fill(ny, 0).view(torch.int32))
    bits = all(eq(a[k], b[k]) for k in ("rows", "weights", "coords", "maxval", "acc"))
    la, lb = float(a["loss"]), float(b["loss"])
    return bits and abs(la - lb) <= 1e-6 * abs(lb)


def run_size(b, h, w, args):
    dev = torch.device("cuda:0")
    sets = max(1, args.sets if b * 17 * h * w * 4 < (64 << 20) else 2)
    data = []
    for s in range(sets):
        joints = synth.joints(b, height=h, width=w, seed=s).to(dev)
        pred = synth.heatmaps(b, height=h, width=w, seed=100 + s, noise=0.02, device=dev)
        tinv = synth.inverse_affines(b, height=h, width=w, seed=s)[0].to(dev)
        data.append((joints, pred, tinv))
    out = {"batch": b, "H": h, "W": w, "input_sets": sets, "reps": args.reps, "rounds": args.rounds}
    ok = True
    for decoder in ("gauss_taylor", "basic"):
        one, ref = HeatmapHotPath(b, 17, h, w, device=dev), HeatmapHotPath(b, 17, h, w, device=dev)
        one.val_step(*data[0], decoder)                       # allocates rows / acc / workspace
        ref.val_step(*data[0], decoder)
        paths = {
            "val_step": lambda i: one.val_step(*data[i % sets], decoder),
            "composed": lambda i: composed(ref, *data[i % sets], decoder),
        }
        if args.check:
            for i in range(sets):
                paths["val_step"](i)
                paths["composed"](i)
                torch.cuda.synchronize()
                if not same(snapshot(one), snapshot(ref)):
                    ok = False
                    out["%s_mismatch_set" % decoder] = i
        # graphs: one captured batch per input set, replayed in rotation
        graphs = {}
        for name, hp in (("val_step", one), ("composed", ref)):
            reps = []
            for i in range(sets):
                if name == "val_step":
                    reps.append(hp.capture_val(*data[i], decoder))
                else:
                    reps.append(hp._capture(lambda i=i: composed(ref, *data[i], decoder)))
                hp._graphs = getattr(hp, "_graphs", []) + [hp._graph]
            graphs[name] = (lambda r: (lambda i: r[i % sets]()))(reps)
        for mode, table in (("eager", paths), ("graph", graphs)):
            for fn in table.values():
                time_us(fn, args.warmup)
            samples = {k: [] for k in table}
            for _ in range(args.rounds):
                for name, fn in table.items():            # alternate the two paths
                    samples[name].append(time_us(fn, args.reps))
            for name, v in samples.items():
                out["%s_%s_%s_us" % (decoder, name, mode)] = round(sorted(v)[len(v) // 2], 2)
        out["%s_launches_composed" % decoder] = 3 if decoder == "gauss_taylor" else 4
    if args.check:
        out["check"] = "identical" if ok else "MISMATCH"
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
        raise SystemExit("bench_val_step.py needs a CUDA device")
    name, power = card()
    all_ok = True
    for b, h, w in SIZES:
        res, ok = run_size(b, h, w, args)
        all_ok &= ok
        res.update({"device": name, "power_limit": power})
        print(json.dumps(res), flush=True)
    if args.check and not all_ok:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
