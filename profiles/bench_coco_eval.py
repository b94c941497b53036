"""COCO keypoint evaluation on the device (metrics/coco_eval.py) on a COCO-val-sized synthetic set: one JSON line
with the sizes, the evaluator's device time (CUDA events around each call, warmed up, median of repeated calls),
the COCOeval oracle's host time on the same inputs, whether the stats equal the oracle's bit for bit, and the card
name and power limit read in the same run.

    python profiles/bench_coco_eval.py [--images 5000] [--seed 1] [--reps 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import coco_eval_oracle as C  # noqa: E402
from simple_pose_b200 import synth  # noqa: E402
from simple_pose_b200.metrics import coco_eval as CE  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception as exc:      # the card name from torch at least
        return torch.cuda.get_device_name(0), "unknown (%s)" % type(exc).__name__


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_coco_eval.py needs a CUDA device")
    dev = torch.device("cuda:0")
    ds, res = synth.coco_keypoint_set(args.images, seed=args.seed, fp=(4, 16))
    gt = CE.CocoKeypointGT(ds, device=dev)
    kps, sc, ids = synth.coco_results_arrays(res)
    kps, sc, pos = kps.to(dev), sc.to(dev), gt.positions(ids)
    first = CE.evaluate(gt, kps, sc, ids.numpy())
    for _ in range(args.warmup):
        CE.evaluate(gt, kps, sc, ids.numpy())
    torch.cuda.synchronize()
    # time the device work of one call: the C entry point on device-resident inputs (image ids already mapped)
    lib = CE._abi.lib()
    n = kps.shape[0]
    need = lib.sp_coco_eval_workspace_bytes(n, gt.num_images, gt.num_gts)
    ws = torch.zeros(need // 8 + 1, dtype=torch.int64, device=dev)
    out = torch.empty(3030 + 30 + 10, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream(dev)
    call = [kps.data_ptr(), 51, sc.data_ptr(), pos.data_ptr(), None, n, gt.kps.data_ptr(), gt.area.data_ptr(),
            gt.bbox.data_ptr(), gt.flags.data_ptr(), gt.seg.data_ptr(), gt.num_images, gt.num_gts, gt.iou_thrs.data_ptr(),
            gt.rec_thrs.data_ptr(), gt.area_rng.data_ptr(), 17, 10, 101, 3, 20, out.data_ptr(), out.data_ptr() + 8 * 3030,
            out.data_ptr() + 8 * 3060, None, None, None, ws.data_ptr(), need, stream.cuda_stream]
    for _ in range(args.warmup):
        CE._abi.check(lib.sp_coco_eval_kps_f32(*call))
    times = []
    for _ in range(args.reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        CE._abi.check(lib.sp_coco_eval_kps_f32(*call))
        b.record(stream)
        b.synchronize()
        times.append(a.elapsed_time(b) * 1000.0)
    device_stats = out[3060:].cpu().numpy()
    t0 = time.perf_counter()
    want = C.coco_eval_kps(ds, res)
    host_s = time.perf_counter() - t0
    name, power = card()
    line = {
        "bench": "coco_eval_kps",
        "images": gt.num_images, "gt_persons": gt.num_gts,
        "gt_without_keypoints": int(sum(1 for a in ds["annotations"] if a["category_id"] == 1 and a["num_keypoints"] == 0)),
        "detections": n, "evaluated_detections": int(sum(min(20, c) for c in np.bincount(pos.cpu().numpy() + 1)[1:])),
        "device_us_median": float(np.median(times)), "device_us_p10": float(np.percentile(times, 10)),
        "device_us_p90": float(np.percentile(times, 90)), "reps": args.reps,
        "oracle_host_s": host_s,
        "stats": [float(v) for v in device_stats],
        "stats_equal_oracle": bool(np.array_equal(device_stats, want["stats"])),
        "precision_equal_oracle": bool(np.array_equal(first.precision.cpu().numpy(), want["precision"])),
        "recall_equal_oracle": bool(np.array_equal(first.recall.cpu().numpy(), want["recall"])),
        "gpu": name, "power_limit": power, "torch": torch.__version__,
    }
    print(json.dumps(line))


if __name__ == "__main__":
    main()
