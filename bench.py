#!/usr/bin/env python
"""Throughput of the heatmap hot path on N B200s of one node (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path
    python bench.py --impl reference [...]                        # the reference's CPU algorithm
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N  # one rank per GPU (N > 1)
    python bench.py ... --dump-outputs DIR                        # also save the last timed step's outputs (.npy)

A step = DarkPose target encoding (joints -> targets, weights), masked-MSE forward+backward (pred, targets, weights ->
loss, grad) and GaussTaylor decode (pred, trans_inv -> keypoints, scores) of the same predicted heatmaps (K = 17, 64x48
float32), issued as BATCH-sized launches of the one-launch step kernel (sp_step_f32) over distinct buffer sets (working
set >> the 126 MB L2, so every launch streams from HBM); one pass over the buffer sets (--persons persons per GPU) makes
one step, and exactly --steps steps are timed. With N > 1 every rank does the same amount of work
on its own persons (weak scaling) and the decoded keypoints of a step are all-gathered over NCCL (double-buffered,
overlapped with the next step).

Prints ONE JSON line (rank 0). `value` = persons/s with inputs resident in HBM; `e2e` = the same path fed from pinned
host buffers through the public Python API (H2D of joints, predicted heatmaps and affines, D2H of loss and keypoints,
all inside the timed region; `e2e_device_heatmaps` = the same with the heatmaps resident, as a backbone leaves them);
`roofline` = the step kernel against the measured HBM copy bandwidth; `ops` / `small_batch` = every kernel at 64x48 and
96x72 and at the reference's literal batch sizes; `eval_job` = BASELINE config 5 through the sharded evaluator with a
bit-for-bit check against a single-device recompute; `cpu_baseline` = the oracle (a CPU restatement of the reference's
algorithm, pinned bit-exact to it) timed on this box's host. Both arms print the same `config`.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # a benchmark run leaves the tree as it found it (it may be read-only)

import torch  # noqa: E402

METRIC = "persons/sec encode+decode (K=17, 64x48 & 96x72) at 1/2/4/8 B200; % HBM roofline"
UNIT = "persons/s"
FALLBACK_HBM_GBS = 6650.0   # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--persons", type=int, default=8192, help="persons per GPU per step")
    ap.add_argument("--batch", type=int, default=1024, help="persons per kernel launch")
    ap.add_argument("--height", type=int, default=64)
    ap.add_argument("--width", type=int, default=48)
    ap.add_argument("--cpu-sample", type=int, default=256, help="persons in the cpu_baseline sample")
    ap.add_argument("--no-ops", action="store_true", help="skip the per-op sweep (64x48 and 96x72)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-eval", action="store_true", help="skip the cfg-5 eval job")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel, height, width, batch):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/r*_traffic.json), if one
    exists for this exact launch shape AND was measured on the library as it is now (the file records the source
    fingerprint of the build it profiled; a retuned kernel makes it stale and the answer None, never an old number)."""
    from simple_pose_b200 import build as _build
    names = {"encode": "encode_refine_kernel<1, 2>", "loss": "mse_ring_kernel<1, 0>", "decode": "decode_tma_kernel<0, 11>",
             "train_fused": "encode_mse_tile_kernel<12, 2, 1, 1>", "flip_decode": "decode_tma_kernel<1, 11>",
             "step": "step_kernel<1, 1, 0>"}
    key = "%s @ %dx%d,P=%d" % (names.get(kernel, kernel), height, width, batch)
    pdir = os.path.join(ROOT, "profiles")
    try:
        fingerprint = _build._fingerprint()
        files = sorted(f for f in os.listdir(pdir) if f.endswith("_traffic.json"))
        for f in reversed(files):
            with open(os.path.join(pdir, f)) as fh:
                table = json.load(fh)
            if table.get("_lib_fingerprint") != fingerprint:
                continue
            if key in table:
                return table[key]["dram_bytes_per_launch"], f
    except Exception:
        pass
    return None, None


# ------------------------------------------------------------------------------- clocks sampler
class ClockSampler(object):
    """nvidia-smi clocks/throttle reasons sampled every 200 ms while the timed region runs."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------- reference arm
def _encode_chunk(args):
    """Worker body (one DataLoader-worker equivalent): per-person Python/NumPy encode."""
    from oracle import heatmap_oracle as O
    joints, width, height = args
    torch.set_num_threads(1)
    t, w = O.encode_batch(joints, 2.0, (width, height))
    return torch.from_numpy(t), torch.from_numpy(w)      # travels back through shared memory


class CpuReference(object):
    """The reference's CPU algorithm for the step (oracle port, pinned bit-exact to the
    reference): encode = per-person Python/NumPy loop, optionally spread over worker processes
    the way the reference's DataLoader does (num_workers: 8 in its configs); loss fwd+bwd and
    decode = ATen on all host threads."""

    def __init__(self, persons, height, width, threads, encode_workers=1):
        from simple_pose_b200 import synth
        self.persons, self.h, self.w = persons, height, width
        torch.set_num_threads(max(1, threads))
        self.joints = synth.joints(persons, height=height, width=width, seed=0).numpy()
        self.tinv = synth.inverse_affines(persons, height=height, width=width, seed=0)[0]
        self.pool = None
        self.workers = encode_workers
        if encode_workers > 1:
            import numpy as np
            import torch.multiprocessing as mp
            self.chunks = [(c, width, height) for c in np.array_split(self.joints, encode_workers * 2) if len(c)]
            self.pool = mp.get_context("fork").Pool(encode_workers)
        self.targets = self.weights = self.pred = None

    def encode(self):
        from oracle import heatmap_oracle as O          # CPU baseline leg: the one product-side use
        if self.pool is not None:
            parts = self.pool.map(_encode_chunk, self.chunks)
            self.targets = torch.cat([p[0] for p in parts])
            self.weights = torch.cat([p[1] for p in parts])
        else:
            t, w = O.encode_batch(self.joints, 2.0, (self.w, self.h))
            self.targets, self.weights = torch.from_numpy(t), torch.from_numpy(w)

    def prepare_pred(self):
        from simple_pose_b200 import synth
        if self.targets is None:
            self.encode()
        self.pred = synth.predictions_like(self.targets, seed=1)

    def loss(self):
        from oracle import heatmap_oracle as O
        return O.masked_mse_loss_and_grad(self.pred, self.targets, self.weights)

    def decode(self):
        from oracle import heatmap_oracle as O
        return O.gauss_taylor_decode(self.pred, self.tinv)

    def timed_step(self):
        t0 = time.perf_counter()
        self.encode()
        t1 = time.perf_counter()
        self.loss()
        t2 = time.perf_counter()
        self.decode()
        t3 = time.perf_counter()
        return {"encode": t1 - t0, "loss": t2 - t1, "decode": t3 - t2, "step": t3 - t0}

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()


def cpu_reference_rates(persons, height, width, threads, reps=3, encode_workers=1):
    """persons/s per op and for the whole step (best of `reps` after one warm-up)."""
    ref = CpuReference(persons, height, width, threads, encode_workers)
    try:
        ref.prepare_pred()
        runs = [ref.timed_step() for _ in range(reps + 1)][1:]
    finally:
        ref.close()
    best = {k: min(r[k] for r in runs) for k in runs[0]}
    return {k: persons / v for k, v in best.items()}


def run_reference(args):
    if args.dump_outputs:
        raise SystemExit("bench.py: --dump-outputs writes the outputs of this repo's CUDA path; the reference arm has none")
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    workers = min(cores, 32)
    sample = args.cpu_sample * 4
    ref = CpuReference(sample, args.height, args.width, cores, encode_workers=workers)
    try:
        ref.prepare_pred()
        for _ in range(args.warmup):
            ref.timed_step()
        times = [ref.timed_step() for _ in range(args.steps)]
    finally:
        ref.close()
    total = sum(t["step"] for t in times)
    value = sample * len(times) / total
    per_op = {k: sample * len(times) / sum(t[k] for t in times) for k in ("encode", "loss", "decode")}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args, args.gpus),
        "sample_persons_per_step": sample,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d persons per step; encode in %d worker processes (the reference's DataLoader "
                                   "workers), loss fwd+bwd and decode on %d ATen threads; per-op persons/s: encode %.0f, "
                                   "loss %.0f, decode %.0f" % (sample, workers, cores, per_op["encode"], per_op["loss"], per_op["decode"])},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------- our arm
def bind_near_gpu(local):
    """Pin this rank's CPU affinity to the cores next to its GPU (NVML's ideal affinity) so that the
    pinned host buffers of the e2e leg are first-touched on the GPU's own NUMA node. Without it all
    8 ranks of a node tend to allocate on one socket and the e2e leg is bound by that socket's memory
    and the inter-socket link instead of 8 PCIe links. Best effort: returns a short description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        props = torch.cuda.get_device_properties(local)
        handle = None
        try:
            bus = "%08x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
            handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode() if hasattr(bus, "encode") else bus)
        except Exception:
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            index = int(visible.split(",")[local]) if visible and visible.split(",")[local].isdigit() else local
            handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        after = sorted(os.sched_getaffinity(0))
        return "cpu affinity %d -> %d cores (%d..%d)" % (before, len(after), after[0], after[-1])
    except Exception as exc:          # not fatal: the run proceeds with the inherited affinity
        return "unchanged (%s)" % type(exc).__name__


def make_inputs(persons, batch, height, width, device, seed):
    """Per-batch input sets generated on the device: joints, predicted heatmaps, affines."""
    from simple_pose_b200 import synth
    sets = []
    for i in range(persons // batch):
        s = seed + 1000 * i
        joints = synth.joints(batch, height=height, width=width, seed=s, device=device)
        pred = synth.heatmaps(batch, height=height, width=width, seed=s, noise=0.01, device=device)
        tinv = synth.inverse_affines(batch, height=height, width=width, seed=s, device=device)[0]
        sets.append((joints, pred, tinv))
    return sets


def time_ops(device, height, width, persons, batch, peak_gbs, only=None):
    """Per-op persons/s and roofline fraction (CUDA events around each launch, distinct buffers: the
    persons // batch buffer sets together exceed the 126 MB L2 several times over)."""
    from simple_pose_b200.pipeline import HeatmapHotPath, ALGO_BYTES
    from simple_pose_b200 import synth
    nb = max(1, persons // batch)
    sets = make_inputs(nb * batch, batch, height, width, device, seed=50)
    flips = [synth.heatmaps(batch, height=height, width=width, seed=900 + i, noise=0.01, device=device) for i in range(nb)]
    paths = [HeatmapHotPath(batch, 17, height, width, device=device) for _ in range(nb)]
    perm = paths[0].decoder._perm_on(device, 17, None)
    from simple_pose_b200.commons.transforms import encode_heat_maps_basic
    input_joints = [torch.cat([s[0][..., :2] * 4.0, s[0][..., 2:]], dim=-1).contiguous() for s in sets]
    ops = {
        "encode": lambda i: paths[i].encode(sets[i][0]),
        "loss": lambda i: paths[i].loss_fwd_bwd(sets[i][1]),
        "train_fused": lambda i: paths[i].train_fused(sets[i][0], sets[i][1]),
        "decode": lambda i: paths[i].decode(sets[i][1], sets[i][2]),
        "flip_decode": lambda i: paths[i].decode(sets[i][1], sets[i][2], flips[i], perm),
        "step": lambda i: paths[i].step_one_launch(sets[i][0], sets[i][1], sets[i][2]),
        # BasicSimpleTransform.get_heat_map (the ResNet solvers' quantised 13x13 encoder), joints in input pixels
        "encode_basic": lambda i: encode_heat_maps_basic(input_joints[i], 2.0, (width, height), 4, out=(paths[i].targets, paths[i].weights)),
    }
    if only is not None:
        ops = {k: v for k, v in ops.items() if k in only}
    out = {}
    for name, fn in ops.items():
        for i in range(nb):
            fn(i)
        torch.cuda.synchronize(device)
        times = []
        for _ in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(nb):
                fn(i)
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b) / nb)
        ms = statistics.median(times)
        bytes_per_launch = ALGO_BYTES["encode" if name == "encode_basic" else name](17, height, width) * batch
        gbs = bytes_per_launch / (ms * 1e-3) / 1e9
        out[name] = {"persons_per_s": batch / (ms * 1e-3), "ms_per_launch": ms, "GBps": gbs, "frac": gbs / peak_gbs,
                     "persons_per_launch": batch}
    del paths, sets, flips
    torch.cuda.empty_cache()
    return out


def train_side_numbers(device, persons=8192, reps=20, cpu_sample=256):
    """Train-side caller of the encoder (RefineSimpleTransform.__call__ minus the image work): boxes +
    image-pixel joints + augmentation draws -> heatmap-pixel joints + trans_inv in one launch
    (latency-bound, 240 B in / 280 B out per person: persons/s only), next to the oracle port on one core."""
    import numpy as np
    from simple_pose_b200 import synth
    from simple_pose_b200.commons.transforms import train_geometry
    smp = {k: v.to(device) for k, v in synth.train_samples(persons, seed=77).items()}
    args = (smp["boxes"], smp["joints"], smp["img_w"], smp["scale_ratio"], smp["rot"], smp["flip"].to(torch.uint8))
    for _ in range(3):
        train_geometry(*args)
    torch.cuda.synchronize(device)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        train_geometry(*args)
    b.record()
    b.synchronize()
    ms = a.elapsed_time(b) / reps
    from oracle import heatmap_oracle as O          # CPU baseline leg only
    cpu = synth.train_samples(cpu_sample, seed=77)
    t0 = time.perf_counter()
    for i in range(cpu_sample):
        box, w = cpu["boxes"][i].tolist(), int(cpu["img_w"][i])
        c, sc = O.box_center_scale(box[0], box[1], box[2] - box[0], box[3] - box[1], 0.75)
        sc = sc * np.float32(float(cpu["scale_ratio"][i]))
        j = cpu["joints"][i].numpy()
        if bool(cpu["flip"][i]):
            j = O.flip_joints_only(j, w)
        fwd, _ = O.affine_pair(c, sc, (48, 64), float(cpu["rot"][i]))
        O.affine_joints(j, fwd)
    cpu_s = time.perf_counter() - t0
    return {"persons": persons, "ms_per_launch": ms, "persons_per_s": persons / (ms * 1e-3), "launches": 1,
            "cpu_port_persons_per_s": cpu_sample / cpu_s, "cpu_cores": 1,
            "note": "sp_train_geometry_f32 (Python call included); CPU = oracle restatement of box_to_center_scale + "
                    "flip_joints + get_affine_transform(rot) + affine_transform_batch on %d persons" % cpu_sample}


def small_batch_numbers(device, height, width, batch=128, nbatch=64):
    """The literal cfg-1/cfg-2 shape (batch 128 = 26.7 MB per tensor, launch-latency regime) over `nbatch` distinct
    buffer sets (working set >> L2). Three ways to run the same step (encode + loss fwd/bwd + decode, identical
    outputs): the three stand-alone kernels, the one-launch step kernel (sp_step_f32), and either replayed from a
    CUDA graph; plus what a Python caller sees for ONE batch: launch from Python + sync, and `HeatmapHotPath.capture`
    (one graph launch) + sync."""
    from simple_pose_b200.pipeline import HeatmapHotPath, ALGO_BYTES
    sets = make_inputs(batch * nbatch, batch, height, width, device, seed=4242)
    paths = [HeatmapHotPath(batch, 17, height, width, device=device) for _ in range(nbatch)]
    side = torch.cuda.Stream(device)
    reps = 20

    def graphed(body):
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            for _ in range(2):
                body()
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            body()
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize(device)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            graph.replay()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / reps

    def eager(body):
        for _ in range(2):
            body()
        torch.cuda.synchronize(device)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            body()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / 5

    def three():
        for i in range(nbatch):
            paths[i].step(*sets[i], one_launch=False)

    def one():
        for i in range(nbatch):
            paths[i].step(*sets[i], one_launch=True)

    def fused_all():
        for i in range(nbatch):
            paths[i].train_fused(sets[i][0], sets[i][1])
            paths[i].decode(sets[i][1], sets[i][2])

    three_graph, one_graph, fused_graph = graphed(three), graphed(one), graphed(fused_all)
    three_eager, one_eager = eager(three), eager(one)

    def latency(call):
        lat = []
        for r in range(40):
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            call(r % nbatch)
            torch.cuda.synchronize(device)
            lat.append(time.perf_counter() - t0)
        return 1e6 * statistics.median(lat[8:])

    lat_three = latency(lambda i: paths[i].step(*sets[i], one_launch=False))
    lat_one = latency(lambda i: paths[i].step(*sets[i], one_launch=True))
    replays = [paths[i].capture(*sets[i]) for i in range(8)]
    lat_captured = latency(lambda i: replays[i % 8]())
    bytes3 = batch * (ALGO_BYTES["encode"](17, height, width) + ALGO_BYTES["loss"](17, height, width) + ALGO_BYTES["decode"](17, height, width))
    bytes1 = batch * ALGO_BYTES["step"](17, height, width)
    peak, _ = hbm_peak()
    out = {"batch": batch, "batches_per_graph": nbatch,
           "three_kernels": {"launches_per_batch": 3, "algorithmic_MB_per_batch": bytes3 / 1e6,
                             "graph_us_per_batch_step": 1e3 * three_graph / nbatch, "eager_us_per_batch_step": 1e3 * three_eager / nbatch,
                             "graph_frac_of_hbm_peak": bytes3 / (three_graph / nbatch * 1e-3) / 1e9 / peak},
           "one_launch": {"launches_per_batch": 1, "algorithmic_MB_per_batch": bytes1 / 1e6,
                          "graph_us_per_batch_step": 1e3 * one_graph / nbatch, "eager_us_per_batch_step": 1e3 * one_eager / nbatch,
                          "graph_frac_of_hbm_peak": bytes1 / (one_graph / nbatch * 1e-3) / 1e9 / peak,
                          "graph_persons_per_s": batch * nbatch / (one_graph * 1e-3)},
           # kept under their round-1 names: the best way to run the literal batch-128 step
           "graph_us_per_batch_step": 1e3 * min(one_graph, three_graph) / nbatch,
           "graph_persons_per_s": batch * nbatch / (min(one_graph, three_graph) * 1e-3),
           "single_batch_step_latency_us": min(lat_one, lat_captured),
           "single_batch_step_latency_detail_us": {"three_kernels_from_python": lat_three, "one_launch_from_python": lat_one,
                                                    "one_launch_captured_graph": lat_captured},
           "fused_graph_us_per_batch_step": 1e3 * fused_graph / nbatch,
           "fused_graph_persons_per_s": batch * nbatch / (fused_graph * 1e-3),
           "note": "one batch-128 tensor is 26.7 MB = 4 us at the HBM roofline; latencies are host wall clock around call + "
                   "synchronize (median of 32); fused_* = fused encode+loss+acc kernel + decode, 2 launches per batch, targets not written"}
    del replays, paths, sets
    torch.cuda.empty_cache()
    return out


def single_device_rows(es, lo, hi, device, height, width):
    """Result rows of global persons [lo, hi) (image-aligned) computed on ONE device with NO collective,
    through the stand-alone kernels (box affine, decode, float64 pack, rescore, NMS) -- a different code
    path from the fused rows kernels ``ShardedPoseEvaluator`` runs. Returns (keypoints f32 [n, 3K],
    keep bool [n], scores f64 [n])."""
    import numpy as np
    from simple_pose_b200.datasets.naive_data import box_affines, pack_keypoints, rescore_and_nms
    from simple_pose_b200.metrics.pose_metrics import GaussTaylorKeyPointDecoder
    i0, i1 = int(np.searchsorted(es.seg, lo)), int(np.searchsorted(es.seg, hi))
    assert es.seg[i0] == lo and es.seg[i1] == hi
    hm = es.heatmaps(lo, hi, device)
    aff = box_affines(es.boxes[lo:hi].to(device), (4 * width, 4 * height), (width, height))
    xy, conf = GaussTaylorKeyPointDecoder()(hm, aff["trans_inv"])
    kps = pack_keypoints(xy, conf)
    seg = (es.seg[i0:i1 + 1] - lo).astype(np.int32)
    keep, scores, _ = rescore_and_nms(kps, es.box_scores[lo:hi].to(device), aff["area"].double(), seg)
    return torch.cat([xy, conf], dim=-1).reshape(hi - lo, -1), keep.bool(), scores


def eval_job_numbers(device, world, rank, persons=104000, mean_group=20.0, height=64, width=48, reps=5, chunks=None,
                     transport="auto"):
    """BASELINE config 5: a COCO-val-sized eval job (~104 k person boxes in ~5 k images, 30 % of them
    near-duplicate detections) through ``ShardedPoseEvaluator``: per rank box -> affine, then per chunk
    GaussTaylor decode into the result rows, rescoring + OKS-NMS on the rows, NCCL all-gather of the chunk
    (in place, overlapped with the next chunk's decode). Fixed total work (strong scaling); device-timed,
    max over ranks. The content of the job depends on the person index only, so ``table_checksum`` must be
    the same number at every N, and ``matches_single_device`` reports a bit-for-bit comparison of the
    gathered table with a collective-free recompute (this rank's first and last image and a fixed slice
    of >= 512 persons around the middle of the global table) through the stand-alone kernels."""
    import numpy as np
    import torch.distributed as dist
    from simple_pose_b200 import synth
    from simple_pose_b200.eval_shard import ShardedPoseEvaluator, row_keep, row_keypoints, row_scores
    es = synth.EvalSet(persons=persons, mean_group=mean_group, height=height, width=width)
    total, images = es.persons, es.images
    ev = ShardedPoseEvaluator(chunks=chunks, transport=transport)
    ev.plan(es.seg)
    lo, hi = ev.my_persons()
    n = hi - lo
    hm = es.heatmaps(lo, hi, device)
    boxes = es.boxes[lo:hi].to(device)
    box_scores = es.box_scores[lo:hi].to(device)
    torch.cuda.synchronize(device)
    times = []
    for r in range(reps + 2):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        raw = ev.run(hm, None, box_scores, None, boxes=boxes, input_shape=(4 * width, 4 * height), compact=False)
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        if r >= 2:
            times.append(ms)
    ms = statistics.median(times)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    table = raw.rows()
    b.record()
    b.synchronize()
    compact_ms = a.elapsed_time(b)
    kept = int(row_keep(table).sum().item())
    checksum = synth.table_checksum(table)
    del hm
    torch.cuda.empty_cache()
    # ---- parity of the sharded, NCCL-gathered table against a collective-free recompute on this device
    seg = es.seg
    mid = int(np.searchsorted(seg, total // 2)) - 12
    mid = max(0, min(mid, images - 1))
    end = mid
    while end < images and seg[end] - seg[mid] < 512:
        end += 1
    i_first, i_last = int(ev.cuts[rank]), int(ev.cuts[rank + 1]) - 1
    ranges = [(int(seg[mid]), int(seg[end]))]
    if i_last >= i_first:
        ranges += [(int(seg[i_first]), int(seg[i_first + 1])), (int(seg[i_last]), int(seg[i_last + 1]))]
    ok, checked = True, 0
    for (p0, p1) in ranges:
        kp, keep, scores = single_device_rows(es, p0, p1, device, height, width)
        part = table[p0:p1]
        ok = ok and torch.equal(row_keypoints(part).reshape(p1 - p0, -1), kp) and torch.equal(row_keep(part), keep) \
            and torch.equal(row_scores(part), scores)
        checked += p1 - p0
    flag = torch.tensor([1 if ok else 0, checksum & 0x7fffffff, (checksum >> 31) & 0x7fffffff], dtype=torch.int64, device=device)
    if world > 1:
        lo_f, hi_f = flag.clone(), flag.clone()
        dist.all_reduce(lo_f, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_f, op=dist.ReduceOp.MAX)
        ok = bool(lo_f[0].item() == 1) and bool(torch.equal(lo_f[1:], hi_f[1:]))      # every rank matches AND holds the same table
    del table
    torch.cuda.empty_cache()
    return {"workload": "cfg5: box->affine + GaussTaylor decode + rescoring + OKS-NMS + all-gather of result rows",
            "persons": total, "images": images, "duplicate_detections": es.duplicates, "n_gpus": world, "scaling": "strong",
            "ms": ms, "persons_per_s": total / (ms * 1e-3), "kept_after_nms": kept, "chunks_per_rank": int(ev.ccuts.shape[1] - 1),
            "transport": ev.transport, "compact_ms": compact_ms, "table_checksum": "%016x" % (checksum & 0xffffffffffffffff),
            "matches_single_device": bool(ok), "persons_rechecked_per_rank": checked,
            "decode_read_GBps_per_gpu": (n * (17 * height * width * 4)) / (ms * 1e-3) / 1e9}


def step_cycles():
    """Passes over the rotating buffer sets per step: one, so that a step is a fixed amount of work (--persons persons
    per GPU) and --steps sets how much work is timed. SP_BENCH_CYCLES overrides it (a profiling aid)."""
    if os.environ.get("SP_BENCH_CYCLES"):
        return max(1, int(os.environ["SP_BENCH_CYCLES"]))
    return 1


def bench_config(args, world):
    """The `config` object: identical in the product and the reference arm (same workload, same sizes)."""
    from simple_pose_b200.pipeline import ALGO_BYTES
    H, W, B = args.height, args.width, args.batch
    base = max(B, (args.persons // B) * B)
    cycles = step_cycles()
    per_person = ALGO_BYTES["encode"](17, H, W) + ALGO_BYTES["loss"](17, H, W) + ALGO_BYTES["decode"](17, H, W)
    return {"workload": "cfg2+cfg1 step: DarkPose target encoding + masked joints-MSE fwd/bwd + GaussTaylor decode of the same "
                        "predicted heatmaps (+ NCCL all-gather of the keypoints when N>1), K=17, %dx%d float32" % (H, W),
            "persons_per_gpu_per_step": base * cycles, "persons_per_launch": B, "height": H, "width": W, "joints": 17,
            "distinct_buffer_sets": base // B, "passes_over_the_buffer_sets_per_step": cycles,
            "l2": "inputs larger than L2: %d distinct buffer sets of %d persons, %.0f MB of separate-kernel traffic per pass" %
                  (base // B, B, base * per_person / 1e6),
            "parallelism": "persons sharded, dp%d" % world}


DUMP_LIMIT_BYTES = 64 << 20


def dump_sample_size(world, P, B, H, W):
    """Persons in the targets / gradient sample of `dump_outputs`: what fits in 64 MB beside the keypoints, losses and
    weights (4 KB kept for the .npy headers). Every rank calls it before the timed steps, so a table too large to dump
    stops all ranks there."""
    fixed = world * P * 17 * 3 * 4 + (P // B) * 4 + P * 17 * 4
    n = min(P, (DUMP_LIMIT_BYTES - 4096 - fixed) // (2 * 17 * H * W * 4 + 8))
    if n < 1:
        raise SystemExit("bench.py: --dump-outputs: the keypoint table alone exceeds 64 MB; use fewer --persons")
    return n


def dump_outputs(out_dir, paths, keypoints, world, P, N, cycles, B, H, W):
    """Writes what the last timed step handed its caller, as float32 / float64 .npy files in `out_dir`:

        coords [world*P, 17, 2], maxval [world*P, 17, 1]   decoded keypoints of the step's last pass (every rank's when
                                                           world > 1: the all-gathered table; earlier passes repeat them)
        loss [P // B]                                      per-launch loss of this rank
        weights [P, 17]                                    this rank's target weights
        targets_sample, grad_sample [n, 17, H, W]          targets and loss gradient of n persons of this rank, a fixed
        sample_persons [n] (float64)                       seeded sample (person indices) sized to keep the total <= 64 MB

    The inputs depend on the flags only (seeded), so two builds run with the same flags can be compared array by array."""
    import numpy as np
    last = slice((cycles - 1) * P, cycles * P)
    blocks = keypoints.view(world, N * 17 * 3)
    out = {"coords": blocks[:, :N * 17 * 2].reshape(world, N, 17, 2)[:, last].reshape(world * P, 17, 2),
           "maxval": blocks[:, N * 17 * 2:].reshape(world, N, 17, 1)[:, last].reshape(world * P, 17, 1),
           "loss": torch.stack([p.loss for p in paths]),
           "weights": torch.cat([p.weights for p in paths])}
    out = {k: v.cpu().numpy() for k, v in out.items()}
    n = dump_sample_size(world, P, B, H, W)
    idx = np.sort(np.random.default_rng(2024).choice(P, size=n, replace=False))
    out["targets_sample"] = torch.stack([paths[j // B].targets[j % B] for j in idx]).cpu().numpy()
    out["grad_sample"] = torch.stack([paths[j // B].grad[j % B] for j in idx]).cpu().numpy()
    out["sample_persons"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print("bench.py: wrote %s to %s" % (", ".join(sorted(out)), out_dir), file=sys.stderr, flush=True)


def run_ours(args):
    import torch.distributed as dist
    from simple_pose_b200 import _abi
    from simple_pose_b200.pipeline import HeatmapHotPath, ALGO_BYTES, run_batches

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    numa = {"text": "not requested"}
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    _abi.lib()
    peak_gbs, peak_src = hbm_peak()
    config = bench_config(args, world)
    H, W, B = args.height, args.width, args.batch
    P = max(B, (args.persons // B) * B)          # persons per pass over the buffer sets
    nb = P // B
    cycles = step_cycles()
    if args.dump_outputs:
        dump_sample_size(world, P, B, H, W)

    sets = make_inputs(P, B, H, W, device, seed=rank * 7919)
    # decoded keypoints of all batches of all passes of a step land in one flat send buffer: [N*17*2 coords | N*17
    # scores], N = P * cycles persons; ONE all-gather per step (few large collectives beat many small ones), and two
    # send / receive buffers alternate between steps so that a step never waits for the previous step's all-gather
    N = P * cycles
    kp_local = [torch.empty(N * 17 * 3, dtype=torch.float32, device=device) for _ in range(2)]
    views = [[[(kp[:N * 17 * 2].view(N, 17, 2)[(c * nb + i) * B:(c * nb + i + 1) * B],
                kp[N * 17 * 2:].view(N, 17, 1)[(c * nb + i) * B:(c * nb + i + 1) * B]) for i in range(nb)]
              for c in range(cycles)] for kp in kp_local]
    paths = [HeatmapHotPath(B, 17, H, W, device=device, coords=views[0][0][i][0], maxval=views[0][0][i][1]) for i in range(nb)]
    kp_all = [torch.empty(world * N * 17 * 3, dtype=torch.float32, device=device) for _ in range(2)] if world > 1 else None
    one_launch = paths[0].one_launch_supported()
    pending = [None, None]
    state = {"step": 0}

    def finish_gather(side=None):
        for sd in ((0, 1) if side is None else (side,)):
            if pending[sd] is not None:
                pending[sd].wait()        # stream-level wait (no host block): this buffer may be overwritten again
                pending[sd] = None

    def step(three_kernels=not one_launch):
        side = state["step"] & 1
        state["step"] += 1
        finish_gather(side)               # the all-gather that read this send buffer two steps ago

        def start_gather():
            # asynchronous: NCCL's stream waits for the kernels enqueued so far; whatever follows on the compute
            # stream (the rest of this step, the next step) overlaps the collective
            if world > 1:
                pending[side] = dist.all_gather_into_tensor(kp_all[side], kp_local[side], async_op=True)
        for c in range(cycles):
            for i in range(nb):
                paths[i].coords, paths[i].maxval = views[side][c][i]
            last = c == cycles - 1
            if three_kernels:
                run_batches(paths, sets, after_decode=start_gather if last else None)
            else:
                for i in range(nb):
                    paths[i].step_one_launch(sets[i][0], sets[i][1], sets[i][2])
                if last:
                    start_gather()

    def barrier():
        finish_gather()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def timed(fn, steps):
        """ms per call of `fn` over `steps` calls: CUDA events on the launching stream, max over ranks."""
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            fn()
        finish_gather()                   # the last all-gather is inside the timed region
        t1.record()
        barrier()
        ms = t0.elapsed_time(t1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    def kernel_ms(fn, rounds):
        """Average launch duration of one kernel: CUDA events around nb back-to-back launches
        (one per distinct buffer set) on the launching stream; median over `rounds`."""
        per_round = []
        for _ in range(rounds):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(nb):
                fn(i)
            b.record()
            b.synchronize()
            per_round.append(a.elapsed_time(b) / nb)
        return statistics.median(per_round)      # a round that collides with an nvidia-smi poll is an outlier

    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_per_step = timed(step, args.steps)                         # THE timed region: exactly --steps steps
    if args.dump_outputs and rank == 0:                           # before anything below overwrites the step's outputs
        side = (state["step"] - 1) & 1
        dump_outputs(args.dump_outputs, paths, kp_all[side] if world > 1 else kp_local[side], world, P, N, cycles, B, H, W)
    value = world * P * cycles / (ms_per_step * 1e-3)
    # per-kernel durations, still under the clock sampler
    rounds = max(3, min(20, args.steps))
    op_ms = {"encode": kernel_ms(lambda i: paths[i].encode(sets[i][0]), rounds),
             "loss": kernel_ms(lambda i: paths[i].loss_fwd_bwd(sets[i][1]), rounds),
             "decode": kernel_ms(lambda i: paths[i].decode(sets[i][1], sets[i][2]), rounds)}
    if one_launch:
        op_ms["step"] = kernel_ms(lambda i: paths[i].step_one_launch(sets[i][0], sets[i][1], sets[i][2]), rounds)
    side_steps = max(3, min(50, args.steps))
    # the same step through the three stand-alone kernels (round 1's headline: encode, loss fwd/bwd and decode launched
    # separately, grouped by kernel, the all-gather overlapped with the last pass's encode/loss kernels)
    step(True)
    three_ms = timed(lambda: step(True), 3) / cycles
    three = {"persons_per_s": world * P / (three_ms * 1e-3), "ms_per_pass": three_ms, "launches_per_pass": 3 * nb,
             "algorithmic_bytes_per_person": ALGO_BYTES["encode"](17, H, W) + ALGO_BYTES["loss"](17, H, W) + ALGO_BYTES["decode"](17, H, W),
             "note": "sp_encode_f32 + sp_mse_fwd_bwd_f32 + sp_decode_ws_f32 per batch (pred read twice, targets written and read back)"}
    # ... and through the fused training kernel (encode + loss + HeatMapAcc argmaxes in one pass, targets never
    # materialised: SURVEY 8f ranks 1-2) followed by the decode; no all-gather in this loop
    def fused_pass():
        for i in range(nb):
            paths[i].train_fused(sets[i][0], sets[i][1])
            paths[i].decode(sets[i][1], sets[i][2])
    for _ in range(2):
        fused_pass()
    fused_ms = timed(fused_pass, side_steps)
    fused = {"persons_per_s": world * P / (fused_ms * 1e-3), "ms_per_pass": fused_ms, "launches_per_pass": 2 * nb,
             "algorithmic_bytes_per_person": ALGO_BYTES["train_fused"](17, H, W) + ALGO_BYTES["decode"](17, H, W),
             "note": "same persons, loss/grad/weights/keypoints identical; encode+loss+HeatMapAcc fused into one pass "
                     "(targets never written), then decode; no all-gather in this loop"}
    clocks = sampler.stop() if rank == 0 else None

    headline = "step" if one_launch else max(("encode", "loss", "decode"), key=op_ms.get)
    dom_bytes = ALGO_BYTES[headline](17, H, W) * B
    achieved = dom_bytes / (op_ms[headline] * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic(headline, H, W, B)
    launch_ms = {"step": op_ms["step"]} if one_launch else {k: op_ms[k] for k in ("encode", "loss", "decode")}
    roofline = {"bound": "hbm", "kernel": headline, "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                "frac": achieved / peak_gbs, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dom_bytes, "ms_per_launch": op_ms[headline],
                "share_of_step": op_ms[headline] / sum(launch_ms.values()),
                "step_ms_explained_by_kernel_launches": cycles * nb * sum(launch_ms.values()),
                "all_kernels": {k: {"ms_per_launch": op_ms[k],
                                    "GBps": ALGO_BYTES[k](17, H, W) * B / (op_ms[k] * 1e-3) / 1e9,
                                    "frac": ALGO_BYTES[k](17, H, W) * B / (op_ms[k] * 1e-3) / 1e9 / peak_gbs}
                                for k in op_ms}}

    # end to end through the public Python API, host buffers in, host results out
    e2e = e2e_dev = None
    if not args.no_e2e:
        saved_affinity = os.sched_getaffinity(0)
        if not os.environ.get("SP_BENCH_NO_BIND"):
            numa["text"] = bind_near_gpu(local)          # pinned host buffers land on the GPU's NUMA node
        try:
            e2e = run_e2e(args, device, world, rank, P, B, H, W)
            e2e_dev = run_e2e_device_heatmaps(args, device, world, rank, P, B, H, W, sets)
        finally:
            os.sched_setaffinity(0, saved_affinity)      # the CPU baseline below uses every core again
    del paths, sets, views, kp_local, kp_all, pending
    torch.cuda.empty_cache()

    # per-op sweep, literal small batches, train-side caller: one GPU's worth of numbers, measured by rank 0 at every N
    # (the other ranks wait at the barrier below)
    ops = small = train_side = None
    if rank == 0 and not args.no_ops:
        ops = {"64x48": time_ops(device, 64, 48, 8192, 1024, peak_gbs),
               "96x72": time_ops(device, 96, 72, 4096, 512, peak_gbs),
               # the literal BASELINE batch sizes (launch-latency regime): cfg 1/2 = batch 128, cfg 3 = batch 256 flip test
               "64x48_batch128": time_ops(device, 64, 48, 8192, 128, peak_gbs),
               "64x48_batch256": time_ops(device, 64, 48, 8192, 256, peak_gbs, only=("flip_decode", "decode", "step"))}
        small = small_batch_numbers(device, H, W)
        train_side = train_side_numbers(device)
    if world > 1:
        dist.barrier()

    eval_job = None
    if not args.no_eval:
        eval_job = eval_job_numbers(device, world, rank, height=H, width=W)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        r = cpu_reference_rates(args.cpu_sample, H, W, cores, reps=3, encode_workers=1)
        cpu = {"value": r["step"], "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "%d persons, best of 3: encode %.0f/s (1 core, Python loop), loss fwd+bwd %.0f/s and decode "
                         "%.0f/s (ATen, %d threads)" % (args.cpu_sample, r["encode"], r["loss"], r["decode"], cores),
               "per_op": {k: r[k] for k in ("encode", "loss", "decode")}}

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        if eval_job is not None and not eval_job["matches_single_device"]:
            raise SystemExit(3)
        return
    launches_per_pass = nb if one_launch else 3 * nb
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
        "step_path": ("sp_step_f32: one launch per batch does decode + encode + loss fwd/bwd on one staged copy of each map "
                      "(same outputs as the three stand-alone kernels, see three_kernel_step)") if one_launch else
                     "three stand-alone kernels per batch, grouped by kernel",
        "e2e_host_binding": numa["text"],
        "clocks": clocks, "e2e": e2e, "e2e_device_heatmaps": e2e_dev,
        "gpu_launches": args.steps * cycles * launches_per_pass,
        "roofline": roofline, "cpu_baseline": cpu, "ops": ops, "small_batch": small, "eval_job": eval_job,
        "three_kernel_step": three, "fused_step": fused, "train_side": train_side,
    }
    print(json.dumps(line), flush=True)
    if eval_job is not None and not eval_job["matches_single_device"]:
        raise SystemExit("bench.py: the sharded eval table differs from the single-device recompute")


def run_e2e(args, device, world, rank, P, B, H, W):
    """Same step through the public API with HOST buffers: per batch, H2D of joints, predicted
    heatmaps and affines from pinned memory on a copy stream (double-buffered against compute),
    then encode/loss/decode, then D2H of the loss and the keypoints."""
    import torch.distributed as dist
    from simple_pose_b200 import synth
    from simple_pose_b200.commons.transforms import encode_heat_maps
    from simple_pose_b200.metrics.pose_metrics import GaussTaylorKeyPointDecoder
    from simple_pose_b200.processors.loss import JointsMSELoss

    nb = P // B
    # host inputs (pinned). One batch of heatmaps is generated on the device and replicated on
    # the host side with a cheap perturbation so that host memory holds P distinct persons.
    h_joints = torch.empty((P, 17, 3), dtype=torch.float32).pin_memory()
    h_pred = torch.empty((P, 17, H, W), dtype=torch.float32).pin_memory()
    h_tinv = torch.empty((P, 2, 3), dtype=torch.float32).pin_memory()
    for i in range(nb):
        s = 31 + 1000 * i + rank
        h_joints[i * B:(i + 1) * B].copy_(synth.joints(B, height=H, width=W, seed=s, device=device))
        h_pred[i * B:(i + 1) * B].copy_(synth.heatmaps(B, height=H, width=W, seed=s, device=device))
        h_tinv[i * B:(i + 1) * B].copy_(synth.inverse_affines(B, height=H, width=W, seed=s, device=device)[0])
    # contiguous destinations: a device -> host copy into a strided slice goes through a staging tensor and a host-side
    # copy that waits for the stream, which would serialise the batches
    h_xy = torch.empty((P, 17, 2), dtype=torch.float32).pin_memory()
    h_conf = torch.empty((P, 17, 1), dtype=torch.float32).pin_memory()
    h_loss = torch.empty((nb,), dtype=torch.float32).pin_memory()
    torch.cuda.synchronize(device)

    dec = GaussTaylorKeyPointDecoder()
    crit = JointsMSELoss()
    copy_stream = torch.cuda.Stream(device)
    compute = torch.cuda.current_stream(device)
    slots = [dict(j=torch.empty((B, 17, 3), device=device), p=torch.empty((B, 17, H, W), device=device),
                  t=torch.empty((B, 2, 3), device=device), ready=torch.cuda.Event(), free=torch.cuda.Event())
             for _ in range(2)]

    def upload(i):
        s = slots[i % 2]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(s["free"])
            s["j"].copy_(h_joints[i * B:(i + 1) * B], non_blocking=True)
            s["p"].copy_(h_pred[i * B:(i + 1) * B], non_blocking=True)
            s["t"].copy_(h_tinv[i * B:(i + 1) * B], non_blocking=True)
            s["ready"].record(copy_stream)

    def step():
        upload(0)
        for i in range(nb):
            if i + 1 < nb:
                upload(i + 1)
            s = slots[i % 2]
            compute.wait_event(s["ready"])
            targets, weights = encode_heat_maps(s["j"])
            pred = s["p"].requires_grad_(True)
            loss = crit(pred, targets, weights)
            loss.backward()                                   # grad stays on the device (feeds the backbone)
            xy, conf = dec(pred.detach(), s["t"])
            pred.grad = None
            s["p"].requires_grad_(False)
            h_xy[i * B:(i + 1) * B].copy_(xy, non_blocking=True)
            h_conf[i * B:(i + 1) * B].copy_(conf.reshape(B, 17, 1), non_blocking=True)
            h_loss[i:i + 1].copy_(loss.detach().reshape(1), non_blocking=True)
            s["free"].record(compute)
        torch.cuda.synchronize(device)
        return float(h_loss.sum())

    for s in slots:
        s["free"].record(compute)
    for _ in range(2):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize(device)
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    h2d = P * (17 * 3 * 4 + 17 * H * W * 4 + 24)
    d2h = P * 17 * 3 * 4 + nb * 4
    return {"value": world * P * steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "steps": steps, "ms_per_step": 1e3 * dt / steps, "h2d_GBps_per_gpu": h2d * steps / dt / 1e9,
            "note": "public API (encode_heat_maps, JointsMSELoss+backward, GaussTaylorKeyPointDecoder) on pinned host "
                    "inputs incl. the predicted heatmaps; PCIe-bound"}


def run_e2e_device_heatmaps(args, device, world, rank, P, B, H, W, sets):
    """The realistic end-to-end leg: what a training / validation loop ships per batch is the joints and the affines
    (H2D, pinned); the predicted heatmaps are the backbone's output and already live on the device (here: the resident
    synthetic ones); the loss and the keypoints go back to the host (D2H). One `HeatmapHotPath.step` per batch."""
    import torch.distributed as dist
    from simple_pose_b200.pipeline import HeatmapHotPath
    nb = P // B
    h_joints = torch.empty((P, 17, 3), dtype=torch.float32).pin_memory()
    h_tinv = torch.empty((P, 2, 3), dtype=torch.float32).pin_memory()
    for i in range(nb):
        h_joints[i * B:(i + 1) * B].copy_(sets[i][0])
        h_tinv[i * B:(i + 1) * B].copy_(sets[i][2])
    h_xy = torch.empty((P, 17, 2), dtype=torch.float32).pin_memory()         # contiguous destinations, see run_e2e
    h_conf = torch.empty((P, 17, 1), dtype=torch.float32).pin_memory()
    h_loss = torch.empty((nb,), dtype=torch.float32).pin_memory()
    hp = [HeatmapHotPath(B, 17, H, W, device=device) for _ in range(2)]          # double-buffered outputs
    d_joints = [torch.empty((B, 17, 3), device=device) for _ in range(2)]
    d_tinv = [torch.empty((B, 2, 3), device=device) for _ in range(2)]
    torch.cuda.synchronize(device)

    replays = None
    # three streams, two slots: the upload of batch i+1 and the read-back of batch i-1 run beside the kernel of batch i
    compute = torch.cuda.current_stream(device)
    up, down = torch.cuda.Stream(device), torch.cuda.Stream(device)
    ev_in = [torch.cuda.Event() for _ in range(2)]        # slot's inputs are on the device
    ev_done = [torch.cuda.Event() for _ in range(2)]      # slot's kernel has finished: inputs reusable, outputs readable
    ev_out = [torch.cuda.Event() for _ in range(2)]       # slot's outputs are on the host: outputs reusable

    def upload(i):
        s = i & 1
        with torch.cuda.stream(up):
            up.wait_event(ev_done[s])
            d_joints[s].copy_(h_joints[i * B:(i + 1) * B], non_blocking=True)
            d_tinv[s].copy_(h_tinv[i * B:(i + 1) * B], non_blocking=True)
            ev_in[s].record(up)

    def step():
        upload(0)
        for i in range(nb):
            s = i & 1
            if i + 1 < nb:
                upload(i + 1)
            compute.wait_event(ev_in[s])
            compute.wait_event(ev_out[s])
            if replays is None:
                loss, xy, conf = hp[s].step(d_joints[s], sets[i][1], d_tinv[s])
            else:                                   # the same step replayed from the graph HeatmapHotPath.capture made
                replays[i]()
                loss, xy, conf = hp[s].loss, hp[s].coords, hp[s].maxval
            ev_done[s].record(compute)
            with torch.cuda.stream(down):
                down.wait_event(ev_done[s])
                h_xy[i * B:(i + 1) * B].copy_(xy, non_blocking=True)
                h_conf[i * B:(i + 1) * B].copy_(conf.reshape(B, 17, 1), non_blocking=True)
                h_loss[i:i + 1].copy_(loss.reshape(1), non_blocking=True)
                ev_out[s].record(down)
        torch.cuda.synchronize(device)
        return float(h_loss.sum())

    for _ in range(2):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    steps = max(3, min(args.steps, 20))
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    check_eager = (float(h_loss.sum()), h_xy.clone(), h_conf.clone())
    # the same loop with the per-batch step replayed from a captured graph (one graph per input buffer set). An extra, not the
    # leg's number: if the capture fails on a box, say so and keep the collectives of the ranks matched
    dt_graph = same = graph_error = None
    try:
        replays = [hp[i & 1].capture(d_joints[i & 1], sets[i][1], d_tinv[i & 1]) for i in range(nb)]
        for _ in range(2):
            step()
    except RuntimeError as exc:
        graph_error, replays = repr(exc)[:200], None
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    if graph_error is None:
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt_graph = time.perf_counter() - t0
        # keypoints bit-identical; the loss to its float64 summation order (maps of the dynamic tail go to whichever warp asks first)
        same = abs(float(h_loss.sum()) - check_eager[0]) <= 1e-6 * abs(check_eager[0]) and torch.equal(h_xy, check_eager[1]) \
            and torch.equal(h_conf, check_eager[2])
    if world > 1:
        t = torch.tensor([dt, dt_graph or 0.0, 0.0 if graph_error is None else 1.0, 0.0 if same else 1.0],
                         dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t[0].item())
        if float(t[2].item()) > 0.0:                 # some rank could not capture
            dt_graph, graph_error = None, graph_error or "graph capture failed on another rank"
        else:
            dt_graph, same = float(t[1].item()), float(t[3].item()) == 0.0
    return {"value": world * P * steps / dt, "unit": UNIT, "h2d_bytes_per_step": P * (17 * 3 * 4 + 24),
            "d2h_bytes_per_step": P * 17 * 3 * 4 + nb * 4, "steps": steps, "ms_per_step": 1e3 * dt / steps,
            "persons_per_step": P, "graph_replay_value": (world * P * steps / dt_graph) if dt_graph else None,
            "graph_replay_ms_per_step": (1e3 * dt_graph / steps) if dt_graph else None,
            "graph_replay_same_results": bool(same) if dt_graph else None, "graph_replay_error": graph_error,
            "note": "joints + affines H2D from pinned memory, heatmaps resident on the device (backbone output), loss + keypoints "
                    "D2H; HeatmapHotPath.step per batch (upload, kernel and read-back on three streams, two slots), host wall clock incl. "
                    "the final synchronize; graph_replay_* = the same loop with the step replayed from HeatmapHotPath.capture's graph"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
