"""TEST INFRASTRUCTURE ONLY -- randomised pin of the restatement against the mounted reference.

    python -m oracle.fuzz_vs_reference [--seconds 120 | --rounds N] [--seed 0]

Draws random shapes / parameters for every row of the hot path, runs the unmodified reference
(``oracle/ref_loader.py``) and the restatement (``oracle/heatmap_oracle.py``) on the same inputs and
demands bit equality; prints a per-row case count. The draws depend on the seed only, so ``run`` with a
round count also returns one digest per round of the restatement's outputs (``oracle/pins.py``): with
``ref=None`` the same rounds run without the reference and are checked against recorded digests
(tests/test_oracle_vs_reference.py::test_randomised_pin_short).
"""
import argparse
import sys
import time
import warnings

import numpy as np
import torch

from oracle import heatmap_oracle as O
from oracle import pins
from oracle import ref_loader
from simple_pose_b200 import synth


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def run(ref, seed, rounds=None, seconds=None):
    """Runs `rounds` rounds (or as many as fit in `seconds`) and returns (rounds run, per-row case counts, one digest
    per round of the restatement's outputs). `ref` is ref_loader.load() or None (restatement only, nothing compared)."""
    rng = np.random.default_rng(seed)
    counts = {}
    digests = []
    t_end = time.time() + (seconds if seconds is not None else float("inf"))
    it = 0
    while (it < rounds) if rounds is not None else (time.time() < t_end):
        it += 1
        ours = []
        w, h = int(rng.integers(2, 25)) * 4, int(rng.integers(8, 100))
        k = int(rng.integers(1, 20))
        seed = int(rng.integers(0, 2 ** 31 - 1))
        # encode (Refine + Basic)
        sigma = float(rng.choice([1.0, 1.5, 2.0, 2.5, 3.0]))
        joints = synth.joints(2, num_joints=k, height=h, width=w, seed=seed).numpy()
        joints[0, 0, :2] = rng.choice([-1e4, 1e4, -7.0, 0.0, w - 1, w + 6.0], size=2)
        for j in joints:
            ot, ow = O.encode_person(j, sigma, (w, h))
            ours += [ot, ow]
            if ref:
                rt, rw = ref.get_heat_map(j, sigma, (w, h))
                assert np.array_equal(bits(rt), bits(ot)) and np.array_equal(rw, ow), ("encode", w, h, sigma, seed)
            jb = j.copy(); jb[:, :2] *= 4
            ot, ow = O.encode_person_basic(jb, sigma, (w, h), 4)
            ours += [ot, ow]
            if ref:
                rt, rw = ref.get_heat_map_basic(jb, sigma, (w, h), 4)
                assert np.array_equal(bits(rt), bits(ot)) and np.array_equal(rw, ow), ("encode_basic", w, h, sigma, seed)
        counts["encode"] = counts.get("encode", 0) + 4
        # decoders (the reference's GaussTaylor is fixed to 17 joints by its depthwise conv)
        if h >= 12 and w >= 12:
            noise = float(rng.choice([0.0, 0.005, 0.02, 0.05]))
            hm = synth.heatmaps(2, joints=17, height=h, width=w, seed=seed, noise=noise)
            tinv = synth.inverse_affines(2, height=h, width=w, seed=seed)[0]
            ks = int(rng.choice([3, 5, 7, 11, 13]))
            oc, om = O.gauss_taylor_decode(hm, tinv, ks)
            ob, _ = O.basic_decode(hm, tinv)
            od, odm = O.dark_original_decode(hm, tinv, ks)
            ours += [oc, om, ob, od, odm]
            if ref:
                rc, rm = ref.GaussTaylorKeyPointDecoder(ks)(hm.clone(), tinv)
                assert torch.equal(rc, oc) and torch.equal(rm, om), ("decode", w, h, ks, noise, seed)
                rb, _ = ref.BasicKeyPointDecoder()(hm.clone(), tinv)
                assert torch.equal(rb, ob), ("basic_decode", w, h, seed)
                rd, rdm = ref.DarkPoseOriginalKeyPointDecoder(ks)(hm.clone(), tinv)
                assert torch.equal(rd, od) and torch.equal(rdm, odm), ("dark_decode", w, h, ks, seed)
            counts["decode"] = counts.get("decode", 0) + 3
            # HeatMapAcc (17 joints in the reference's loop over channels: any K works)
            tgt = torch.from_numpy(O.encode_batch(synth.joints(2, num_joints=17, height=h, width=w, seed=seed + 1).numpy(), 2.0, (w, h))[0])
            pred = synth.predictions_like(tgt, seed=seed + 2, noise=float(rng.choice([0.05, 0.3, 1.0])))
            acc = float(O.heat_map_acc(pred, tgt))
            ours.append(acc)
            assert not ref or float(ref.HeatMapAcc()(pred, tgt)) == acc, ("acc", w, h, seed)
            counts["acc"] = counts.get("acc", 0) + 1
        # loss + grad
        b = int(rng.integers(1, 4))
        pred = torch.randn(b, k, h, w, generator=torch.Generator().manual_seed(seed))
        tgt = torch.rand(b, k, h, w, generator=torch.Generator().manual_seed(seed + 1))
        msk = torch.from_numpy(rng.choice([0.0, 1.0, 0.5, 2.0], size=(b, k)).astype(np.float32))
        p = pred.clone().requires_grad_(True)
        rl = 0.5 * torch.nn.MSELoss()(p.mul(msk[[..., None, None]]), tgt.mul(msk[[..., None, None]]))
        rl.backward()
        ol, og = O.masked_mse_loss_and_grad(pred, tgt, msk)
        ours += [ol, og]
        assert torch.equal(ol, rl.detach()) and torch.equal(og, p.grad), ("loss", b, k, h, w, seed)
        counts["loss"] = counts.get("loss", 0) + 1
        # OKS / NMS (17 joints: the reference's default sigmas), with and without the visibility threshold
        kps, box, area, seg = synth.nms_groups(3, mean_group=float(rng.choice([2.0, 8.0, 14.0])), seed=seed % 100000)
        kps, box, area, seg = kps.numpy(), box.numpy(), area.numpy(), seg.numpy()
        for s in range(3):
            lo, hi = seg[s], seg[s + 1]
            thr = float(rng.choice([0.5, 0.8, 0.9, 0.95]))
            vis = None if rng.uniform() < 0.5 else float(rng.choice([0.1, 0.3, 0.6]))
            o = O.oks_greedy_nms(kps[lo:hi], box[lo:hi], area[lo:hi], thr, in_vis_thresh=vis)
            c = O.oks_similarity(kps[lo], kps[lo:hi], area[lo], area[lo:hi], in_vis_thresh=vis)
            ours += [[int(i) for i in o], c]
            if ref:
                r = ref.oks_nms(kps[lo:hi], box[lo:hi], area[lo:hi], thr, in_vis_thresh=vis)
                assert [int(i) for i in r] == [int(i) for i in o], ("nms", thr, vis, seed)
                a = ref.oks_iou(kps[lo], kps[lo:hi], area[lo], area[lo:hi], in_vis_thresh=vis)
                assert np.array_equal(bits(a), bits(c)), ("oks", vis, seed)
        counts["oks_nms"] = counts.get("oks_nms", 0) + 3
        # box -> affine and the train-side transform
        inp = (int(rng.integers(8, 100)) * 4, int(rng.integers(8, 100)) * 4)
        outp = (inp[0] // 4, inp[1] // 4)
        smp = synth.train_samples(4, seed=seed % 1000003)
        for i in range(4):
            box4, iw = smp["boxes"][i].tolist(), int(smp["img_w"][i])
            rot = float(rng.choice([0.0, float(smp["rot"][i]), 90.0, -179.5, 1e-7]))
            draws = (float(smp["scale_ratio"][i]), rot, bool(smp["flip"][i]))
            basic = bool(rng.uniform() < 0.3)
            o = O.train_sample_geometry(box4, iw, smp["joints"][i].numpy(), *draws, input_shape=inp, output_shape=outp, basic=basic)
            ours += [o["trans_inv"], o["joints_input"], o["heat_map"], o["mask"]]
            if not ref:
                continue
            kp = ref_loader.run_train_transform(ref, box4, iw, 480, smp["joints"][i].numpy(), *draws, O.COCO_JOINT_PAIRS, inp, outp, basic=basic)
            assert np.array_equal(bits(kp.trans_inv), bits(o["trans_inv"])), ("train trans_inv", inp, draws, seed)
            assert np.array_equal(bits(kp.joints), bits(o["joints_input"])), ("train joints", inp, draws, seed)
            assert np.array_equal(bits(kp.heat_map), bits(o["heat_map"])) and np.array_equal(kp.mask, o["mask"]), ("train map", inp, draws, basic, seed)
        counts["train_geometry"] = counts.get("train_geometry", 0) + 4
        digests.append(pins.digest(ours))
    return it, counts, digests


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=120.0)
    ap.add_argument("--rounds", type=int, default=None, help="a fixed number of rounds instead of a time bound")
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    warnings.filterwarnings("ignore")
    t0 = time.time()
    it, counts, _ = run(ref_loader.load(), args.seed, rounds=args.rounds, seconds=args.seconds)
    print("fuzz ok: %d rounds in %.0f s;" % (it, time.time() - t0), ", ".join("%s %d" % kv for kv in sorted(counts.items())))
    return 0


if __name__ == "__main__":
    sys.exit(main())
