"""CPU: pins the oracle restatement against the unmodified reference (liangheming/simple_pose).

Where the reference tree is mounted (``oracle/ref_loader.py``, ``SIMPLE_POSE_REFERENCE``) every test runs the
reference's own functions on its inputs and demands bit equality with the oracle. Everywhere else each test checks the
oracle's values against ``tests/golden/reference_pins.json`` (``oracle/pins.py``): per test, one digest per item (person,
segment, round, ...) of exactly the values that are compared with the reference. Where the tree is mounted both checks
run, so a wrong record fails there too.

The record was taken from the oracle as of the commit that added it, without the reference tree: it holds what the
oracle computed while it was pinned bit-identical to the reference by this module and by ``oracle/fuzz_vs_reference.py``
(DESIGN.md section 2). ``SP_RECORD_REFERENCE_PINS=1`` rewrites entries, and only with the reference mounted, after the
test's live comparisons have passed; ``SP_RECORD_REFERENCE_PINS=missing`` adds entries for tests that have none, from the
oracle, and never changes an existing one."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import heatmap_oracle as O
from oracle import pins as P
from oracle import ref_loader
from simple_pose_b200 import synth
from conftest import GOLDEN, bits

PINS = os.path.join(GOLDEN, "reference_pins.json")
FUZZ_ROUNDS = 120


@pytest.fixture(scope="module")
def ref():
    """The reference's callables, or None where its tree is not mounted."""
    return ref_loader.load() if ref_loader.available() else None


@pytest.fixture(scope="module")
def _pins():
    mode = os.environ.get("SP_RECORD_REFERENCE_PINS", "")
    if mode not in ("", "1", "missing"):
        raise pytest.UsageError("SP_RECORD_REFERENCE_PINS must be 1 or missing")
    if mode == "1" and not ref_loader.available():
        raise pytest.UsageError("SP_RECORD_REFERENCE_PINS=1 records the reference's values: mount the reference tree")
    with open(PINS) as fh:
        table = json.load(fh)
    state = {"table": table, "mode": mode, "changed": False}
    yield state
    if state["changed"]:
        with open(PINS, "w") as fh:
            json.dump(table, fh, indent=1, sort_keys=True)
            fh.write("\n")


@pytest.fixture
def pin(_pins, request):
    """pin(values), called once the test's live comparisons (if any) have passed: the oracle's values that the test
    compares with the reference must reproduce the recorded digests, item by item."""
    def check(values):
        table, key, got = _pins["table"], request.node.name, P.item_digests(values)
        if _pins["mode"] == "1" or (_pins["mode"] == "missing" and key not in table):
            table[key], _pins["changed"] = got, True
            return
        assert key in table, "no recorded reference values for %s" % key
        bad = P.mismatch(table[key], got)
        assert bad is None, "%s: the oracle no longer reproduces the reference's recorded values: %s" % (key, bad)
    return check


@pytest.mark.parametrize("shape", [(48, 64), (72, 96), (20, 12)])
def test_encode(ref, pin, shape):
    w, h = shape
    joints = synth.joints(24, height=h, width=w, seed=101).numpy()
    t, wt = O.encode_batch(joints, 2.0, shape)
    for b in range(joints.shape[0]) if ref else ():
        rt, rw = ref.get_heat_map(joints[b], 2.0, shape)
        assert np.array_equal(bits(rt), bits(t[b])) and np.array_equal(rw, wt[b])
    pin([[t[b], wt[b]] for b in range(joints.shape[0])])


@pytest.mark.parametrize("hw,noise", [((64, 48), 0.01), ((96, 72), 0.01), ((64, 48), 0.05), ((32, 24), 0.02)])
def test_decode(ref, pin, hw, noise):
    h, w = hw
    hm = synth.heatmaps(16, height=h, width=w, seed=202, noise=noise)
    tinv = synth.inverse_affines(16, height=h, width=w, seed=202)[0]
    oc, om = O.gauss_taylor_decode(hm, tinv)
    ob, _ = O.basic_decode(hm, tinv)
    if ref:
        rc, rm = ref.GaussTaylorKeyPointDecoder()(hm.clone(), tinv)
        assert torch.equal(rc, oc) and torch.equal(rm, om)
        rb, _ = ref.BasicKeyPointDecoder()(hm.clone(), tinv)
        assert torch.equal(rb, ob)
    pin([[oc[i], om[i], ob[i]] for i in range(hm.shape[0])])


def test_decode_does_not_mutate_input():
    hm = synth.heatmaps(2, seed=5)
    keep = hm.clone()
    O.gauss_taylor_decode(hm, synth.identity_affines(2))
    assert torch.equal(hm, keep)


def test_loss():
    """The solvers' loss expression (``0.5 * MSELoss`` on masked maps) under autograd, restated."""
    tgt = torch.from_numpy(O.encode_batch(synth.joints(8, seed=7).numpy())[0])
    msk = torch.from_numpy(O.encode_batch(synth.joints(8, seed=7).numpy())[1])
    pred = synth.predictions_like(tgt, seed=8)
    p = pred.clone().requires_grad_(True)
    ref_loss = 0.5 * torch.nn.MSELoss()(p.mul(msk[[..., None, None]]), tgt.mul(msk[[..., None, None]]))
    ref_loss.backward()
    loss, grad = O.masked_mse_loss_and_grad(pred, tgt, msk)
    assert torch.equal(loss, ref_loss.detach()) and torch.equal(grad, p.grad)


def test_oks_and_nms(ref, pin):
    kps, box, area, seg = synth.nms_groups(40, seed=9)
    kps, box, area, seg = kps.numpy(), box.numpy(), area.numpy(), seg.numpy()
    ours = []
    for s in range(40):
        lo, hi = seg[s], seg[s + 1]
        o = O.oks_greedy_nms(kps[lo:hi], box[lo:hi], area[lo:hi], 0.9)
        b = O.oks_similarity(kps[lo], kps[lo:hi], area[lo], area[lo:hi])
        ours.append([[int(i) for i in o], b])
        if ref:
            r = ref.oks_nms(kps[lo:hi], box[lo:hi], area[lo:hi], 0.9)
            assert [int(i) for i in r] == [int(i) for i in o]
            a = ref.oks_iou(kps[lo], kps[lo:hi], area[lo], area[lo:hi])
            assert np.array_equal(bits(a), bits(b))
    pin(ours)


def test_nms_score_ties_are_the_only_freedom(ref, pin):
    """`oks_nms` visits `scores.argsort()[::-1]` (datasets/naive_data.py:163). With distinct scores that order
    is unique and the restatement equals the reference for every image size. With EQUAL scores NumPy's default
    sort decides, and its tie order depends on the SIMD sort it dispatches to on the host CPU (AVX-512 / AVX2
    builds reorder ties even below 16 elements), so the reference's keep list is then a property of the
    machine. Pinned here: (1) distinct scores: exact; (2) ties made explicit by `detie_scores` (higher index
    first -- the rule the CUDA kernel implements): the reference itself, fed the de-tied scores, returns the
    same keep list as the restatement; (3) with the reference's own visiting order injected the greedy pass is
    reproduced exactly, i.e. nothing but the order of equal scores differs."""
    rng = np.random.RandomState(0)
    order_differs = keep_differs = cases = 0
    ours = []
    for trial in range(120):
        n = int(rng.choice([4, 8, 12, 17, 20, 33, 60]))
        kps, _, area, _ = synth.nms_groups(1, mean_group=float(n), seed=trial)
        kps, area = kps.numpy(), area.numpy()
        m = kps.shape[0]
        distinct = rng.permutation(m) / m
        keep_distinct = [int(i) for i in O.oks_greedy_nms(kps, distinct, area, 0.9)]
        tied = rng.choice([0.3, 0.5, 0.7, 0.9], size=m)
        detied = O.detie_scores(tied)
        assert np.array_equal(np.argsort(detied)[::-1], np.argsort(tied, kind="stable")[::-1])
        want = [int(i) for i in O.oks_greedy_nms(kps, detied, area, 0.9)]
        ours.append([keep_distinct, want])
        if not ref:
            continue
        assert [int(i) for i in ref.oks_nms(kps, distinct, area, 0.9)] == keep_distinct
        assert [int(i) for i in ref.oks_nms(kps, detied, area, 0.9)] == want
        got = [int(i) for i in ref.oks_nms(kps, tied, area, 0.9)]
        cases += 1
        order_differs += int(not np.array_equal(tied.argsort()[::-1], np.argsort(tied, kind="stable")[::-1]))
        keep_differs += int(sorted(got) != sorted(want))
    pin(ours)
    # informational: how often this host's NumPy breaks ties differently from the stable rule
    print("tied-score images: %d, visiting order differs in %d, keep set differs in %d" % (cases, order_differs, keep_differs))


def test_heat_map_acc(ref, pin):
    tgt = torch.from_numpy(O.encode_batch(synth.joints(8, seed=17).numpy())[0])
    pred = synth.predictions_like(tgt, seed=18, noise=0.3)
    acc = float(O.heat_map_acc(pred, tgt))
    assert not ref or float(ref.HeatMapAcc()(pred, tgt)) == acc
    pin(acc)


@pytest.mark.parametrize("inp,outp", [((192, 256), (48, 64)), ((288, 384), (72, 96)), ((256, 256), (64, 64))])
def test_box_affines(ref, pin, inp, outp):
    """box_to_center_scale + get_affine_transform(rot=0) (the body of BasicTransform.__call__): the
    oracle's restatement of OpenCV's 6x6 LU is bit-identical to cv2, both directions."""
    boxes = synth.detection_boxes(400, seed=77, ratio_exact_every=16, ratio=inp[0] / inp[1]).tolist()
    boxes += [[10.0, 20.0, 10.001, 20.002], [-1.5, 7.0, -0.5, 9.0], [100.0, 50.0, 100.0, 50.0], [0.0, 0.0, 1e6, 3.0]]
    c, s, a, tinv = O.box_affines(boxes, inp, outp)
    ours = []
    for i, (x1, y1, x2, y2) in enumerate(boxes):
        oc, os_ = O.box_center_scale(x1, y1, x2 - x1, y2 - y1, inp[0] / inp[1])
        ot, oti = O.affine_pair(oc, os_, outp)
        ours.append([oc, os_, ot, oti])
        # the batched restatement agrees with the per-box one
        assert np.array_equal(bits(c[i]), bits(oc)) and np.array_equal(bits(s[i]), bits(os_)), i
        assert np.float32(os_[0] * os_[1]) == a[i]
        assert np.array_equal(bits(tinv[i]), bits(torch.from_numpy(oti).float().numpy())), i
        if ref:
            rc, rs = ref.box_to_center_scale(x1, y1, x2 - x1, y2 - y1, inp[0] / inp[1])
            rt, rti = ref.get_affine_transform(rc, rs, 0, outp)
            assert oc.dtype == rc.dtype and os_.dtype == rs.dtype
            assert np.array_equal(bits(rc), bits(oc)) and np.array_equal(bits(rs), bits(os_)), i
            assert np.array_equal(bits(rt), bits(ot)) and np.array_equal(bits(rti), bits(oti)), i
    pin(ours)


@pytest.mark.parametrize("inp,outp", [((192, 256), (48, 64)), ((288, 384), (72, 96))])
def test_train_geometry(ref, pin, inp, outp):
    """RefineSimpleTransform.__call__ itself (commons/transforms.py:193-223), random draws scripted,
    against the oracle's restatement of its joint/affine/target half: bit equality."""
    smp = synth.train_samples(120, seed=303)
    ours = []
    for i in range(120):
        args = (smp["boxes"][i].tolist(), int(smp["img_w"][i]))
        draws = (float(smp["scale_ratio"][i]), float(smp["rot"][i]), bool(smp["flip"][i]))
        o = O.train_sample_geometry(args[0], args[1], smp["joints"][i].numpy(), *draws, input_shape=inp, output_shape=outp)
        flipped = O.flip_joints_only(smp["joints"][i].numpy(), args[1])
        moved = O.affine_joints(smp["joints"][i].numpy(), o["joint_trans"])
        ours.append([o["trans_inv"], o["joints_input"], o["heat_map"], o["mask"], o["joint_trans"], flipped, moved])
        if not ref:
            continue
        kp = ref_loader.run_train_transform(ref, args[0], args[1], 480, smp["joints"][i].numpy(), *draws,
                                            O.COCO_JOINT_PAIRS, inp, outp)
        assert np.array_equal(bits(kp.trans_inv), bits(o["trans_inv"])), i
        assert np.array_equal(bits(kp.joints), bits(o["joints_input"])), i
        assert np.array_equal(bits(kp.heat_map), bits(o["heat_map"])) and np.array_equal(kp.mask, o["mask"]), i
        rt, rti = ref.get_affine_transform(o["center"], o["scale"], draws[1], outp)
        assert np.array_equal(bits(rt), bits(o["joint_trans"])) and np.array_equal(bits(rti), bits(o["trans_inv"]))
        fj = ref.flip_joints(np.zeros((4, args[1], 3), np.uint8), smp["joints"][i].numpy(), [list(p) for p in O.COCO_JOINT_PAIRS])[1]
        assert np.array_equal(bits(fj), bits(flipped))
        aj = ref.joint_utils.affine_transform_batch(smp["joints"][i].numpy(), rt)
        assert np.array_equal(bits(aj), bits(moved))
    pin(ours)


def test_dark_original_decoder(ref, pin):
    """DarkPoseOriginalKeyPointDecoder itself (on a clone: it overwrites its input) vs the restatement."""
    import warnings
    ours = []
    for hw, seed in (((64, 48), 31), ((96, 72), 32), ((40, 36), 33)):
        h, w = hw
        hm = synth.heatmaps(6, height=h, width=w, seed=seed, noise=0.02)
        tinv = synth.inverse_affines(6, height=h, width=w, seed=seed)[0]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            oc, om = O.dark_original_decode(hm, tinv)
            ours.append([oc, om])
            if ref:
                rc, rm = ref.DarkPoseOriginalKeyPointDecoder()(hm.clone(), tinv)
                assert rc.dtype == oc.dtype and torch.equal(rc, oc) and torch.equal(rm, om)
    pin(ours)


def test_train_geometry_basic_transform(ref, pin):
    """BasicSimpleTransform.__call__ (commons/transforms.py:118-148), draws scripted: the quantised encoder
    runs on the input-pixel joints; trans_inv and targets bit-identical."""
    smp = synth.train_samples(60, seed=304)
    ours = []
    for i in range(60):
        box, w = smp["boxes"][i].tolist(), int(smp["img_w"][i])
        draws = (float(smp["scale_ratio"][i]), float(smp["rot"][i]), bool(smp["flip"][i]))
        o = O.train_sample_geometry(box, w, smp["joints"][i].numpy(), *draws, basic=True)
        ours.append([o["trans_inv"], o["joints_input"], o["heat_map"], o["mask"]])
        if not ref:
            continue
        kp = ref_loader.run_train_transform(ref, box, w, 480, smp["joints"][i].numpy(), *draws, O.COCO_JOINT_PAIRS, basic=True)
        assert np.array_equal(bits(kp.trans_inv), bits(o["trans_inv"])) and np.array_equal(bits(kp.joints), bits(o["joints_input"]))
        assert np.array_equal(bits(kp.heat_map), bits(o["heat_map"])) and np.array_equal(kp.mask, o["mask"]), i
    pin(ours)


def test_randomised_pin_short(ref, pin):
    """A short run of the randomised pin (oracle/fuzz_vs_reference.py: random shapes, sigmas, blur sizes
    3-13, Basic encoder, K != 17, masks, NMS thresholds, visibility thresholds, rotations incl. 90 / -179.5
    degrees), a fixed seed and round count: bit equality on every row with the reference mounted, the
    recorded per-round digests without it. The long form found the fixed OpenCV tables behind
    ``cv.getGaussianKernel(n <= 9, 0)``."""
    import warnings
    from oracle import fuzz_vs_reference
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        rounds, counts, digests = fuzz_vs_reference.run(ref, seed=7, rounds=FUZZ_ROUNDS)
    assert rounds == FUZZ_ROUNDS and all(counts.get(row, 0) > 0 for row in
                                         ("encode", "decode", "acc", "loss", "oks_nms", "train_geometry")), counts
    pin(digests)


@pytest.mark.parametrize("vis,thr", [(0.2, 0.9), (0.5, 0.8), (0.05, 0.95)])
def test_eval_rescoring_and_nms_through_the_reference_function(ref, pin, vis, thr):
    """A9: the reference's own temp_read_in_and_filter (eval.py:153-197, JSON in / JSON out, COCO evaluation
    stubbed) against the restatement's rescore_and_nms: kept persons, their order, scores and keypoints."""
    kps, box, area, seg = synth.nms_groups(25, mean_group=9.0, seed=int(vis * 100))
    kps, box, area, seg = kps.numpy(), box.numpy(), area.numpy(), seg.numpy()
    img_ids = np.repeat(np.arange(25) * 7 + 3, np.diff(seg))
    keep, scores, picks = O.rescore_and_nms(kps, box, area, seg, vis, thr)
    flat = [i for p in picks for i in p]
    ours = [{"image_id": int(img_ids[i]), "category_id": 1, "score": float(scores[i]), "keypoints": kps[i].reshape(-1).tolist()}
            for i in flat]
    assert len(flat) == int(keep.sum())
    if ref:
        out = ref_loader.run_eval_filter(kps, box, area, img_ids, vis, thr)
        assert len(out) == len(flat)
        for rec, i in zip(out, flat):
            assert rec["image_id"] == int(img_ids[i]) and rec["category_id"] == 1
            assert rec["score"] == scores[i]
            assert rec["keypoints"] == kps[i].reshape(-1).tolist()
    pin(ours)


def test_kps_to_dict_host_formatting(ref, pin):
    """A10: the restatement of the reference's per-person loop (metrics/pose_metrics.py:172-179) on host
    tensors: identical lists of dicts. (The product's kernel is compared with it under -m gpu.)"""
    from oracle import heatmap_oracle as O
    g = torch.Generator().manual_seed(0)
    ours = []
    for _ in range(50):
        n = 9
        pred = torch.randn(n, 17, 2, generator=g) * 100
        sc = torch.rand(n, 17, 1, generator=g)
        b = []
        O.kps_to_dict(pred, sc, list(range(100, 100 + n)), b)
        ours.append(b)
        if ref:
            a = []
            ref.kps_to_dict_(pred, sc, list(range(100, 100 + n)), a)
            assert a == b
    pin(ours)
