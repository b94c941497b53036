"""GPU: the COCO keypoint evaluator (csrc/sp_coco_eval.cu through metrics/coco_eval.py) against the COCOeval oracle:
OKS to 1e-14 relative, matched / ignored flags identical, precision, recall and stats bit for bit -- on the known
answers of test_coco_eval_cpu.py, on seeded synthetic sets up to COCO-val size, and at the end of the eval job."""
import numpy as np
import pytest
import torch

from oracle import coco_eval_oracle as C
from simple_pose_b200 import synth
from simple_pose_b200.metrics import coco_eval as CE
import test_coco_eval_cpu as K

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def run_device(ds, res, **kw):
    gt = CE.CocoKeypointGT(ds, device=DEV, **kw)
    kps, sc, ids = synth.coco_results_arrays(res)
    return gt, CE.evaluate(gt, kps.to(DEV), sc.to(DEV), ids, diagnostics=True)


def assert_matches_oracle(ds, res, img_ids=None):
    gt, got = run_device(ds, res, img_ids=img_ids)
    want = C.coco_eval_kps(ds, res, img_ids=img_ids)
    seg = gt.seg.cpu().numpy()
    oks = got.oks.cpu().numpy()
    flags = got.det_flags.cpu().numpy().view(np.uint64)
    n_img = len(want["img_ids"])
    assert list(gt.img_ids) == want["img_ids"]
    for i, img in enumerate(want["img_ids"]):
        ious = want["ious"][img]
        g0, G = int(seg[i]), int(seg[i + 1] - seg[i])
        if len(ious):
            D = ious.shape[0]
            dev = oks[20 * g0:20 * g0 + D * G].reshape(D, G)
            assert np.all(np.abs(dev - ious) <= 1e-14 * np.abs(ious)), (img, np.abs(dev - ious).max())
        for a in range(3):
            e = want["eval_imgs"][a * n_img + i]
            if e is None:
                continue
            D = len(e["dtScores"])
            for t in range(10):
                bit = np.uint64(a * 10 + t)
                m = ((flags[i * 20:i * 20 + D] >> bit) & np.uint64(1)).astype(bool)
                ig = ((flags[i * 20:i * 20 + D] >> (bit + np.uint64(32))) & np.uint64(1)).astype(bool)
                assert np.array_equal(m, e["dtMatches"][t] != 0), (img, a, t)
                assert np.array_equal(ig, e["dtIgnore"][t].astype(bool)), (img, a, t)
    assert np.array_equal(got.precision.cpu().numpy(), want["precision"])
    assert np.array_equal(got.recall.cpu().numpy(), want["recall"])
    assert np.array_equal(got.stats.cpu().numpy(), want["stats"]), (got.stats.cpu().numpy(), want["stats"])
    return got, want


def known_cases():
    g, d, p, ds = K.gt_ann, K.det, K.person, K.dataset
    xy, far = p(seed=7), p(seed=7) + 300.0
    xy2 = p(seed=8)
    gts4 = [p(seed=20 + i, x0=100.0 * i) for i in range(4)]
    fp32 = np.stack([np.array([400.0, 432.0] + [410.0] * 15), np.array([300.0, 332.0] + [310.0] * 15)], 1)
    box = (10.0, 20.0, 40.0, 80.0)
    return {
        "perfect": (ds([5, 9], [g(1, 5, p(seed=1), area=2000.0), g(2, 9, p(300, 50, 150, 200, seed=2), area=20000.0)]),
                    [d(9, p(300, 50, 150, 200, seed=2), 0.4), d(5, p(seed=1), 0.9)]),
        "between_thresholds": (ds([1], [g(1, 1, p(seed=3), area=5000.0)]),
                               [d(1, p(seed=3) + np.stack([np.sqrt(2 * 0.3285 * K.VARS * 5000.0), np.zeros(17)], 1), 0.5)]),
        "crowd_zero_kp": (ds([1, 2, 3], [g(1, 1, p(seed=5), iscrowd=1), g(2, 2, None, bbox=(10.0, 10.0, 40.0, 80.0)), g(3, 3, p(seed=4))]),
                          [d(1, p(seed=5), 0.9), d(1, p(seed=5) + 0.5, 0.9), d(2, np.stack([np.full(17, 20.0), np.full(17, 50.0)], 1), 0.8),
                           d(3, p(seed=4), 0.1)]),
        "box_distance": (ds([1, 2], [g(1, 1, None, area=3000.0, bbox=box), g(2, 2, p(seed=12))]),
                         [d(1, np.stack([np.full(17, 97.0), np.linspace(20, 100, 17)], 1), 0.5),
                          d(1, np.stack([np.full(17, -37.0), np.full(17, -67.0)], 1), 0.6), d(2, p(seed=12) + 2.0, 0.4)]),
        "truncation": (ds([1], [g(1, 1, xy)]), [d(1, far, 0.9 - 0.01 * i) for i in range(19)] + [d(1, xy, 0.05)] + [d(1, far, 0.01)] * 3),
        "truncated_away": (ds([1], [g(1, 1, xy)]), [d(1, far, 0.9 - 0.01 * i) for i in range(20)] + [d(1, xy, 0.05)]),
        "ties_within": (ds([1], [g(1, 1, xy)]), [d(1, far, 0.5), d(1, xy, 0.5)]),
        "ties_across": (ds([2, 1], [g(1, 1, xy), g(2, 2, xy2)]), [d(2, xy2, 0.0), d(1, far, 0.0)]),
        "area_bounds": (ds([1], [g(1, 1, p(seed=9), area=96.0 ** 2)]), [d(1, fp32, 0.9), d(1, p(seed=9), 0.5)]),
        "npig_zero": (ds([1, 2], [g(1, 1, None), g(2, 2, p(seed=10), iscrowd=1)]), [d(1, p(seed=11), 0.3), d(2, p(seed=10), 0.7)]),
        "recall_on_threshold": (ds([1], [g(i + 1, 1, q) for i, q in enumerate(gts4)]),
                                [d(1, gts4[0], 0.9), d(1, gts4[1], 0.8), d(1, gts4[0] + 1000.0, 0.7), d(1, gts4[2], 0.6)]),
        "no_detections": (ds([1, 2], [g(1, 1, xy)]), []),
    }


@pytest.mark.parametrize("case", sorted(known_cases()))
def test_known_answers_match_oracle(case):
    ds, res = known_cases()[case]
    assert_matches_oracle(ds, res)


@pytest.mark.parametrize("variant,seed,images", [("all", 11, 300), ("medium", 12, 200), ("large", 13, 200), ("all", 14, 5000)])
def test_synthetic_sets_match_oracle(variant, seed, images):
    ds, res = synth.coco_keypoint_set(images, seed=seed, variant=variant, fp=(0, 3) if images < 1000 else (4, 16))
    got, want = assert_matches_oracle(ds, res)
    if variant != "all":
        assert (want["stats"] == -1).sum() == 2


def test_narrowed_image_set_matches_oracle():
    ds, res = synth.coco_keypoint_set(120, seed=15)
    ids = sorted(i["id"] for i in ds["images"])[::3]
    assert_matches_oracle(ds, res, img_ids=ids)


def test_image_with_many_gts():
    """250 GTs in one image (plus a small one): the OKS matrix and the lanes' match rows live in the workspace."""
    rng = np.random.default_rng(5)
    anns, res = [], []
    for j in range(250):
        xy = K.person(x0=float(rng.uniform(0, 2000)), y0=float(rng.uniform(0, 2000)), seed=100 + j)
        zero = j % 5 == 0
        anns.append(K.gt_ann(j + 1, 1, None if zero else xy, area=float(rng.uniform(500, 20000)),
                             bbox=(float(xy[0, 0]), float(xy[0, 1]), 50.0, 100.0), iscrowd=int(j % 17 == 0)))
        if j % 9 == 0:
            res.append(K.det(1, xy + rng.normal(0, 2, (17, 2)), float(rng.integers(0, 10)) / 10))
    anns.append(K.gt_ann(999, 2, K.person(seed=3)))
    res.append(K.det(2, K.person(seed=3), 0.3))
    assert_matches_oracle(K.dataset([1, 2], anns), res)


def test_eval_job_end_to_end_table():
    """EvalSet -> ShardedPoseEvaluator (one rank) -> evaluate_table; the oracle reads the copied-back table as
    eval.py lists it: per image, the kept persons in NMS pick order (score descending, ties higher index first)."""
    from simple_pose_b200 import eval_shard
    es = synth.EvalSet(persons=3000, mean_group=7.0, seed=51)
    n = es.persons
    ev = eval_shard.ShardedPoseEvaluator()
    ev.plan(es.seg)
    rows = ev.run(es.heatmaps(0, n, DEV), None, es.box_scores, None, boxes=es.boxes.to(DEV))
    kps = eval_shard.row_keypoints(rows).cpu().numpy()
    keep = eval_shard.row_keep(rows).cpu().numpy()
    scores = eval_shard.row_scores(rows).cpu().numpy()
    ds, img_ids = synth.eval_set_ground_truth(es, kps, seed=52)
    gt = CE.CocoKeypointGT(ds, device=DEV)
    got = CE.evaluate_table(gt, rows, es.seg, img_ids)
    results = []
    for i in range(es.images):
        lo, hi = int(es.seg[i]), int(es.seg[i + 1])
        kept = [q for q in range(lo, hi) if keep[q]]
        for q in sorted(kept, key=lambda q: (-scores[q], -q)):
            results.append({"image_id": int(img_ids[i]), "category_id": 1, "score": float(scores[q]),
                            "keypoints": kps[q].reshape(-1).astype(np.float64).tolist()})
    want = C.coco_eval_kps(ds, results)
    assert np.array_equal(got.stats.cpu().numpy(), want["stats"])
    assert np.array_equal(got.precision.cpu().numpy(), want["precision"])
    assert want["stats"][0] > 0


def test_kps_to_dict_rows_path():
    """person_rows (the kps_to_dict_ table) in loader order, score = float32 last column widened."""
    from simple_pose_b200.metrics import pose_metrics as PM
    es = synth.EvalSet(persons=1200, mean_group=5.0, seed=61)
    n = es.persons
    tinv, _ = synth.inverse_affines(n, seed=62)
    xy, conf = PM.GaussTaylorKeyPointDecoder()(es.heatmaps(0, n, DEV), tinv.to(DEV))
    rows = PM.person_rows(xy, conf)
    per_person = np.repeat(np.arange(1, es.images + 1), np.diff(es.seg))
    kps3 = rows[:, :-1].reshape(n, 17, 3).cpu().numpy()
    ds, _ = synth.eval_set_ground_truth(es, kps3, seed=63, jitter=1.0)
    listed = []
    PM.kps_to_dict_(xy, conf, per_person.tolist(), listed)
    want = C.coco_eval_kps(ds, listed)
    got = CE.evaluate_person_rows(CE.CocoKeypointGT(ds, device=DEV), rows, per_person)
    assert np.array_equal(got.stats.cpu().numpy(), want["stats"])
    assert np.array_equal(got.recall.cpu().numpy(), want["recall"])


def test_workspace_reuse_gives_identical_results():
    a = synth.coco_keypoint_set(300, seed=21)
    b = synth.coco_keypoint_set(100, seed=22, variant="large")
    first = run_device(*a)[1]
    again = [run_device(*x)[1] for x in (a, b, a, a)]          # the call on b reuses, and rewrites, the workspace
    for r in (again[0], again[2], again[3]):
        assert torch.equal(r.stats, first.stats) and torch.equal(r.precision, first.precision)
        assert torch.equal(r.oks.nan_to_num(-7.0), first.oks.nan_to_num(-7.0)) and torch.equal(r.det_flags, first.det_flags)
    assert not torch.equal(again[1].stats, first.stats)
    assert np.array_equal(again[1].stats.cpu().numpy(), C.coco_eval_kps(*b)["stats"])


def test_argument_errors_and_cpu_refusal():
    ds, res = synth.coco_keypoint_set(20, seed=31)
    gt = CE.CocoKeypointGT(ds, device=DEV)
    kps, sc, ids = synth.coco_results_arrays(res)
    with pytest.raises(RuntimeError, match="no CPU path"):
        CE.evaluate(gt, kps, sc, ids)
    with pytest.raises(ValueError):
        CE.evaluate(gt, kps.to(DEV), sc[:-1].to(DEV), ids)
    with pytest.raises(ValueError):
        CE.evaluate(gt, kps[:, :50].to(DEV), sc.to(DEV), ids)
    bad_ids = ids.clone()
    bad_ids[3] = 10 ** 9
    with pytest.raises(ValueError):
        CE.evaluate(gt, kps.to(DEV), sc.to(DEV), bad_ids)
    with pytest.raises(ValueError):
        CE.evaluate(gt, kps.to(DEV), sc.to(DEV), bad_ids.to(DEV))
    ok = CE.evaluate(gt, kps.to(DEV), sc.to(DEV), ids.to(DEV))          # ids as a CUDA tensor
    assert np.array_equal(ok.stats.cpu().numpy(), C.coco_eval_kps(ds, res)["stats"])
    with pytest.raises(RuntimeError, match="no CPU path"):
        CE.evaluate_person_rows(gt, torch.zeros(3, 52), [1, 1, 1])
    from simple_pose_b200 import _abi
    lib = _abi.lib()
    n = kps.shape[0]
    need = lib.sp_coco_eval_workspace_bytes(n, gt.num_images, gt.num_gts)
    assert need > 0
    out = torch.empty(10 * 101 * 3 + 30 + 10, dtype=torch.float64, device=DEV)
    ws = torch.zeros(need // 8 + 2, dtype=torch.int64, device=DEV)
    k, s, p = kps.to(DEV), sc.to(DEV), gt.positions(ids)
    args = [k.data_ptr(), 51, s.data_ptr(), p.data_ptr(), None, n, gt.kps.data_ptr(), gt.area.data_ptr(), gt.bbox.data_ptr(),
            gt.flags.data_ptr(), gt.seg.data_ptr(), gt.num_images, gt.num_gts, gt.iou_thrs.data_ptr(), gt.rec_thrs.data_ptr(),
            gt.area_rng.data_ptr(), 17, 10, 101, 3, 20, out.data_ptr(), out.data_ptr() + 8 * 3030, out.data_ptr() + 8 * 3060,
            None, None, None, ws.data_ptr(), need - 16, _abi.stream_ptr(DEV)]
    assert lib.sp_coco_eval_kps_f32(*args) == -3                                 # workspace too small
    assert lib.sp_coco_eval_kps_f32(*(args[:28] + [need] + args[29:])) == 0
    torch.cuda.synchronize()
    assert torch.equal(out[3060:], ok.stats)
