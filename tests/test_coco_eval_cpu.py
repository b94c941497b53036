"""CPU: the COCOeval oracle (oracle/coco_eval_oracle.py) on known answers worked out here from COCOeval's rules,
the GT parser of the device evaluator, the C ABI's argument checks, and -- where pycocotools can be imported --
the oracle against pycocotools itself on the synthetic sets."""
import math

import numpy as np
import pytest

from oracle import coco_eval_oracle as C
from simple_pose_b200 import synth

SIGMAS = np.array([.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89]) / 10.0
VARS = (SIGMAS * 2) ** 2
REC = np.linspace(.0, 1.00, 101, endpoint=True)
P1 = 1.0 / (0.0 + 1.0 + np.spacing(1))          # precision of a lone true positive: tp / (fp + tp + eps)


def gt_ann(ann_id, img, xy=None, area=5000.0, bbox=(100.0, 100.0, 50.0, 100.0), iscrowd=0, vis=None):
    """A person annotation; ``xy`` [17, 2] labelled joints (None = no keypoints)."""
    if xy is None:
        kps, nk = [0] * 51, 0
    else:
        v = np.full(17, 2) if vis is None else np.asarray(vis)
        kps = np.stack([np.asarray(xy)[:, 0], np.asarray(xy)[:, 1], v], 1).reshape(-1).tolist()
        nk = int((v > 0).sum())
    return {"id": ann_id, "image_id": img, "category_id": 1, "iscrowd": iscrowd, "area": area, "bbox": list(bbox),
            "num_keypoints": nk, "keypoints": kps}


def det(img, xy, score):
    xy = np.asarray(xy, dtype=np.float32)
    return {"image_id": img, "category_id": 1, "score": score,
            "keypoints": np.stack([xy[:, 0], xy[:, 1], np.ones(17, np.float32)], 1).reshape(-1).astype(float).tolist()}


def person(x0=100.0, y0=100.0, w=50.0, h=100.0, seed=0):
    r = np.random.default_rng(seed)
    return np.round(np.stack([x0 + r.random(17) * w, y0 + r.random(17) * h], 1))


def dataset(img_ids, anns):
    return {"images": [{"id": i} for i in img_ids], "annotations": anns}


def closed_form_oks(dxy, area, vis=None):
    e = (dxy[:, 0] ** 2 + dxy[:, 1] ** 2) / VARS / (area + np.spacing(1)) / 2
    if vis is not None:
        e = e[vis > 0]
    return np.sum(np.exp(-e)) / e.shape[0]


def test_params_are_linspace_values():
    p = C.kp_params()
    assert p["iouThrs"].shape == (10,) and p["recThrs"].shape == (101,)
    assert np.array_equal(p["recThrs"], REC)
    assert np.count_nonzero(p["iouThrs"] == .5) == 1 and np.count_nonzero(p["iouThrs"] == .75) == 1


def test_perfect_detections_give_one():
    xy1, xy2 = person(seed=1), person(300, 50, 150, 200, seed=2)
    ds = dataset([5, 9], [gt_ann(1, 5, xy1, area=2000.0), gt_ann(2, 9, xy2, area=20000.0)])
    out = C.coco_eval_kps(ds, [det(9, xy2, 0.4), det(5, xy1, 0.9)])
    # all: pr = [1 / (1 + eps), 2 / (2 + eps) = 1]; medium / large: one true positive each, the other detection
    # is matched to the GT that the range ignores
    assert np.all(out["precision"][:, :, 0] == 1.0) and np.all(out["precision"][:, :, 1:] == P1)
    assert np.array_equal(out["recall"], np.ones((10, 3)))
    assert out["stats"][0] == 1.0 and np.allclose(out["stats"][3:5], P1, rtol=1e-15, atol=0)
    assert np.array_equal(out["stats"][5:], np.ones(5))
    assert out["ious"][5][0, 0] == 1.0


def test_single_detection_between_thresholds():
    """One GT, one detection whose OKS is exp(-c) with every joint at the same e = c: matched up to IoU 0.70."""
    area = 5000.0
    c = -math.log(0.72)
    off = np.sqrt(2 * c * VARS * area)
    xy = person(seed=3)
    dxy = np.stack([off, np.zeros(17)], 1)
    d = xy + dxy
    want = closed_form_oks(np.asarray(d, np.float32).astype(np.float64) - xy, area)
    assert 0.70 < want < 0.75
    out = C.coco_eval_kps(dataset([1], [gt_ann(1, 1, xy, area=area)]), [det(1, d, 0.5)])
    assert abs(out["ious"][1][0, 0] - want) <= 1e-15
    matched = C.kp_params()["iouThrs"] <= want
    assert matched.sum() == 5
    want_prec = np.where(matched[:, None], P1, 0.0) * np.ones((10, 101))
    assert np.array_equal(out["precision"][:, :, 0], want_prec) and np.array_equal(out["precision"][:, :, 1], want_prec)
    assert np.array_equal(out["precision"][:, :, 2], -np.ones((10, 101)))
    assert np.array_equal(out["recall"][:, 0], matched.astype(float))
    assert np.allclose(out["stats"], [P1 / 2, P1, 0.0, P1 / 2, -1, 0.5, 1.0, 0.0, 0.5, -1], rtol=1e-15, atol=0)


def test_crowd_and_zero_keypoint_gts_absorb_their_detections():
    """Detections matched to a crowd (several may be) or a zero-keypoint GT are ignored, not false positives."""
    xy = person(seed=4)
    crowd = gt_ann(1, 1, person(seed=5), iscrowd=1)
    zero = gt_ann(2, 2, None, bbox=(10.0, 10.0, 40.0, 80.0))
    normal = gt_ann(3, 3, xy)
    inside = np.stack([np.full(17, 20.0), np.full(17, 50.0)], 1)           # inside the (grown) box: OKS 1
    dts = [det(1, crowd_xy, 0.9) for crowd_xy in (person(seed=5), person(seed=5) + 0.5)]
    dts += [det(2, inside, 0.8), det(3, xy, 0.1)]
    out = C.coco_eval_kps(dataset([1, 2, 3], [crowd, zero, normal]), dts)
    assert out["ious"][2][0, 0] == 1.0
    e_crowd = out["eval_imgs"][0]
    assert np.all(e_crowd["dtIgnore"]) and np.all(e_crowd["dtMatches"] == 1)
    assert np.all(out["eval_imgs"][1]["dtIgnore"])
    assert out["stats"][5] == 1.0
    # without the ignore rule the crowd and zero-keypoint detections would be 3 false positives ranked first
    assert np.all(out["precision"][:, :, 0] == P1)


def test_box_distance_branch():
    """A GT without keypoints: distance to its box grown to [x-w, x+2w] x [y-h, y+2h]."""
    x, y, w, h, area = 10.0, 20.0, 40.0, 80.0, 3000.0
    delta = 7.0
    pts = np.stack([np.full(17, x + 2 * w + delta), np.linspace(y, y + h, 17)], 1)      # right of the grown box
    out = C.coco_eval_kps(dataset([1], [gt_ann(1, 1, None, area=area, bbox=(x, y, w, h))]), [det(1, pts, 0.5)])
    want = np.sum(np.exp(-(delta ** 2 / VARS / (area + np.spacing(1)) / 2))) / 17
    assert abs(out["ious"][1][0, 0] - want) <= 1e-15 * want
    pts2 = np.stack([np.full(17, x - w - delta), np.full(17, y - h - delta)], 1)       # above-left corner
    out2 = C.coco_eval_kps(dataset([1], [gt_ann(1, 1, None, area=area, bbox=(x, y, w, h))]), [det(1, pts2, 0.5)])
    want2 = np.sum(np.exp(-((2 * delta ** 2) / VARS / (area + np.spacing(1)) / 2))) / 17
    assert abs(out2["ious"][1][0, 0] - want2) <= 1e-15 * want2
    assert np.all(out2["stats"] == -1)                                   # the only GT is ignored: npig == 0


def test_truncation_at_twenty():
    xy = person(seed=6)
    far = xy + 300.0
    for rank, recalled in ((20, True), (21, False)):
        dts = [det(1, far, 0.9 - 0.01 * i) for i in range(rank - 1)] + [det(1, xy, 0.05)] + \
              [det(1, far, 0.01) for _ in range(3)]
        out = C.coco_eval_kps(dataset([1], [gt_ann(1, 1, xy)]), dts)
        assert out["ious"][1].shape == (20, 1)
        if recalled:
            assert np.all(out["recall"][:, 0] == 1.0)
            assert np.all(out["precision"][:, :, 0] == 1.0 / (19.0 + 1.0 + np.spacing(1)))
        else:
            assert np.all(out["recall"][:, 0] == 0.0) and np.all(out["precision"][:, :, 0] == 0.0)


def test_tie_order_within_and_across_images():
    xy = person(seed=7)
    far = xy + 300.0
    ds = dataset([1], [gt_ann(1, 1, xy)])
    first_good = C.coco_eval_kps(ds, [det(1, xy, 0.5), det(1, far, 0.5)])
    first_bad = C.coco_eval_kps(ds, [det(1, far, 0.5), det(1, xy, 0.5)])
    assert np.all(first_good["precision"][:, :, 0] == P1)               # [TP, FP]: precision 1 up to recall 1
    assert np.all(first_bad["precision"][:, :, 0] == 1.0 / (1.0 + 1.0 + np.spacing(1)))   # [FP, TP]: 1/2
    # across images equal scores are ordered by image id (params.imgIds), not by the results list
    xy2 = person(seed=8)
    ds2 = dataset([2, 1], [gt_ann(1, 1, xy), gt_ann(2, 2, xy2)])
    out = C.coco_eval_kps(ds2, [det(2, xy2, 0.0), det(1, far, 0.0)])
    want = np.where(REC <= 0.5, 1.0 / (1.0 + 1.0 + np.spacing(1)), 0.0)  # [FP (image 1), TP (image 2)]
    assert np.all(out["precision"][:, :, 0] == want[None, :])


def test_inclusive_area_bounds():
    xy = person(seed=9)
    fp = np.stack([np.array([400.0] + [432.0] + [410.0] * 15), np.array([300.0] + [332.0] + [310.0] * 15)], 1)
    ds = dataset([1], [gt_ann(1, 1, xy, area=96.0 ** 2)])
    out = C.coco_eval_kps(ds, [det(1, fp, 0.9), det(1, xy, 0.5)])
    dts = C.load_res([1], [det(1, fp, 0.9)])
    assert dts[0]["area"] == 32.0 ** 2
    # the GT (area 96^2) counts for medium and large; the false positive (area 32^2) only for all and medium
    half = 1.0 / (1.0 + 1.0 + np.spacing(1))
    assert np.all(out["precision"][:, :, 1] == half) and np.all(out["precision"][:, :, 2] == P1)
    assert np.all(out["precision"][:, :, 0] == half)
    assert out["stats"][8] == 1.0 and out["stats"][9] == 1.0


def test_npig_zero_gives_minus_one():
    ds = dataset([1, 2], [gt_ann(1, 1, None), gt_ann(2, 2, person(seed=10), iscrowd=1)])
    out = C.coco_eval_kps(ds, [det(1, person(seed=11), 0.3), det(2, person(seed=10), 0.7)])
    assert np.all(out["precision"] == -1) and np.all(out["recall"] == -1) and np.all(out["stats"] == -1)


def test_recall_landing_on_a_threshold():
    """npig = 4, detections TP TP FP TP: rc = .25, .5, .5, .75 -- recall thresholds equal to rc values take the
    first index with rc >= thr (searchsorted 'left')."""
    gts = [person(seed=20 + i, x0=100.0 * i) for i in range(4)]
    ds = dataset([1], [gt_ann(i + 1, 1, g) for i, g in enumerate(gts)])
    far = gts[0] + 1000.0
    out = C.coco_eval_kps(ds, [det(1, gts[0], 0.9), det(1, gts[1], 0.8), det(1, far, 0.7), det(1, gts[2], 0.6)])
    rc = np.array([1, 2, 2, 3]) / 4
    pr = np.array([1, 2, 2, 3]) / (np.array([1, 2, 3, 4]) + np.spacing(1))
    assert np.isin(rc, REC).all()
    mono = np.maximum.accumulate(pr[::-1])[::-1]
    want = np.zeros(101)
    for k, thr in enumerate(REC):
        idx = [i for i in range(4) if rc[i] >= thr]
        if idx:
            want[k] = mono[idx[0]]
    assert np.array_equal(out["precision"][0, :, 0], want)
    assert out["recall"][0, 0] == 0.75


def test_detection_on_unknown_image_is_an_error():
    with pytest.raises(AssertionError):
        C.coco_eval_kps(dataset([1], [gt_ann(1, 1, person())]), [det(2, person(), 0.5)])


def test_gt_parser_order_filter_and_errors():
    from simple_pose_b200.metrics.coco_eval import CocoKeypointGT
    xy = person()
    anns = [gt_ann(30, 9, xy), gt_ann(4, 2, xy), gt_ann(12, 9, None), gt_ann(8, 2, xy, iscrowd=1)]
    anns.insert(1, dict(gt_ann(99, 9, xy), category_id=2))
    ds = dataset([9, 2, 5], anns)
    gt = CocoKeypointGT(ds, device="cpu")
    assert list(gt.img_ids) == [2, 5, 9] and list(gt.ann_ids) == [4, 8, 30, 12]          # file order per image
    assert gt.seg.tolist() == [0, 2, 2, 4] and gt.flags.tolist() == [0, 3, 0, 1]
    assert gt.positions([9, 2, 5, 9]).tolist() == [2, 0, 1, 2]
    with pytest.raises(ValueError):
        gt.positions([9, 3])
    narrowed = CocoKeypointGT(ds, img_ids=[9], device="cpu")
    assert narrowed.positions([2, 9]).tolist() == [-1, 0] and narrowed.num_gts == 2
    bad = dataset([1], [{k: v for k, v in gt_ann(1, 1, xy).items() if k != "num_keypoints"}])
    with pytest.raises(KeyError):
        CocoKeypointGT(bad, device="cpu")
    with pytest.raises(ValueError):
        CocoKeypointGT(dataset([1], [gt_ann(0, 1, xy)]), device="cpu")


def test_summary_lines_format():
    from simple_pose_b200.metrics.coco_eval import CocoEvalResult
    import torch
    res = CocoEvalResult(None, None, torch.tensor([0.7123, 0.9, 0.8, 0.6, 0.75, 0.77, 0.93, 0.83, 0.71, -1.0], dtype=torch.float64))
    lines = res.summary()
    assert lines[0] == " Average Precision  (AP) @[ IoU=0.50:0.95 | area=   all | maxDets= 20 ] = 0.712"
    assert lines[2] == " Average Precision  (AP) @[ IoU=0.75      | area=   all | maxDets= 20 ] = 0.800"
    assert lines[9] == " Average Recall     (AR) @[ IoU=0.50:0.95 | area= large | maxDets= 20 ] = -1.000"


def test_synthetic_sets_cover_the_cases():
    ds, res = synth.coco_keypoint_set(120, seed=5)
    anns = ds["annotations"]
    assert any(a["iscrowd"] for a in anns) and any(a["num_keypoints"] == 0 for a in anns)
    assert any(a["category_id"] != 1 for a in anns)
    assert any(a["area"] == 32.0 ** 2 for a in anns) and any(a["area"] == 96.0 ** 2 for a in anns)
    per_img = {}
    for r in res:
        per_img[r["image_id"]] = per_img.get(r["image_id"], 0) + 1
    gt_imgs = {a["image_id"] for a in anns if a["category_id"] == 1}
    assert max(per_img.values()) > 20
    assert gt_imgs - set(per_img) and set(per_img) - gt_imgs            # GT-only and detection-only images
    scores = [r["score"] for r in res]
    assert scores.count(0.0) > 5 and len(set(scores)) < len(scores)
    areas = [d["area"] for d in C.load_res([i["id"] for i in ds["images"]], res)]
    assert 32.0 ** 2 in areas and 96.0 ** 2 in areas
    for variant, minus_one in (("medium", (4, 9)), ("large", (3, 8))):
        out = C.coco_eval_kps(*synth.coco_keypoint_set(80, seed=6, variant=variant))
        assert all(out["stats"][i] == -1 for i in minus_one) and all(out["stats"][i] > 0 for i in (0, 5))


def test_abi_rejects_non_default_params():
    from simple_pose_b200 import build, _abi
    build.build()
    lib = _abi.lib()
    args = [16, 54, 16, 16, None, 4, 16, 16, 16, 16, 16, 2, 3, 16, 16, 16, 17, 10, 101, 3, 20,
            16, 16, 16, None, None, None, 16, 1 << 20, None]
    for i, bad in ((16, 16), (17, 5), (18, 100), (19, 4), (20, 100)):      # K, T, R, A, maxDets
        assert lib.sp_coco_eval_kps_f32(*(args[:i] + [bad] + args[i + 1:])) == -4
    assert lib.sp_coco_eval_kps_f32(*(args[:1] + [50] + args[2:])) == -1                 # stride < 3K
    assert lib.sp_coco_eval_kps_f32(*(args[:21] + [None] + args[22:])) == -1             # no precision output
    assert lib.sp_coco_eval_kps_f32(*(args[:10] + [None] + args[11:])) == -1             # no gt_seg
    assert lib.sp_coco_eval_kps_f32(*(args[:27] + [24] + args[28:])) == -2               # misaligned workspace
    assert lib.sp_coco_eval_workspace_bytes(-1, 2, 3) == 0


def _pycocotools():
    try:
        from pycocotools.coco import COCO
        from pycocotools.cocoeval import COCOeval
        return COCO, COCOeval
    except ImportError:
        return None


@pytest.mark.skipif(_pycocotools() is None, reason="pycocotools is not installed")
@pytest.mark.parametrize("variant,seed", [("all", 1), ("medium", 2), ("large", 3)])
def test_oracle_matches_pycocotools(variant, seed):
    import contextlib
    import copy
    import io
    COCO, COCOeval = _pycocotools()
    ds, res = synth.coco_keypoint_set(150, seed=seed, variant=variant)
    ds = dict(ds, categories=[{"id": 1, "name": "person"}, {"id": 3, "name": "car"}])
    with contextlib.redirect_stdout(io.StringIO()):
        gt = COCO()
        gt.dataset = copy.deepcopy(ds)
        gt.createIndex()
        dt = gt.loadRes(copy.deepcopy(res))
        ev = COCOeval(gt, dt, "keypoints")
        ev.params.catIds = [1]
        ev.evaluate()
        ev.accumulate()
        ev.summarize()
    out = C.coco_eval_kps(ds, res)
    assert np.array_equal(out["precision"], ev.eval["precision"][:, :, 0, :, 0])
    assert np.array_equal(out["recall"], ev.eval["recall"][:, 0, :, 0])
    assert np.array_equal(out["stats"], ev.stats)
