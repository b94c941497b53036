"""TEST INFRASTRUCTURE ONLY -- CPU restatement of pycocotools' COCOeval for ``iouType='keypoints'``.

Nothing in ``simple_pose_b200/`` imports this module. It is the yardstick of the device evaluator
(``simple_pose_b200/metrics/coco_eval.py``, ``csrc/sp_coco_eval.cu``) and of ``profiles/bench_coco_eval.py``.

The reference scores its keypoints with pycocotools 2.0.x (``eval.py:13-27`` and ``evaluate_map`` in
``metrics/pose_metrics.py:182-209``): ``COCO(gt)``, ``loadRes(results)``, ``COCOeval(gt, dt, 'keypoints')``,
``evaluate()``, ``accumulate()``, ``summarize()``. Each function below names the pycocotools function it restates
(``pycocotools/coco.py`` and ``pycocotools/cocoeval.py``) and keeps its NumPy operations and their order, so its
``precision``, ``recall`` and ``stats`` are what pycocotools computes. Only what applies to keypoints with the
keypoint defaults, ``catIds = [1]`` and ``maxDets = [20]`` is restated.
"""
from collections import defaultdict

import numpy as np

PERSON = 1


def kp_params():
    """``Params.setKpParams`` (cocoeval.py): thresholds exactly as pycocotools builds them with ``np.linspace``."""
    return {
        "iouThrs": np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True),
        "recThrs": np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True),
        "maxDets": [20],
        "areaRng": [[0 ** 2, 1e5 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]],
        "areaRngLbl": ["all", "medium", "large"],
        "kpt_oks_sigmas": np.array([.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07,
                                    .87, .87, .89, .89]) / 10.0,
        "catIds": [PERSON],
    }


def load_gt(dataset):
    """``COCO.createIndex`` + ``getImgIds`` + ``getAnnIds(imgIds, catIds=[1])`` + ``loadAnns``: the GT image ids
    (all images of the ``images`` list) and, per image, its person annotations in annotation-file order."""
    img_ids = [img["id"] for img in dataset["images"]]
    per_img = defaultdict(list)
    for ann in dataset["annotations"]:
        if ann["category_id"] == PERSON:
            per_img[ann["image_id"]].append(ann)
    return img_ids, per_img


def load_res(gt_img_ids, results):
    """``COCO.loadRes`` for a list of keypoint results: every result's image must be a GT image (the assertion of
    loadRes); ``area`` is the extent of the keypoints, ``id`` the list position + 1. Returns new dicts."""
    anns = [dict(r) for r in results]
    ann_img_ids = [a["image_id"] for a in anns]
    assert set(ann_img_ids) == (set(ann_img_ids) & set(gt_img_ids)), \
        "Results do not correspond to current coco set"
    for i, ann in enumerate(anns):
        s = ann["keypoints"]
        x = s[0::3]
        y = s[1::3]
        x0, x1, y0, y1 = np.min(x), np.max(x), np.min(y), np.max(y)
        ann["area"] = (x1 - x0) * (y1 - y0)
        ann["id"] = i + 1
        ann["bbox"] = [x0, y0, x1 - x0, y1 - y0]
    return anns


def prepare(gt_per_img, dts, img_ids):
    """``COCOeval._prepare`` (keypoints): ``ignore = iscrowd or num_keypoints == 0`` overwrites any stored flag;
    GT and detections are grouped per image of ``img_ids``, in file / results-list order."""
    gts = {}
    for i in img_ids:
        lst = []
        for g in gt_per_img.get(i, []):
            g = dict(g)
            g["ignore"] = g["ignore"] if "ignore" in g else 0
            g["ignore"] = "iscrowd" in g and g["iscrowd"]
            g["ignore"] = (g["num_keypoints"] == 0) or g["ignore"]
            lst.append(g)
        gts[i] = lst
    wanted = set(img_ids)
    dt_per = defaultdict(list)
    for d in dts:
        if d["image_id"] in wanted and d.get("category_id", PERSON) == PERSON:
            dt_per[d["image_id"]].append(d)
    return gts, dt_per


def compute_oks(gts, dts, p):
    """``COCOeval.computeOks``: detections sorted by ``-score`` (stable) and cut to ``maxDets[-1]``; OKS against
    the visible GT joints, or against the GT box grown to [x-w, x+2w] x [y-h, y+2h] when the GT has none."""
    inds = np.argsort([-d["score"] for d in dts], kind="mergesort")
    dts = [dts[i] for i in inds]
    if len(dts) > p["maxDets"][-1]:
        dts = dts[0:p["maxDets"][-1]]
    if len(gts) == 0 or len(dts) == 0:
        return []
    ious = np.zeros((len(dts), len(gts)))
    sigmas = p["kpt_oks_sigmas"]
    vars = (sigmas * 2) ** 2
    k = len(sigmas)
    for j, gt in enumerate(gts):
        g = np.array(gt["keypoints"])
        xg = g[0::3]
        yg = g[1::3]
        vg = g[2::3]
        k1 = np.count_nonzero(vg > 0)
        bb = gt["bbox"]
        x0 = bb[0] - bb[2]
        x1 = bb[0] + bb[2] * 2
        y0 = bb[1] - bb[3]
        y1 = bb[1] + bb[3] * 2
        for i, dt in enumerate(dts):
            d = np.array(dt["keypoints"])
            xd = d[0::3]
            yd = d[1::3]
            if k1 > 0:
                dx = xd - xg
                dy = yd - yg
            else:
                z = np.zeros((k))
                dx = np.max((z, x0 - xd), axis=0) + np.max((z, xd - x1), axis=0)
                dy = np.max((z, y0 - yd), axis=0) + np.max((z, yd - y1), axis=0)
            e = (dx ** 2 + dy ** 2) / vars / (gt["area"] + np.spacing(1)) / 2
            if k1 > 0:
                e = e[vg > 0]
            ious[i, j] = np.sum(np.exp(-e)) / e.shape[0]
    return ious


def evaluate_img(gt, dt, ious, a_rng, p):
    """``COCOeval.evaluateImg`` for one image and one area range (maxDet = 20). Returns None for an image with
    neither GT nor detections."""
    max_det = p["maxDets"][-1]
    if len(gt) == 0 and len(dt) == 0:
        return None
    for g in gt:
        if g["ignore"] or (g["area"] < a_rng[0] or g["area"] > a_rng[1]):
            g["_ignore"] = 1
        else:
            g["_ignore"] = 0
    gtind = np.argsort([g["_ignore"] for g in gt], kind="mergesort")
    gt = [gt[i] for i in gtind]
    dtind = np.argsort([-d["score"] for d in dt], kind="mergesort")
    dt = [dt[i] for i in dtind[0:max_det]]
    iscrowd = [int(o["iscrowd"]) for o in gt]
    ious = ious[:, gtind] if len(ious) > 0 else ious
    T = len(p["iouThrs"])
    G = len(gt)
    D = len(dt)
    gtm = np.zeros((T, G))
    dtm = np.zeros((T, D))
    gtIg = np.array([g["_ignore"] for g in gt])
    dtIg = np.zeros((T, D))
    if not len(ious) == 0:
        for tind, t in enumerate(p["iouThrs"]):
            for dind, d in enumerate(dt):
                iou = min([t, 1 - 1e-10])
                m = -1
                for gind, g in enumerate(gt):
                    if gtm[tind, gind] > 0 and not iscrowd[gind]:
                        continue
                    if m > -1 and gtIg[m] == 0 and gtIg[gind] == 1:
                        break
                    if ious[dind, gind] < iou:
                        continue
                    iou = ious[dind, gind]
                    m = gind
                if m == -1:
                    continue
                dtIg[tind, dind] = gtIg[m]
                dtm[tind, dind] = gt[m]["id"]
                gtm[tind, m] = d["id"]
    a = np.array([d["area"] < a_rng[0] or d["area"] > a_rng[1] for d in dt]).reshape((1, len(dt)))
    dtIg = np.logical_or(dtIg, np.logical_and(dtm == 0, np.repeat(a, T, 0)))
    return {
        "dtIds": [d["id"] for d in dt],
        "gtIds": [g["id"] for g in gt],
        "dtMatches": dtm,
        "gtMatches": gtm,
        "dtScores": [d["score"] for d in dt],
        "gtIgnore": gtIg,
        "dtIgnore": dtIg,
    }


def accumulate(eval_imgs, n_imgs, p):
    """``COCOeval.accumulate`` for one category and maxDets = [20]: ``precision`` [T, R, A] and ``recall`` [T, A]
    (pycocotools' K = M = 1 axes dropped), -1 where there is no non-ignored GT."""
    T, R, A = len(p["iouThrs"]), len(p["recThrs"]), len(p["areaRng"])
    precision = -np.ones((T, R, A))
    recall = -np.ones((T, A))
    max_det = p["maxDets"][-1]
    for a in range(A):
        E = [eval_imgs[a * n_imgs + i] for i in range(n_imgs)]
        E = [e for e in E if e is not None]
        if len(E) == 0:
            continue
        dtScores = np.concatenate([e["dtScores"][0:max_det] for e in E])
        inds = np.argsort(-dtScores, kind="mergesort")
        dtm = np.concatenate([e["dtMatches"][:, 0:max_det] for e in E], axis=1)[:, inds]
        dtIg = np.concatenate([e["dtIgnore"][:, 0:max_det] for e in E], axis=1)[:, inds]
        gtIg = np.concatenate([e["gtIgnore"] for e in E])
        npig = np.count_nonzero(gtIg == 0)
        if npig == 0:
            continue
        tps = np.logical_and(dtm, np.logical_not(dtIg))
        fps = np.logical_and(np.logical_not(dtm), np.logical_not(dtIg))
        tp_sum = np.cumsum(tps, axis=1).astype(dtype=float)
        fp_sum = np.cumsum(fps, axis=1).astype(dtype=float)
        for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
            tp = np.array(tp)
            fp = np.array(fp)
            nd = len(tp)
            rc = tp / npig
            pr = tp / (fp + tp + np.spacing(1))
            q = np.zeros((R,))
            if nd:
                recall[t, a] = rc[-1]
            else:
                recall[t, a] = 0
            pr = pr.tolist()
            q = q.tolist()
            for i in range(nd - 1, 0, -1):
                if pr[i] > pr[i - 1]:
                    pr[i - 1] = pr[i]
            inds_r = np.searchsorted(rc, p["recThrs"], side="left")
            try:
                for ri, pi in enumerate(inds_r):
                    q[ri] = pr[pi]
            except IndexError:
                pass
            precision[t, :, a] = np.array(q)
    return precision, recall


def summarize_kps(precision, recall, p):
    """``COCOeval.summarize`` -> ``_summarizeKps``: the ten ``np.mean(s[s > -1])`` (-1 when empty). ``iouThr`` is
    selected with ``np.where(iouThr == iouThrs)``, i.e. against the linspace values."""
    def _summarize(ap=1, iouThr=None, areaRng="all"):
        aind = [i for i, lbl in enumerate(p["areaRngLbl"]) if lbl == areaRng]
        if ap == 1:
            s = precision[:, :, None, :, None]          # pycocotools' [T, R, K, A, M]
            if iouThr is not None:
                t = np.where(iouThr == p["iouThrs"])[0]
                s = s[t]
            s = s[:, :, :, aind, [0]]
        else:
            s = recall[:, None, :, None]                # [T, K, A, M]
            if iouThr is not None:
                t = np.where(iouThr == p["iouThrs"])[0]
                s = s[t]
            s = s[:, :, aind, [0]]
        if len(s[s > -1]) == 0:
            return -1
        return np.mean(s[s > -1])

    stats = np.zeros((10,))
    stats[0] = _summarize(1)
    stats[1] = _summarize(1, iouThr=.5)
    stats[2] = _summarize(1, iouThr=.75)
    stats[3] = _summarize(1, areaRng="medium")
    stats[4] = _summarize(1, areaRng="large")
    stats[5] = _summarize(0)
    stats[6] = _summarize(0, iouThr=.5)
    stats[7] = _summarize(0, iouThr=.75)
    stats[8] = _summarize(0, areaRng="medium")
    stats[9] = _summarize(0, areaRng="large")
    return stats


def coco_eval_kps(dataset, results, img_ids=None):
    """``COCOeval(cocoGt, cocoGt.loadRes(results), 'keypoints')`` with ``catIds = [1]``, then ``evaluate()``,
    ``accumulate()`` and the statistics of ``summarize()``. ``dataset``: the GT annotation dict; ``results``: list
    of {"image_id", "category_id", "keypoints", "score"}; ``img_ids`` narrows ``params.imgIds``.

    Returns a dict: ``precision`` [10, 101, 3], ``recall`` [10, 3], ``stats`` [10], and per evaluated image id
    ``ious`` (sorted, truncated detections x GT in file order) and ``eval_imgs`` (evaluateImg results, area-major)."""
    p = kp_params()
    gt_img_ids, gt_per_img = load_gt(dataset)
    dts = load_res(gt_img_ids, results)
    img_ids = sorted(set(gt_img_ids)) if img_ids is None else sorted(set(img_ids))
    gts, dt_per = prepare(gt_per_img, dts, img_ids)
    ious = {i: compute_oks(gts[i], dt_per[i], p) for i in img_ids}
    eval_imgs = [evaluate_img(gts[i], dt_per[i], ious[i], a_rng, p) for a_rng in p["areaRng"] for i in img_ids]
    precision, recall = accumulate(eval_imgs, len(img_ids), p)
    stats = summarize_kps(precision, recall, p)
    return {"precision": precision, "recall": recall, "stats": stats, "ious": ious, "eval_imgs": eval_imgs,
            "img_ids": img_ids, "params": p}

