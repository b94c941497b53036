"""COCO keypoint AP on the device: pycocotools' ``COCOeval(..., 'keypoints')`` (what the reference runs in
``eval_kps``, ``eval.py:13-27``, and in ``evaluate_map``, ``metrics/pose_metrics.py:182-209``) without the result
JSON file and without pycocotools.

    gt = CocoKeypointGT("person_keypoints_val2017.json", device="cuda")     # parsed once per dataset
    res = evaluate(gt, keypoint_rows, scores, image_ids)                     # six launches, no host sync
    res.stats        # float64 [10] on the device: AP, AP50, AP75, APm, APl, AR, AR50, AR75, ARm, ARl
    print("\\n".join(res.summary()))                                          # summarize()'s ten lines

Only the keypoint defaults are supported: person (``catIds = [1]``), 17 joints, ``maxDets = [20]``, the
thresholds and area ranges of ``Params.setKpParams``. Adapters feed the two tables the project produces:
``evaluate_table`` (``ShardedPoseEvaluator``'s result rows) and ``evaluate_person_rows`` (``kps_to_dict_``'s rows).
"""
import json

import numpy as np
import torch

from .. import _abi

NUM_JOINTS = 17
MAX_DETS = 20
PERSON = 1
_GT_IGNORE, _GT_CROWD = 1, 2
_REQUIRED = ("id", "image_id", "category_id", "keypoints", "num_keypoints", "area", "bbox", "iscrowd")


def kp_params():
    """``Params.setKpParams``: (iouThrs [10], recThrs [101], areaRng [3, 2]) as float64 NumPy arrays, built with
    ``np.linspace`` exactly as pycocotools builds them (the summary's IoU .5 / .75 are selected by equality)."""
    iou = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
    rec = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
    area = np.array([[0 ** 2, 1e5 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]], dtype=np.float64)
    return iou, rec, area


class CocoKeypointGT(object):
    """COCO keypoint ground truth, parsed on the host once and kept on ``device``.

    ``dataset``: the annotation dict (``images``, ``annotations``) or a path to its JSON file. Only person
    annotations (``category_id == 1``) are kept. ``img_ids`` (sorted unique image ids of the ``images`` list unless
    narrowed by ``img_ids``) is ``params.imgIds``; each image's persons keep annotation-file order. A missing key
    raises ``KeyError``; an annotation id < 1 or a keypoint list that is not 17 joints raises ``ValueError``."""

    def __init__(self, dataset, img_ids=None, device=None):
        if isinstance(dataset, str):
            with open(dataset) as fh:
                dataset = json.load(fh)
        all_ids = np.array(sorted({int(img["id"]) for img in dataset["images"]}), dtype=np.int64)
        ids = all_ids if img_ids is None else np.array(sorted({int(i) for i in img_ids}), dtype=np.int64)
        if not np.all(np.isin(ids, all_ids)):
            raise ValueError("img_ids names images that are not in the annotation set")
        pos = {int(i): p for p, i in enumerate(ids)}
        per_img = [[] for _ in ids]
        for ann in dataset["annotations"]:
            for key in ("image_id", "category_id"):
                if key not in ann:
                    raise KeyError("annotation without '%s'" % key)
            if ann["category_id"] != PERSON:
                continue
            for key in _REQUIRED:
                if key not in ann:
                    raise KeyError("person annotation %s without '%s'" % (ann.get("id"), key))
            if int(ann["id"]) < 1:
                raise ValueError("annotation ids must be >= 1 (COCOeval tests matches by id)")
            if len(ann["keypoints"]) != 3 * NUM_JOINTS or len(ann["bbox"]) != 4:
                raise ValueError("annotation %s: expected %d keypoints and a 4-value bbox" % (ann["id"], NUM_JOINTS))
            p = pos.get(int(ann["image_id"]))
            if p is not None:
                per_img[p].append(ann)
        anns = [a for lst in per_img for a in lst]
        seg = np.zeros(len(ids) + 1, dtype=np.int32)
        seg[1:] = np.cumsum([len(lst) for lst in per_img])
        kps = np.array([a["keypoints"] for a in anns], dtype=np.float64).reshape(-1, 3 * NUM_JOINTS)
        flags = np.array([(_GT_IGNORE if (a["iscrowd"] or a["num_keypoints"] == 0) else 0) |
                          (_GT_CROWD if int(a["iscrowd"]) else 0) for a in anns], dtype=np.uint8)
        self.all_img_ids = all_ids
        self.img_ids = ids
        self.ann_ids = np.array([int(a["id"]) for a in anns], dtype=np.int64)
        self.num_images, self.num_gts = len(ids), len(anns)
        dev = torch.device(device) if device is not None else _abi.default_device()
        self.device = dev
        self.seg = torch.from_numpy(seg).to(dev)
        self.kps = torch.from_numpy(kps).to(dev)
        self.area = torch.tensor([float(a["area"]) for a in anns], dtype=torch.float64).to(dev)
        self.bbox = torch.tensor([[float(v) for v in a["bbox"]] for a in anns], dtype=torch.float64).reshape(-1, 4).to(dev)
        self.flags = torch.from_numpy(flags).to(dev)
        iou, rec, area = kp_params()
        self.iou_thrs = torch.from_numpy(iou).to(dev)
        self.rec_thrs = torch.from_numpy(rec).to(dev)
        self.area_rng = torch.from_numpy(area).to(dev)

    def positions(self, image_ids):
        """COCO image ids of detections (host sequence or a CUDA tensor) -> int32 CUDA positions in ``img_ids``
        (-1 for a GT image outside a narrowed ``img_ids``). An id that is not a GT image raises ``ValueError``, as
        ``loadRes`` asserts; for a CUDA tensor that check reads one flag back from the device."""
        if isinstance(image_ids, torch.Tensor) and image_ids.is_cuda:
            ids = image_ids.reshape(-1).to(torch.int64)
            all_ids = torch.from_numpy(self.all_img_ids).to(ids.device)
            j = torch.searchsorted(all_ids, ids).clamp(max=max(len(self.all_img_ids) - 1, 0))
            if ids.numel() and (len(self.all_img_ids) == 0 or not bool((all_ids[j] == ids).all())):
                raise ValueError("detections name images that are not in the annotation set")
            ev = torch.from_numpy(self.img_ids).to(ids.device)
            k = torch.searchsorted(ev, ids).clamp(max=max(len(self.img_ids) - 1, 0))
            hit = (ev[k] == ids) if len(self.img_ids) else torch.zeros_like(ids, dtype=torch.bool)
            return torch.where(hit, k, torch.full_like(k, -1)).to(torch.int32)
        ids = np.asarray(image_ids.cpu() if isinstance(image_ids, torch.Tensor) else image_ids, dtype=np.int64).reshape(-1)
        if ids.size and not np.all(np.isin(ids, self.all_img_ids)):
            raise ValueError("detections name images that are not in the annotation set")
        k = np.searchsorted(self.img_ids, ids)
        hit = (k < len(self.img_ids)) & (self.img_ids[np.minimum(k, max(len(self.img_ids) - 1, 0))] == ids) \
            if len(self.img_ids) else np.zeros(ids.shape, dtype=bool)
        return torch.from_numpy(np.where(hit, k, -1).astype(np.int32)).to(self.device)


_SUMMARY = [(1, None, "all"), (1, .5, "all"), (1, .75, "all"), (1, None, "medium"), (1, None, "large"),
            (0, None, "all"), (0, .5, "all"), (0, .75, "all"), (0, None, "medium"), (0, None, "large")]


class CocoEvalResult(object):
    """Device tensors: ``precision`` float64 [10, 101, 3] (IoU threshold, recall threshold, area range),
    ``recall`` [10, 3], ``stats`` [10]; with ``diagnostics=True`` also ``oks``, ``det_flags`` and ``det_order`` in
    the layouts of ``sp_coco_eval_kps_f32``."""

    def __init__(self, precision, recall, stats, oks=None, det_flags=None, det_order=None):
        self.precision, self.recall, self.stats = precision, recall, stats
        self.oks, self.det_flags, self.det_order = oks, det_flags, det_order

    def summary(self):
        """The ten lines ``COCOeval.summarize()`` prints for keypoints (reads the stats back to the host)."""
        out = []
        for (ap, iou, area), v in zip(_SUMMARY, self.stats.cpu().tolist()):
            title = "Average Precision" if ap == 1 else "Average Recall"
            iou_s = "0.50:0.95" if iou is None else "{:0.2f}".format(iou)
            out.append(" {:<18} {} @[ IoU={:<9} | area={:>6s} | maxDets={:>3d} ] = {:0.3f}".format(
                title, "(AP)" if ap == 1 else "(AR)", iou_s, area, MAX_DETS, v))
        return out


def evaluate(gt, keypoint_rows, scores, image_ids, keep=None, diagnostics=False):
    """COCOeval for keypoints over detections given as CUDA tensors.

    ``keypoint_rows``: float32 [N, W] with x of joint k at column 3k and y at 3k+1 (W >= 51; row stride W, columns
    contiguous), or [N, 17, 3]. ``scores``: [N] (widened to float64). ``image_ids``: [N] COCO image ids (host
    sequence or CUDA tensor). ``keep``: optional [N] bool / uint8 mask of the detections that are results.
    Within an image, the order of the rows is the results-list order (it decides equal scores)."""
    rows = keypoint_rows
    dev = _abi.require_cuda(rows, scores, keep)
    if dev is None:
        raise RuntimeError("simple_pose_b200: expected CUDA tensors (there is no CPU path)")
    if dev != gt.device:
        raise RuntimeError("simple_pose_b200: detections on %s, ground truth on %s" % (dev, gt.device))
    if rows.dim() == 3:
        rows = rows.reshape(rows.shape[0], -1)
    if rows.dim() != 2 or rows.shape[1] < 3 * NUM_JOINTS:
        raise ValueError("keypoint_rows must be [N, >= %d] or [N, %d, 3]" % (3 * NUM_JOINTS, NUM_JOINTS))
    if rows.dtype != torch.float32 or rows.stride(1) != 1 or (rows.shape[0] > 1 and rows.stride(0) < rows.shape[1]):
        rows = _abi.dense(rows, torch.float32)
    n = int(rows.shape[0])
    sc = _abi.dense(scores.reshape(-1), torch.float64)
    if sc.shape[0] != n:
        raise ValueError("scores must have one value per row")
    pos = gt.positions(image_ids)
    if pos.shape[0] != n:
        raise ValueError("image_ids must have one id per row")
    kp = None if keep is None else _abi.dense(keep.reshape(-1), torch.uint8)
    if kp is not None and kp.shape[0] != n:
        raise ValueError("keep must have one flag per row")
    I, G = gt.num_images, gt.num_gts
    precision = torch.empty((10, 101, 3), dtype=torch.float64, device=dev)
    recall = torch.empty((10, 3), dtype=torch.float64, device=dev)
    stats = torch.empty((10,), dtype=torch.float64, device=dev)
    oks = det_flags = det_order = None
    if diagnostics:
        oks = torch.full((MAX_DETS * G,), float("nan"), dtype=torch.float64, device=dev)
        det_flags = torch.zeros((I * MAX_DETS,), dtype=torch.int64, device=dev)
        det_order = torch.full((I * MAX_DETS,), -1, dtype=torch.int32, device=dev)
    lib = _abi.lib()
    stride = int(rows.stride(0)) if n > 0 else int(rows.shape[1])
    with torch.cuda.device(dev):
        nbytes = lib.sp_coco_eval_workspace_bytes(n, I, G)
        if nbytes == 0:
            raise RuntimeError("simple_pose_b200: COCO eval workspace size query failed")
        stream = _abi.stream_ptr(dev)
        ws = _abi.scratch(dev, stream, nbytes, "coco_eval")
        _abi.check(lib.sp_coco_eval_kps_f32(
            rows.data_ptr() if n else None, stride, sc.data_ptr() if n else None, pos.data_ptr() if n else None,
            _abi.ptr(kp) if n else None, n,
            gt.kps.data_ptr() if G else None, gt.area.data_ptr() if G else None, gt.bbox.data_ptr() if G else None,
            gt.flags.data_ptr() if G else None, gt.seg.data_ptr(), I, G,
            gt.iou_thrs.data_ptr(), gt.rec_thrs.data_ptr(), gt.area_rng.data_ptr(), NUM_JOINTS, 10, 101, 3, MAX_DETS,
            precision.data_ptr(), recall.data_ptr(), stats.data_ptr(),
            _abi.ptr(oks) if G else None, _abi.ptr(det_flags) if I else None, _abi.ptr(det_order) if I else None,
            ws.data_ptr(), ws.numel() * 8, stream))
    if diagnostics:
        return CocoEvalResult(precision, recall, stats, oks, det_flags, det_order)
    return CocoEvalResult(precision, recall, stats)


def evaluate_table(gt, rows, seg_offsets, image_ids):
    """AP of ``ShardedPoseEvaluator``'s result table: ``rows`` [N, 3K+3] (kept rows are the results, their score is
    the float64 rescored score), ``seg_offsets`` [I+1] the persons of each eval image, ``image_ids`` [I] the COCO
    id of each eval image (host). eval.py lists an image's kept persons in NMS pick order -- descending score, equal
    scores higher person index first -- so the table is handed over reversed: the evaluator's stable order of equal
    scores is then eval.py's."""
    from ..eval_shard import ROW_EXTRA, row_keep, row_scores
    _abi.require_cuda(rows)
    seg = np.asarray(seg_offsets, dtype=np.int64)
    ids = np.asarray(image_ids, dtype=np.int64).reshape(-1)
    if ids.shape[0] != seg.shape[0] - 1 or rows.shape[0] != int(seg[-1]) or rows.shape[1] != 3 * NUM_JOINTS + ROW_EXTRA:
        raise ValueError("rows [N, %d], seg_offsets [I+1] and image_ids [I] must describe the same persons"
                         % (3 * NUM_JOINTS + ROW_EXTRA))
    per_person = np.repeat(ids, np.diff(seg))[::-1]
    rev = rows.flip(0)
    return evaluate(gt, rev, row_scores(rev), np.ascontiguousarray(per_person), keep=row_keep(rev))


def evaluate_person_rows(gt, rows, image_ids):
    """AP of ``kps_to_dict_``'s rows (``person_rows``: [N, 3K+1] float32, the score in the last column, widened to
    float64 as the JSON round trip does) in loader order, ``image_ids`` [N] one COCO image id per row."""
    _abi.require_cuda(rows)
    if rows.dim() != 2 or rows.shape[1] != 3 * NUM_JOINTS + 1:
        raise ValueError("rows must be [N, %d]" % (3 * NUM_JOINTS + 1))
    return evaluate(gt, rows, rows[:, -1].to(torch.float64), image_ids)
