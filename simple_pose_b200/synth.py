"""Fixed-seed synthetic inputs for the heatmap hot path (SURVEY.md section 8d).

Used by the parity tests (generated on CPU so the oracle and the kernels see identical
bits), by ``bench.py`` (generated directly on the GPU for the large configurations) and
by ``__graft_entry__.smoke()``. Pure torch (NumPy for the COCO annotation sets); no oracle and no CUDA
extension involved.
"""
import math

import torch

COCO_JOINT_PAIRS = ((1, 2), (3, 4), (5, 6), (7, 8), (9, 10), (11, 12), (13, 14), (15, 16))


def _gen(seed, device):
    g = torch.Generator(device=device)
    g.manual_seed(int(seed))
    return g


def swap_permutation(num_joints=17, joint_pairs=COCO_JOINT_PAIRS):
    perm = list(range(num_joints))
    for a, b in joint_pairs:
        perm[a], perm[b] = perm[b], perm[a]
    return perm


def peak_centres(persons, joints=17, height=64, width=48, seed=0, device="cpu",
                 border_frac=0.03):
    """Peak centres [P,K,2] (x, y): uniform over the map, ``border_frac`` of them pushed to
    within 2 px of a border so the unrefined decoder branches are exercised."""
    g = _gen(seed, device)
    mu = torch.rand(persons, joints, 2, generator=g, device=device)
    mu[..., 0] *= (width - 1)
    mu[..., 1] *= (height - 1)
    edge = torch.rand(persons, joints, generator=g, device=device) < border_frac
    side = torch.randint(0, 4, (persons, joints), generator=g, device=device)
    near = torch.rand(persons, joints, generator=g, device=device) * 2.0
    x = torch.where(edge & (side == 0), near, mu[..., 0])
    x = torch.where(edge & (side == 1), (width - 1) - near, x)
    y = torch.where(edge & (side == 2), near, mu[..., 1])
    y = torch.where(edge & (side == 3), (height - 1) - near, y)
    return torch.stack([x, y], dim=-1)


def heatmaps_from_centres(mu, height=64, width=48, seed=0, noise=0.01, dead_frac=0.01,
                          amp_lo=0.3, amp_hi=1.0, chunk=4096):
    """hm = amp * exp(-|p - mu|^2 / 8) + N(0, noise^2); ``dead_frac`` of the maps are
    all <= 0 (peak removed, |noise| negated)."""
    device = mu.device
    persons, joints = mu.shape[:2]
    g = _gen(seed + 7919, device)
    out = torch.empty(persons, joints, height, width, dtype=torch.float32, device=device)
    xs = torch.arange(width, dtype=torch.float32, device=device)
    ys = torch.arange(height, dtype=torch.float32, device=device)
    for lo in range(0, persons, chunk):
        hi = min(persons, lo + chunk)
        m = mu[lo:hi]
        amp = amp_lo + (amp_hi - amp_lo) * torch.rand(hi - lo, joints, generator=g, device=device)
        dead = torch.rand(hi - lo, joints, generator=g, device=device) < dead_frac
        ex = torch.exp(-(xs[None, None, :] - m[..., 0:1]) ** 2 / 8.0)
        ey = torch.exp(-(ys[None, None, :] - m[..., 1:2]) ** 2 / 8.0)
        blob = amp[..., None, None] * ey[..., :, None] * ex[..., None, :]
        nz = torch.randn(hi - lo, joints, height, width, generator=g, device=device) * noise
        hm = blob + nz
        hm = torch.where(dead[..., None, None], -nz.abs(), hm)
        out[lo:hi] = hm
    return out


def heatmaps(persons, joints=17, height=64, width=48, seed=0, noise=0.01, device="cpu",
             border_frac=0.03, dead_frac=0.01):
    mu = peak_centres(persons, joints, height, width, seed, device, border_frac)
    return heatmaps_from_centres(mu, height, width, seed, noise, dead_frac)


def flip_pair(persons, joints=17, height=64, width=48, seed=0, noise=0.01, device="cpu",
              jitter=0.25, joint_pairs=COCO_JOINT_PAIRS):
    """(hm, hm_flip): ``hm_flip`` is what a network would emit for the mirrored image --
    a second draw (same centres jittered by N(0, jitter^2) px) mirrored in x with the
    left/right channels swapped."""
    mu = peak_centres(persons, joints, height, width, seed, device)
    hm = heatmaps_from_centres(mu, height, width, seed, noise)
    g = _gen(seed + 104729, device)
    mu2 = mu + jitter * torch.randn(mu.shape, generator=g, device=device)
    mu2[..., 0].clamp_(0, width - 1)
    mu2[..., 1].clamp_(0, height - 1)
    second = heatmaps_from_centres(mu2, height, width, seed + 1, noise)
    perm = swap_permutation(joints, joint_pairs)
    hm_flip = second.flip(-1)[:, perm].contiguous()
    return hm, hm_flip


def inverse_affines(persons, height=64, width=48, seed=0, device="cpu"):
    """trans_inv [P,2,3] float32 and area [P] float64 for random COCO-like boxes
    (w ~ U(40,300), h ~ U(80,480), centre inside 640x480), rotation 0. Closed form of
    what ``box_to_center_scale`` + ``get_affine_transform(c, s, 0, (W,H))`` yield
    (reference commons/joint_utils.py:39-56,115-152): uniform scale s = scale_w / W,
    translation c - s * (W/2, H/2); area = scale_w * scale_h (datasets/naive_data.py:55)."""
    g = _gen(seed + 15485863, device)
    u = torch.rand(persons, 4, generator=g, device=device, dtype=torch.float64)
    bw = 40.0 + 260.0 * u[:, 0]
    bh = 80.0 + 400.0 * u[:, 1]
    cx = 640.0 * u[:, 2]
    cy = 480.0 * u[:, 3]
    aspect = width / height
    wide = bw > aspect * bh
    bw2 = torch.where(wide, bw, bh * aspect)
    bh2 = torch.where(wide, bw / aspect, bh)
    sw, sh = bw2 * 1.25, bh2 * 1.25
    s = sw / width
    t = torch.zeros(persons, 2, 3, dtype=torch.float64, device=device)
    t[:, 0, 0] = s
    t[:, 1, 1] = s
    t[:, 0, 2] = cx - s * (width * 0.5)
    t[:, 1, 2] = cy - s * (height * 0.5)
    return t.float(), (sw * sh)


def identity_affines(persons, device="cpu"):
    t = torch.zeros(persons, 2, 3, dtype=torch.float32, device=device)
    t[:, 0, 0] = 1.0
    t[:, 1, 1] = 1.0
    return t


def joints(persons, num_joints=17, height=64, width=48, seed=0, device="cpu", vis_p=0.8):
    """Heatmap-space joints [P,K,3] float32: x ~ U(-8, W+8), y ~ U(-8, H+8),
    vis ~ Bernoulli(vis_p). Covers both branches of the encoder's cull test."""
    g = _gen(seed + 32452843, device)
    u = torch.rand(persons, num_joints, 3, generator=g, device=device)
    out = torch.empty(persons, num_joints, 3, dtype=torch.float32, device=device)
    out[..., 0] = -8.0 + (width + 16.0) * u[..., 0]
    out[..., 1] = -8.0 + (height + 16.0) * u[..., 1]
    out[..., 2] = (u[..., 2] < vis_p).float()
    return out


def predictions_like(targets, seed=1, noise=0.05):
    """pred = target + N(0, noise^2) (what a partly trained network emits)."""
    g = _gen(seed + 49979687, targets.device)
    return targets + noise * torch.randn(targets.shape, generator=g, device=targets.device)


def nms_groups(images, mean_group=20.0, seed=0, num_joints=17, dup_frac=0.5, jitter=2.0):
    """Synthetic detections for OKS-NMS, float64 on CPU.

    Returns (kps [N,K,3], box_scores [N], areas [N], seg_offsets [I+1] int32). Group size is
    1 + Poisson(mean_group); inside a group poses come in clusters of near duplicates
    (jitter N(0, jitter^2) px) so a non-trivial fraction exceeds OKS 0.9; box scores are
    distinct (no sort ties)."""
    g = _gen(seed + 67867967, "cpu")
    sizes = 1 + torch.poisson(torch.full((images,), float(mean_group)), generator=g).long()
    seg = torch.zeros(images + 1, dtype=torch.int64)
    seg[1:] = torch.cumsum(sizes, 0)
    n = int(seg[-1])
    kps = torch.empty(n, num_joints, 3, dtype=torch.float64)
    areas = torch.empty(n, dtype=torch.float64)
    for i in range(images):
        lo, hi = int(seg[i]), int(seg[i + 1])
        m = hi - lo
        n_proto = max(1, int(math.ceil(m * (1.0 - dup_frac))))
        centre = torch.rand(n_proto, 2, generator=g, dtype=torch.float64) * torch.tensor([640.0, 480.0], dtype=torch.float64)
        size = 60.0 + 240.0 * torch.rand(n_proto, generator=g, dtype=torch.float64)
        shape = (torch.rand(n_proto, num_joints, 2, generator=g, dtype=torch.float64) - 0.5)
        proto = centre[:, None, :] + shape * size[:, None, None]
        which = torch.randint(0, n_proto, (m,), generator=g)
        which[:n_proto] = torch.arange(n_proto)
        pose = proto[which] + jitter * torch.randn(m, num_joints, 2, generator=g, dtype=torch.float64)
        conf = 0.05 + 0.95 * torch.rand(m, num_joints, generator=g, dtype=torch.float64)
        kps[lo:hi, :, :2] = pose
        kps[lo:hi, :, 2] = conf
        areas[lo:hi] = (size[which] * 1.25) ** 2 * 0.75
    perm = torch.randperm(n, generator=g).double()
    box_scores = (perm + 0.5) / n
    return kps, box_scores, areas, seg.to(torch.int32)


def detection_boxes(persons, seed=0, ratio_exact_every=0, ratio=0.75):
    """COCO-like detection boxes [P,4] float64 (x1, y1, x2, y2): w ~ U(8,400), h ~ U(8,560), top-left
    corner in [-40,640) x [-40,480) (detectors do emit slightly negative corners). With
    ``ratio_exact_every`` > 0 every n-th box has w == ratio * h exactly (neither branch of the
    aspect fix of ``box_to_center_scale``)."""
    g = _gen(seed + 982451653, "cpu")
    u = torch.rand(persons, 4, generator=g, dtype=torch.float64)
    w = 8.0 + 392.0 * u[:, 0]
    h = 8.0 + 552.0 * u[:, 1]
    x = -40.0 + 680.0 * u[:, 2]
    y = -40.0 + 520.0 * u[:, 3]
    if ratio_exact_every:
        h[::ratio_exact_every] = torch.floor(h[::ratio_exact_every] / 4.0) * 4.0
        w[::ratio_exact_every] = h[::ratio_exact_every] * ratio
    return torch.stack([x, y, x + w, y + h], dim=1)


def train_samples(persons, num_joints=17, seed=0, img_w=(200, 640), img_h=(200, 480), vis_p=0.8,
                  scale=(0.7, 1.3), rot=(-40.0, 40.0), flip_p=0.5):
    """Inputs of the train-side transform (``RefineSimpleTransform.__call__``, commons/transforms.py:
    193-223) after its random draws: per person an image width, a ground-truth box inside the image
    (float64 [x1, y1, x2, y2]), image-pixel joints [K,3] float32 (x, y, vis in {0,1}; most inside the
    box, some outside so that the encoder's cull test fires), and the three draws of :204-211 --
    ``scale_ratio`` ~ U(scale), ``rot`` ~ U(rot) degrees (every 8th exactly 0), ``flip`` ~ B(flip_p).
    Returns a dict of CPU tensors."""
    g = _gen(seed + 49979687, "cpu")
    u = torch.rand(persons, 8, generator=g, dtype=torch.float64)
    w_img = torch.floor(img_w[0] + (img_w[1] - img_w[0]) * u[:, 0])
    h_img = torch.floor(img_h[0] + (img_h[1] - img_h[0]) * u[:, 1])
    bw = 20.0 + (w_img - 24.0) * u[:, 2]
    bh = 30.0 + (h_img - 34.0) * u[:, 3]
    x1 = (w_img - bw - 1.0).clamp(min=0.0) * u[:, 4]
    y1 = (h_img - bh - 1.0).clamp(min=0.0) * u[:, 5]
    boxes = torch.stack([x1, y1, x1 + bw, y1 + bh], dim=1)
    ju = torch.rand(persons, num_joints, 3, generator=g, dtype=torch.float64)
    jx = x1[:, None] + bw[:, None] * (1.5 * ju[..., 0] - 0.25)
    jy = y1[:, None] + bh[:, None] * (1.5 * ju[..., 1] - 0.25)
    vis = (ju[..., 2] < vis_p).to(torch.float64)
    joints_img = torch.stack([jx, jy, vis], dim=-1).to(torch.float32)
    scale_ratio = scale[0] + (scale[1] - scale[0]) * u[:, 6]
    rot_deg = rot[0] + (rot[1] - rot[0]) * u[:, 7]
    rot_deg[::8] = 0.0
    flip = torch.rand(persons, generator=g, dtype=torch.float64) < flip_p
    return {"img_w": w_img.to(torch.int32), "boxes": boxes, "joints": joints_img,
            "scale_ratio": scale_ratio, "rot": rot_deg, "flip": flip}


class EvalSet(object):
    """A COCO-val-sized synthetic eval job (BASELINE config 5) whose content depends on the PERSON index
    only -- never on how the persons are sharded -- so that the result table of a 1-, 2-, 4- or 8-GPU run
    must be bit-identical. Images hold 1 + Poisson(mean_group) detections; inside an image a fraction
    ``dup_frac`` of the detections are near-duplicates of another detection of the same image (the same
    box jittered by N(0, box_jitter^2) px, the same peak centres jittered by N(0, jitter^2) heatmap px)
    so that the OKS-NMS has something to suppress (SURVEY section 8d). Box scores are distinct.

    Host metadata (``seg``, ``boxes``, ``box_scores``, ``leader``, ``mu``) is generated at once on the CPU;
    heatmaps are rendered on the device in fixed global blocks of ``block`` persons (``heatmaps(lo, hi)``
    renders any person range on any rank)."""

    def __init__(self, persons=104000, mean_group=20.0, joints=17, height=64, width=48, seed=12345,
                 dup_frac=0.3, jitter=0.3, box_jitter=0.5, noise=0.01, block=2048):
        g = _gen(seed, "cpu")
        images = max(1, int(persons / (1.0 + mean_group)))
        sizes = 1 + torch.poisson(torch.full((images,), float(mean_group)), generator=g).long()
        seg = torch.zeros(images + 1, dtype=torch.int64)
        seg[1:] = torch.cumsum(sizes, 0)
        n = int(seg[-1])
        self.seg = seg.numpy()
        self.persons, self.images = n, images
        self.joints, self.height, self.width = joints, height, width
        self.seed, self.noise, self.block = int(seed), noise, int(block)
        image_of = torch.repeat_interleave(torch.arange(images), sizes)
        first = seg[:-1][image_of]                                   # first person of each person's image
        pos = torch.arange(n) - first
        # a follower copies an EARLIER detection of its image (position 0 is always an original)
        is_dup = (torch.rand(n, generator=g) < dup_frac) & (pos > 0)
        pick = (torch.rand(n, generator=g) * pos.clamp(min=1).double()).long().clamp(max=(pos - 1).clamp(min=0))
        leader = torch.where(is_dup, first + pick, torch.arange(n))
        for _ in range(8):                                            # followers of followers -> the original
            leader = leader[leader]
        self.leader = leader
        boxes = detection_boxes(n, seed=seed + 1)
        boxes = boxes[leader] + torch.where(is_dup[:, None], box_jitter * torch.randn(n, 4, generator=g, dtype=torch.float64),
                                            torch.zeros(n, 4, dtype=torch.float64))
        self.boxes = boxes
        mu = peak_centres(n, joints, height, width, seed + 2, "cpu")
        mu = mu[leader] + torch.where(is_dup[:, None, None], jitter * torch.randn(n, joints, 2, generator=g), torch.zeros(n, joints, 2))
        mu[..., 0].clamp_(0, width - 1)
        mu[..., 1].clamp_(0, height - 1)
        self.mu = mu
        self.box_scores = (torch.randperm(n, generator=g).double() + 0.5) / n
        self.duplicates = int(is_dup.sum())

    def heatmaps(self, lo, hi, device):
        """float32 [hi-lo, K, H, W] on ``device`` for global persons [lo, hi)."""
        out = torch.empty((hi - lo, self.joints, self.height, self.width), dtype=torch.float32, device=device)
        b0 = lo // self.block
        while b0 * self.block < hi:
            s, e = b0 * self.block, min((b0 + 1) * self.block, self.persons)
            a, b = max(s, lo), min(e, hi)
            if b > a:
                maps = heatmaps_from_centres(self.mu[s:e].to(device), self.height, self.width, self.seed + 100 + b0, self.noise)
                out[a - lo:b - lo] = maps[a - s:b - s]
            b0 += 1
        return out


def table_checksum(rows):
    """Order-sensitive 64-bit digest of a float32 table (wrapping int64 arithmetic on the raw bits): equal
    digests across runs <=> bit-identical tables in the same row order (up to 2^-64 collisions)."""
    bits = rows.contiguous().view(torch.int32).to(torch.int64)
    n, w = bits.shape
    weight = (torch.arange(n, device=rows.device, dtype=torch.int64)[:, None] * 1000003 +
              torch.arange(w, device=rows.device, dtype=torch.int64)[None, :] * 7919 + 1)
    return int((bits * weight).sum().item())


def coco_keypoint_set(images=200, seed=0, variant="all", max_gt=4, fp=(0, 3), crowded_frac=0.05, zero_kp_frac=0.3):
    """A seeded COCO-shaped keypoint set for the COCO evaluator: (annotation dict, results list).

    Per image 0-``max_gt`` person GTs (normal ones with some unlabeled joints, ``zero_kp_frac`` with no keypoints,
    a few crowds; areas include exactly 32^2 and 96^2) and a non-person annotation now and then; per GT 0-3
    detections at graded distances (the ones of zero-keypoint GTs land around the box: the box-distance branch of
    computeOks), ``fp`` false positives per image, ``crowded_frac`` of the images with 25 more (over maxDets = 20);
    images with GT only and with detections only; scores with ties inside and across images, many exactly 0.0;
    detections whose keypoint extent is exactly 32 x 32 or 96 x 96. ``variant`` "medium" / "large" keeps every GT
    area inside [32^2, 96^2] / above 96^2, so that the other range has no GT. Image ids are not in sorted order in
    the ``images`` list; the results list is shuffled across images. Keypoints of results are float32 values."""
    import numpy as np
    rng = np.random.default_rng(seed)
    img_ids = (rng.permutation(3 * images)[:images] + 1).tolist()
    dataset = {"images": [{"id": i, "width": 640, "height": 480} for i in img_ids], "annotations": [],
               "categories": [{"id": 1, "name": "person"}]}
    results = []
    ann_id = 7

    def det(kps_xy, score, img):
        k = np.asarray(kps_xy, dtype=np.float32).reshape(17, 2)
        conf = rng.random(17).astype(np.float32)
        row = np.stack([k[:, 0], k[:, 1], conf], 1).reshape(-1)
        results.append({"image_id": img, "category_id": 1, "keypoints": [float(v) for v in row], "score": score})

    def score():
        u = rng.random()
        if u < 0.15:
            return 0.0
        if u < 0.55:
            return float(rng.integers(0, 21)) / 20.0
        return float(rng.random())

    for img in img_ids:
        kind = rng.random()
        n_gt = 0 if kind < 0.1 else int(rng.integers(1, max_gt + 1))
        gt_only = 0.1 <= kind < 0.18
        for _ in range(n_gt):
            u = rng.random()
            if variant == "medium":
                area = 1024.0 if u < 0.15 else float(rng.uniform(1100, 9100))
            elif variant == "large":
                area = float(rng.uniform(9300, 60000))
            else:
                area = 1024.0 if u < 0.05 else (9216.0 if u < 0.1 else float(rng.uniform(200, 60000)))
            ratio = rng.uniform(0.4, 1.0)
            bw, bh = math.sqrt(area * ratio), math.sqrt(area / ratio)
            bx, by = float(rng.uniform(0, 640 - bw)), float(rng.uniform(0, 480 - bh))
            t = rng.random()
            crowd = t < 0.05
            zero = (not crowd) and t < 0.05 + zero_kp_frac
            v = np.zeros(17, np.int64) if zero else rng.choice([0, 1, 2], 17, p=[0.3, 0.2, 0.5])
            if not zero and not v.any():
                v[0] = 2
            x = np.round(bx + rng.random(17) * bw)
            y = np.round(by + rng.random(17) * bh)
            x[v == 0] = 0
            y[v == 0] = 0
            kps = np.stack([x, y, v], 1).reshape(-1)
            dataset["annotations"].append({
                "id": ann_id, "image_id": img, "category_id": 1, "iscrowd": int(crowd), "area": area,
                "bbox": [bx, by, bw, bh], "num_keypoints": int((v > 0).sum()), "keypoints": [int(q) if q == int(q) else float(q) for q in kps]})
            ann_id += int(rng.integers(1, 4))
            if rng.random() < 0.1:
                dataset["annotations"].append({"id": ann_id, "image_id": img, "category_id": 3, "iscrowd": 0, "area": 50.0,
                                               "bbox": [0, 0, 5, 10], "num_keypoints": 0, "keypoints": [0] * 51})
                ann_id += 1
            if gt_only:
                continue
            base = np.stack([bx + rng.random(17) * bw, by + rng.random(17) * bh], 1)
            labelled = v > 0
            base[labelled, 0], base[labelled, 1] = x[labelled], y[labelled]
            for _d in range(int(rng.integers(0, 4))):
                if zero:            # around the box, partly outside it: the grown-box distance
                    xy = np.stack([rng.uniform(bx - 1.2 * bw, bx + 2.2 * bw, 17), rng.uniform(by - 1.2 * bh, by + 2.2 * bh, 17)], 1)
                else:
                    sigma = float(rng.choice([0.0, 0.01, 0.03, 0.06, 0.1, 0.2, 0.5])) * math.sqrt(area)
                    xy = base + rng.normal(0.0, 1.0, (17, 2)) * sigma
                det(xy, score(), img)
        if gt_only:
            continue
        n_fp = int(rng.integers(fp[0], fp[1] + 1)) + (25 if rng.random() < crowded_frac else 0)
        for _ in range(n_fp):
            u = rng.random()
            if u < 0.05:                # keypoint extent exactly 32 x 32 or 96 x 96
                side = 32.0 if rng.random() < 0.5 else 96.0
                x0, y0 = float(rng.integers(0, 500)), float(rng.integers(0, 350))
                xy = np.stack([x0 + rng.integers(0, int(side) + 1, 17), y0 + rng.integers(0, int(side) + 1, 17)], 1).astype(np.float64)
                xy[0] = (x0, y0)
                xy[1] = (x0 + side, y0 + side)
            else:
                cx, cy, s = rng.uniform(0, 640), rng.uniform(0, 480), rng.uniform(5, 200)
                xy = np.stack([cx + rng.normal(0, 1, 17) * s, cy + rng.normal(0, 1, 17) * s], 1)
            det(xy, score(), img)
    order = rng.permutation(len(results))
    return dataset, [results[i] for i in order]


def coco_results_arrays(results):
    """Results list -> (keypoints float32 [N, 51], scores float64 [N], image ids int64 [N]) as CPU tensors."""
    import numpy as np
    kps = np.array([r["keypoints"] for r in results], dtype=np.float32).reshape(-1, 51)
    scores = np.array([r["score"] for r in results], dtype=np.float64)
    ids = np.array([r["image_id"] for r in results], dtype=np.int64)
    return torch.from_numpy(kps), torch.from_numpy(scores), torch.from_numpy(ids)


def eval_set_ground_truth(es, keypoints, seed=0, jitter=2.0, zero_kp_frac=0.4):
    """COCO-shaped GT for an ``EvalSet``, so that the whole eval job can end in AP: image i has id i + 1; every
    original person of it (not a near-duplicate) becomes a GT whose keypoints are its decoded image-space
    keypoints (``keypoints`` [N, K, >=2], host) moved by N(0, jitter^2) px, its box the detection box;
    ``zero_kp_frac`` of them carry no keypoints. Returns (annotation dict, image ids [I])."""
    import numpy as np
    rng = np.random.default_rng(seed)
    kp = np.asarray(keypoints, dtype=np.float64)
    boxes = es.boxes.numpy()
    leader = es.leader.numpy()
    ids = np.arange(1, es.images + 1, dtype=np.int64)
    anns = []
    for i in range(es.images):
        for p in range(int(es.seg[i]), int(es.seg[i + 1])):
            if leader[p] != p:
                continue
            x1, y1, x2, y2 = (float(v) for v in boxes[p])
            w, h = max(x2 - x1, 1.0), max(y2 - y1, 1.0)
            zero = rng.random() < zero_kp_frac
            xy = kp[p, :, :2] + rng.normal(0.0, jitter, (kp.shape[1], 2))
            v = np.zeros(kp.shape[1]) if zero else np.full(kp.shape[1], 2.0)
            k = np.stack([np.where(v > 0, xy[:, 0], 0), np.where(v > 0, xy[:, 1], 0), v], 1).reshape(-1)
            anns.append({"id": len(anns) + 1, "image_id": int(ids[i]), "category_id": 1, "iscrowd": 0,
                         "area": w * h * 0.7, "bbox": [x1, y1, w, h], "num_keypoints": int((v > 0).sum()),
                         "keypoints": k.tolist()})
    return {"images": [{"id": int(i)} for i in ids], "annotations": anns}, ids
