"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's heatmap hot path.

Nothing in ``simple_pose_b200/`` imports this module. It exists so that the CUDA
path can be checked (``tests/``, ``__graft_entry__.smoke()``) and so that
``bench.py`` can time the reference's CPU algorithm next to the GPU numbers
(``cpu_baseline`` and ``--impl reference``). It is never the thing shipped.

Parity status: **pinned**. The reference has no tests of its own (SURVEY.md
section 4), so the pin is (a) ``tests/test_oracle_vs_reference.py`` which, in
the build container where ``/root/reference`` is mounted, runs the reference's
own functions (through ``oracle/ref_loader.py``) against every function below
and demands bit equality, and (b) the fixtures in ``tests/golden/`` generated
from the reference by ``oracle/make_golden.py`` which travel to the GPU box.

Each function cites the reference lines it restates (paths relative to the
reference root). The arithmetic (dtype promotions, operation order, library
calls) follows the reference so that results are bit-identical on CPU; the
code itself is written independently.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

COCO_JOINT_PAIRS = ((1, 2), (3, 4), (5, 6), (7, 8), (9, 10), (11, 12), (13, 14), (15, 16))
COCO_OKS_SIGMAS = np.array(
    [.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89]) / 10.0


# --------------------------------------------------------------------------- encode
def encode_person(joints, sigma=2.0, shape=(48, 64)):
    """DarkPose-style unbiased target encoder for one person.

    Restates ``RefineSimpleTransform.get_heat_map`` (commons/transforms.py:167-191).
    ``joints`` is [K,3] float32 (x, y, vis) in heatmap pixels, ``shape`` is (W, H).
    Returns (targets [K,H,W] float32, weights [K] float32).

    Arithmetic notes that matter for bit parity:
      * the cull test uses ``int()`` (truncation toward zero) of float32 expressions
        ``mu - 3*sigma`` and ``mu + 3*sigma + 1`` (transforms.py:181-182). With NumPy 2
        scalar promotion a float32 scalar combined with a Python float stays float32.
      * the Gaussian is evaluated in float64 over the *whole* map (int64 grid minus a
        float32 centre promotes to float64, transforms.py:188-190) and rounded to
        float32 on assignment.
    """
    joints = np.asarray(joints)
    width, height = int(shape[0]), int(shape[1])
    n = joints.shape[0]
    weights = np.array(joints[:, 2], copy=True)
    targets = np.zeros((n, height, width), dtype=np.float32)
    reach = sigma * 3
    cols = np.arange(width)
    rows = np.arange(height)
    for j in range(n):
        cx, cy = joints[j, 0], joints[j, 1]
        lo_x, lo_y = int(cx - reach), int(cy - reach)
        hi_x, hi_y = int(cx + reach + 1), int(cy + reach + 1)
        if lo_x >= width or lo_y >= height or hi_x < 0 or hi_y < 0:
            weights[j] = 0.
            continue
        if weights[j] > 0.5:
            gx, gy = np.meshgrid(cols, rows)
            grid = np.stack([gx, gy], axis=-1)
            centre = np.array([cx, cy])
            targets[j] = np.exp(-np.sum((grid - centre) ** 2, axis=-1) / (2 * sigma ** 2))
    return targets, weights


def encode_batch(joints, sigma=2.0, shape=(48, 64)):
    """[B,K,3] -> ([B,K,H,W], [B,K]); the stacking done by ``MSCOCO.collate_fn``
    (datasets/coco.py:138-146)."""
    joints = np.asarray(joints)
    maps, wts = [], []
    for b in range(joints.shape[0]):
        t, w = encode_person(joints[b], sigma, shape)
        maps.append(t)
        wts.append(w)
    return np.stack(maps), np.stack(wts)


def encode_person_basic(joints, sigma=2.0, shape=(48, 64), stride=4):
    """Quantised 13x13 encoder: ``BasicSimpleTransform.get_heat_map``
    (commons/transforms.py:80-116). ``joints`` are in *input* pixels."""
    joints = np.asarray(joints)
    width, height = int(shape[0]), int(shape[1])
    n = joints.shape[0]
    weights = np.array(joints[:, 2], copy=True)
    targets = np.zeros((n, height, width), dtype=np.float32)
    reach = sigma * 3
    side = 2 * reach + 1
    ax = np.arange(0, side, 1, np.float32)
    mid = side // 2
    patch = np.exp(-((ax[None, :] - mid) ** 2 + (ax[:, None] - mid) ** 2) / (2 * (sigma ** 2)))
    for j in range(n):
        mx = int(joints[j, 0] / stride + 0.5)
        my = int(joints[j, 1] / stride + 0.5)
        lo = (int(mx - reach), int(my - reach))
        hi = (int(mx + reach + 1), int(my + reach + 1))
        if lo[0] >= width or lo[1] >= height or hi[0] < 0 or hi[1] < 0:
            weights[j] = 0.
            continue
        px = (max(0, -lo[0]), min(hi[0], width) - lo[0])
        py = (max(0, -lo[1]), min(hi[1], height) - lo[1])
        ix = (max(0, lo[0]), min(hi[0], width))
        iy = (max(0, lo[1]), min(hi[1], height))
        if weights[j] > 0.5:
            targets[j, iy[0]:iy[1], ix[0]:ix[1]] = patch[py[0]:py[1], px[0]:px[1]]
    return targets, weights


# --------------------------------------------------------------------------- loss
def masked_mse_loss(pred, target, mask):
    """``0.5 * nn.MSELoss()(pred.mul(mask[..., None, None]), target.mul(mask[..., None, None]))``
    -- the inline expression of processors/dp_pose_hrnet_solver.py:86,106 (same in
    dp_pose_resnet_solver.py:107 and ddp_pose_resnet_solver.py:117). Mean over *all*
    B*K*H*W elements. Returns a 0-d tensor attached to ``pred``'s graph."""
    m = mask[..., None, None]
    return 0.5 * torch.nn.MSELoss()(pred.mul(m), target.mul(m))


def masked_mse_loss_and_grad(pred, target, mask):
    """Loss value and d loss / d pred via autograd of the expression above."""
    p = pred.detach().clone().requires_grad_(True)
    loss = masked_mse_loss(p, target, mask)
    loss.backward()
    return loss.detach(), p.grad.detach()


def masked_mse_loss_and_grad_scaled(pred, target, mask, scale=1.0):
    """The AMP branch, processors/dp_pose_hrnet_solver.py:111-120: ``pred`` is the autocast output (float16 or
    bfloat16), ``pred.mul(mask)`` promotes to float32 (as it does under autocast; ``mse_loss`` is on autocast's
    float32 list anyway), the loss is float32, and ``scaler.scale(loss).backward()`` sends ``scale`` as the upstream
    gradient: d loss / d pred comes back in ``pred``'s dtype, cast once after the scale has been applied in float32."""
    p = pred.detach().clone().requires_grad_(True)
    loss = masked_mse_loss(p, target, mask)
    (loss * scale).backward()
    return loss.detach(), p.grad.detach()


# --------------------------------------------------------------------------- decode
def argmax_coords(heat_map):
    """``BasicKeyPointDecoder.heat_map_to_axis`` (metrics/pose_metrics.py:11-24).

    [B,K,H,W] -> (coords [B,K,2] float32 as (x, y), max_val [B,K,1]). First maximal
    index on ties, NaN propagates (``torch.max`` semantics); x = idx % W and
    y = floor(idx / W) are computed in float32; both are zeroed when max_val <= 0."""
    b, k, h, w = heat_map.shape
    flat = heat_map.reshape(b, k, h * w)
    peak, where = flat.max(dim=-1, keepdim=True)
    xy = where.repeat(1, 1, 2).float()
    xy[..., 0] = xy[..., 0] % w
    xy[..., 1] = (xy[..., 1] / w).floor()
    xy = xy * (peak > 0.).repeat(1, 1, 2).float()
    return xy, peak


def argmax_index(heat_map):
    """Flat argmax index per (b,k) as int64 [B,K] (the integer the float coords of
    ``argmax_coords`` are derived from; used for the bit-exact index gate)."""
    b, k, h, w = heat_map.shape
    return heat_map.reshape(b, k, h * w).max(dim=-1)[1]


# cv::getGaussianKernel's fixed tables for sigma <= 0 and small odd sizes (OpenCV 4.x, imgproc/smooth;
# the 9-tap row exists since 4.5). The reference only ever uses 11, which takes the closed form.
_OPENCV_SMALL_GAUSSIAN = {
    1: [1.0],
    3: [0.25, 0.5, 0.25],
    5: [0.0625, 0.25, 0.375, 0.25, 0.0625],
    7: [0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125],
    9: [4.0 / 256, 13.0 / 256, 30.0 / 256, 51.0 / 256, 60.0 / 256, 51.0 / 256, 30.0 / 256, 13.0 / 256, 4.0 / 256],
}


def gaussian_taps(kernel_size=11):
    """1-D taps of ``cv.getGaussianKernel(kernel_size, 0)`` (metrics/pose_metrics.py:57): OpenCV's fixed
    tables for n <= 9, else sigma = 0.3*((n-1)*0.5-1)+0.8 and the normalised ``exp(-x^2/(2 sigma^2))``
    in float64. For n = 11 (sigma = 2.0) the float32 outer product is bit-equal to OpenCV 4.13's
    (checked in the tests; the fuzzer compares 3..13)."""
    n = int(kernel_size)
    if n in _OPENCV_SMALL_GAUSSIAN:
        return np.array(_OPENCV_SMALL_GAUSSIAN[n], dtype=np.float64)
    sigma = 0.3 * ((n - 1) * 0.5 - 1) + 0.8
    x = np.arange(n, dtype=np.float64) - (n - 1) * 0.5
    g = np.exp(-(x * x) / (2.0 * sigma * sigma))
    return g / g.sum()


def blur_weights(kernel_size=11):
    """float32 [n,n] = float32(k64 k64^T) (metrics/pose_metrics.py:57-60)."""
    k = gaussian_taps(kernel_size).reshape(-1, 1)
    return (k * k.T).astype(np.float32)


def gauss_taylor_decode(heat_map, trans_inv, kernel_size=11, return_heatmap_space=False):
    """``GaussTaylorKeyPointDecoder.__call__`` (metrics/pose_metrics.py:62-107), CPU.

    heat_map [B,K,H,W] float32, trans_inv [B,2,3] float32 ->
    (coords [B,K,2] float32 in image px, max_val [B,K,1] float32).
    Steps: argmax on the original map (:66); depthwise kxk blur with zero padding (:68);
    rescale by ori_max / blur_max, clamp at 1e-10, log (:71-73); for peaks with
    1 < x < W-2 and 1 < y < H-2 (:78) central differences of the log map (:80-93);
    keep those with dxx*dyy - dxy^2 != 0 (:94); offset = -H^-1 g through
    ``torch.inverse`` (:95-100); coords = clamp(coords + offset, min=0) for those
    joints only (:101-103); affine back-projection (:105-106)."""
    heat_map = heat_map.detach()
    b, k, h, w = heat_map.shape
    wts = torch.from_numpy(blur_weights(kernel_size))[None, None].repeat(k, 1, 1, 1)
    coords, peak = argmax_coords(heat_map)
    blurred = F.conv2d(heat_map, wts, bias=None, stride=1, padding=(kernel_size - 1) // 2, groups=k)
    ori_max = heat_map.reshape(b, k, -1).max(dim=-1)[0]
    blur_max = blurred.reshape(b, k, -1).max(dim=-1)[0]
    logmap = (blurred * ori_max[..., None, None] / blur_max[..., None, None]).clamp(min=1e-10).log()

    flat = logmap.reshape(b * k, h * w)
    xi = coords[..., 0].long().reshape(-1)
    yi = coords[..., 1].long().reshape(-1)
    inner = (xi > 1) & (xi < w - 2) & (yi > 1) & (yi < h - 2)
    rows = torch.nonzero(inner).reshape(-1)
    vx, vy = xi[rows], yi[rows]

    def at(dy, dx):
        return flat[rows, (vy + dy) * w + (vx + dx)]

    c = at(0, 0)
    dx = 0.5 * (at(0, 1) - at(0, -1))
    dy = 0.5 * (at(1, 0) - at(-1, 0))
    dxx = 0.25 * (at(0, 2) - 2 * c + at(0, -2))
    dxy = 0.25 * (at(1, 1) - at(-1, 1) - at(1, -1) + at(-1, -1))
    dyy = 0.25 * (at(2, 0) - 2 * c + at(-2, 0))
    solvable = dxx * dyy - dxy ** 2 != 0
    hess = torch.stack([torch.stack([dxx, dxy], dim=-1), torch.stack([dxy, dyy], dim=-1)], dim=-2)[solvable]
    grad = torch.stack([dx, dy], dim=-1).unsqueeze(-1)[solvable]
    step = (-hess.inverse() @ grad).transpose(1, 2).squeeze(1)
    out = coords.reshape(-1, 2).clone()
    refine_rows = rows[solvable]
    out[refine_rows] = (out[refine_rows] + step).clamp(min=0.)
    out = out.reshape(b, k, 2)
    if return_heatmap_space:
        return out, peak
    return back_project(out, trans_inv), peak


def back_project(coords, trans_inv):
    """Last two lines of both decoders (metrics/pose_metrics.py:50-51,105-106):
    out[b,c,a] = sum_d [x, y, 1][d] * trans_inv[b,a,d] via ``torch.einsum``."""
    homog = torch.cat([coords, torch.ones_like(coords[..., [0]])], dim=-1)
    return torch.einsum("bcd,bad->bca", homog, trans_inv)


def basic_decode(heat_map, trans_inv):
    """``BasicKeyPointDecoder.__call__`` (metrics/pose_metrics.py:26-52): argmax, then a
    quarter-pixel shift toward the larger neighbour for 1 < x < W-1, 1 < y < H-1."""
    heat_map = heat_map.detach()
    b, k, h, w = heat_map.shape
    coords, peak = argmax_coords(heat_map)
    flat = heat_map.reshape(b * k, h * w)
    xi = coords[..., 0].long().reshape(-1)
    yi = coords[..., 1].long().reshape(-1)
    inner = (xi > 1) & (xi < w - 1) & (yi > 1) & (yi < h - 1)
    rows = torch.nonzero(inner).reshape(-1)
    vx, vy = xi[rows], yi[rows]
    sx = (flat[rows, vy * w + vx + 1] - flat[rows, vy * w + vx - 1]).sign()
    sy = (flat[rows, (vy + 1) * w + vx] - flat[rows, (vy - 1) * w + vx]).sign()
    out = coords.reshape(-1, 2).clone()
    out[rows] = out[rows] + torch.stack([sx, sy], dim=-1) * 0.25
    return back_project(out.reshape(b, k, 2), trans_inv), peak


def dark_original_decode(heat_map, trans_inv, kernel_size=11):
    """``DarkPoseOriginalKeyPointDecoder.__call__`` (metrics/pose_metrics.py:110-169), the reference's
    NumPy/OpenCV decoder: argmax on the original map; per joint a zero-padded ``cv.GaussianBlur`` in
    float64 written back to the float32 map, ``*= origin_max / blurred_max`` in float32,
    ``log(maximum(., 1e-10))``; Taylor step with float32 scalars and ``np.matrix`` inverse when
    ``1 < px < W-2 and 1 < py < H-2`` and the determinant is non-zero; NO clamp at 0; float32
    ``einsum`` with ``trans_inv``. Works on a copy (the reference overwrites its input).
    heat_map [B,K,H,W] float32 tensor -> (coords [B,K,2] float32 tensor, max_val [B,K,1])."""
    import cv2 as cv
    coords, max_val = argmax_coords(heat_map)
    coords = coords.detach().cpu().numpy().copy()
    hm = heat_map.detach().cpu().numpy().copy()
    border = (kernel_size - 1) // 2
    b, k, h, w = hm.shape
    for i in range(b):
        for j in range(k):
            origin_max = np.max(hm[i, j])
            dr = np.zeros((h + 2 * border, w + 2 * border))
            dr[border:-border, border:-border] = hm[i, j].copy()
            dr = cv.GaussianBlur(dr, (kernel_size, kernel_size), 0)
            hm[i, j] = dr[border:-border, border:-border].copy()
            hm[i, j] *= origin_max / np.max(hm[i, j])
    hm = np.log(np.maximum(hm, 1e-10))
    for n in range(b):
        for p in range(k):
            m, c = hm[n][p], coords[n][p]
            px, py = int(c[0]), int(c[1])
            if 1 < px < w - 2 and 1 < py < h - 2:
                dx = 0.5 * (m[py][px + 1] - m[py][px - 1])
                dy = 0.5 * (m[py + 1][px] - m[py - 1][px])
                dxx = 0.25 * (m[py][px + 2] - 2 * m[py][px] + m[py][px - 2])
                dxy = 0.25 * (m[py + 1][px + 1] - m[py - 1][px + 1] - m[py + 1][px - 1] + m[py - 1][px - 1])
                dyy = 0.25 * (m[py + 2][px] - 2 * m[py][px] + m[py - 2][px])
                if dxx * dyy - dxy ** 2 != 0:
                    offset = -np.matrix([[dxx, dxy], [dxy, dyy]]).I * np.matrix([[dx], [dy]])
                    c += np.squeeze(np.array(offset.T), axis=0)
    xyz = np.concatenate([coords, np.ones_like(coords[..., [0]])], axis=-1)
    out = np.einsum("bcd,bad->bca", xyz, trans_inv.detach().cpu().numpy())
    return torch.from_numpy(out), max_val.detach().cpu()


# --------------------------------------------------------------------------- flip test
def swap_permutation(num_joints=17, joint_pairs=COCO_JOINT_PAIRS):
    """Channel permutation equivalent to the pair swap in ``flip_joints``
    (commons/joint_utils.py:109-111) with ``joint_pairs`` of datasets/coco.py:26."""
    perm = list(range(num_joints))
    for a, b in joint_pairs:
        perm[a], perm[b] = perm[b], perm[a]
    return perm


def flip_average(heat_map, heat_map_flip, joint_pairs=COCO_JOINT_PAIRS):
    """NOT IN THE REFERENCE (SURVEY.md section 8a row A6) -- composed from its primitives:
    avg[b,k,y,x] = 0.5 * (hm[b,k,y,x] + hm_flip[b,perm[k],y,W-1-x]); pure mirror
    ``x -> W-1-x`` and pair swap as in ``flip_joints`` (commons/joint_utils.py:102-112),
    no 1-px shift."""
    perm = swap_permutation(heat_map.shape[1], joint_pairs)
    return 0.5 * (heat_map + heat_map_flip.flip(-1)[:, perm])


def flip_decode(heat_map, heat_map_flip, trans_inv, joint_pairs=COCO_JOINT_PAIRS, kernel_size=11,
                return_heatmap_space=False):
    return gauss_taylor_decode(flip_average(heat_map, heat_map_flip, joint_pairs), trans_inv,
                               kernel_size, return_heatmap_space)


# --------------------------------------------------------------------------- OKS / NMS
def oks_similarity(pick_kps, cand_kps, pick_area, cand_area, sigmas=None, in_vis_thresh=None):
    """``oks_iou`` (datasets/naive_data.py:120-150). pick [K,3], cand [n,K,3] -> [n] float64.
    e = (dx^2+dy^2)/var/((a_p+a_c)/2 + 1e-12)/2 ; oks = sum(exp(-e)*vis)/(sum(vis)+1e-12);
    vis is float32 ones unless a visibility threshold is given."""
    if not isinstance(sigmas, np.ndarray):
        sigmas = COCO_OKS_SIGMAS
    var = (sigmas * 2) ** 2
    dx = cand_kps[..., 0] - pick_kps[:, 0]
    dy = cand_kps[..., 1] - pick_kps[:, 1]
    e = (dx ** 2 + dy ** 2) / var / ((pick_area + cand_area)[:, None] / 2 + 1e-12) / 2
    vis = np.ones_like(cand_kps[..., 2], dtype=np.float32)
    if in_vis_thresh is not None:
        pick_vis = np.tile((pick_kps[:, 2] > in_vis_thresh)[None, :], (cand_kps.shape[0], 1))
        vis = ((cand_kps[..., 2] > in_vis_thresh) & pick_vis).astype(np.float32)
    return (np.exp(-e) * vis).sum(-1) / (vis.sum(-1) + 1e-12)


def oks_greedy_nms(kps, scores, areas, thresh, sigmas=None, in_vis_thresh=None):
    """``oks_nms`` (datasets/naive_data.py:153-173): visit persons by descending score
    (``argsort()[::-1]``), keep the head, drop every remaining one whose OKS with it is
    > thresh. Returns the kept indices in pick order."""
    pending = scores.argsort()[::-1]
    kept = []
    while pending.size > 0:
        head = pending[0]
        kept.append(head)
        pending = pending[1:]
        if pending.size == 0:
            break
        sim = oks_similarity(kps[head], kps[pending], areas[head], areas[pending], sigmas, in_vis_thresh)
        pending = pending[sim <= thresh]
    return kept


def rescore_person(box_score, kps, in_vis_thre=0.2):
    """eval.py:168-175: score = box_score * mean(joint_score[joint_score > thr]) (0 if none)."""
    js = np.asarray(kps, dtype=np.float64).reshape(-1, 3)[:, -1]
    sel = js > in_vis_thre
    mean = js[sel].mean() if sel.sum() > 0 else 0.
    return box_score * mean


def rescore_and_nms(kps, box_scores, areas, seg_offsets, in_vis_thre=0.2, oks_thre=0.9):
    """eval.py:153-197 without the JSON round trip: per image (segment) rescore, run
    ``oks_nms`` and return (keep mask [N] bool, scores [N] float64, kept index lists)."""
    kps = np.asarray(kps, dtype=np.float64)
    n = kps.shape[0]
    scores = np.array([rescore_person(box_scores[i], kps[i], in_vis_thre) for i in range(n)], dtype=np.float64)
    keep = np.zeros(n, dtype=bool)
    picks = []
    for s in range(len(seg_offsets) - 1):
        lo, hi = int(seg_offsets[s]), int(seg_offsets[s + 1])
        if hi <= lo:
            picks.append([])
            continue
        sel = oks_greedy_nms(kps[lo:hi], scores[lo:hi], np.asarray(areas[lo:hi], dtype=np.float64), oks_thre)
        sel = [int(i) + lo for i in sel]
        keep[sel] = True
        picks.append(sel)
    return keep, scores, picks


# --------------------------------------------------------------------------- accuracy metric
def heat_map_acc(predicts, targets, distance_thresh=0.5, norm_frac=10.):
    """``HeatMapAcc.__call__`` (metrics/pose_metrics.py:212-245): per-joint fraction of
    persons whose argmax lies within ``distance_thresh`` (in units of (W,H)/norm_frac) of the
    target argmax, over persons whose target argmax has x > 1 and y > 1; averaged over joints
    that have at least one such person."""
    p, _ = argmax_coords(predicts)
    t, _ = argmax_coords(targets)
    return heat_map_acc_from_axes(p, t, predicts.shape[-2], predicts.shape[-1], distance_thresh, norm_frac)


def heat_map_acc_from_axes(p, t, height, width, distance_thresh=0.5, norm_frac=10.):
    """The epilogue of ``heat_map_acc`` (metrics/pose_metrics.py:225-245) on the two [B,K,2] float32
    ``argmax_coords`` tables ``p`` (predictions) and ``t`` (targets) of [B,K,height,width] maps."""
    norm = torch.tensor([width, height], dtype=torch.float) / norm_frac
    ok = (t[..., 0] > 1) & (t[..., 1] > 1)
    dist = torch.norm(p / norm - t / norm, dim=-1)
    dist[~ok] = -1.
    total, used = 0., 0.
    for j in range(dist.shape[1]):
        dj, oj = dist.T[j], ok.T[j]
        if oj.sum().item() < 1:
            continue
        total = total + (dj[oj] < distance_thresh).sum().float() / (oj.sum())
        used += 1
    if used > 0:
        return total / used
    return torch.tensor(0.)


def kps_score(max_val):
    """Person score of ``kps_to_dict_`` (metrics/pose_metrics.py:176): mean + max of the
    joint peak values. max_val [B,K,1] -> [B]."""
    return max_val.mean(dim=(1, 2)) + max_val.amax(dim=(1, 2))


# --------------------------------------------------------------------------- box -> affine (eval-side caller)
def box_center_scale(x, y, w, h, aspect_ratio=1.0, scale_mult=1.25):
    """``box_to_center_scale`` (commons/joint_utils.py:39-56). x, y, w, h are Python floats
    (float64 arithmetic); centre and scale are float32 arrays; ``scale * scale_mult`` is a
    float32 multiplication (NumPy 2 keeps float32 for array * Python scalar)."""
    center = np.zeros(2, dtype=np.float32)
    center[0] = x + w * 0.5
    center[1] = y + h * 0.5
    if w > aspect_ratio * h:
        h = w / aspect_ratio
    elif w < aspect_ratio * h:
        w = h * aspect_ratio
    scale = np.array([w, h], dtype=np.float32)
    if center[0] != -1:
        scale = scale * np.float32(scale_mult)
    return center, scale


def affine_triangles(center, scale, output_size, rot=0.0):
    """The two point triples of ``get_affine_transform(center, scale, rot, output_size)``
    (commons/joint_utils.py:115-150) for shift = 0, as float32 [3,2] arrays. ``rot`` is a Python
    float in degrees: ``rot_rad = np.pi * rot / 180`` and ``get_dir`` (:78-85) are float64
    (``0 * cs - p * sn``, ``0 * sn + p * cs`` with p = float32 ``src_w * -0.5`` promoted), the
    second points are float64 sums rounded to float32 (float32 array + list of float64), the third
    points float32 arithmetic (``get_3rd_point`` :72-75). NumPy >= 2 promotion rules (a Python
    scalar never widens a float32)."""
    center = np.asarray(center, dtype=np.float32)
    src_w = np.float32(scale[0])
    dst_w, dst_h = output_size[0], output_size[1]
    half = np.float64(src_w * np.float32(-0.5))                  # src_w * -0.5 stays float32, then float64 in get_dir
    rot_rad = np.pi * float(rot) / 180
    sn, cs = np.sin(rot_rad), np.cos(rot_rad)
    dir_x = 0 * cs - half * sn
    dir_y = 0 * sn + half * cs
    src = np.zeros((3, 2), dtype=np.float32)
    dst = np.zeros((3, 2), dtype=np.float32)
    src[0] = center
    src[1, 0] = np.float64(center[0]) + dir_x
    src[1, 1] = np.float64(center[1]) + dir_y
    dst[0] = [dst_w * 0.5, dst_h * 0.5]
    dst[1, 0] = dst_w * 0.5 + 0.0
    dst[1, 1] = dst_h * 0.5 + np.float64(np.float32(dst_w * -0.5))
    for tri in (src, dst):
        direct = tri[0] - tri[1]
        tri[2] = tri[1] + np.array([-direct[1], direct[0]], dtype=np.float32)
    return src, dst


def solve_affine_lu(p_from, p_to):
    """``cv.getAffineTransform(p_from, p_to)`` restated: OpenCV (pinned by the reference only as
    ``opencv-python``, README.md:12; 4.13.0 here) fills the 6x6 system
    [x y 1 0 0 0; 0 0 0 x y 1] m = (x', y') per point in float64 and solves it with its in-place
    partial-pivot LU (first row of maximal |pivot|, ``d = -1/pivot``, ``row_j += (a_ji * d) * row_i``,
    back substitution ``(b_i - sum a_ik x_k) / a_ii``), no fused multiply-add. Bit-identical to
    cv2 on every probe (tests/test_oracle_vs_reference.py). Returns float64 [2,3]."""
    a = np.zeros((6, 6), dtype=np.float64)
    b = np.zeros(6, dtype=np.float64)
    for i in range(3):
        px, py = float(p_from[i][0]), float(p_from[i][1])
        a[2 * i, 0:3] = (px, py, 1.0)
        a[2 * i + 1, 3:6] = (px, py, 1.0)
        b[2 * i] = float(p_to[i][0])
        b[2 * i + 1] = float(p_to[i][1])
    n = 6
    for i in range(n):
        k = i
        for j in range(i + 1, n):
            if abs(a[j, i]) > abs(a[k, i]):
                k = j
        if abs(a[k, i]) < np.finfo(np.float64).eps * 100:
            return np.zeros((2, 3), dtype=np.float64)            # singular: OpenCV leaves the result zero
        if k != i:
            a[[i, k]] = a[[k, i]]
            b[[i, k]] = b[[k, i]]
        d = -1.0 / a[i, i]
        for j in range(i + 1, n):
            alpha = a[j, i] * d
            for c in range(i + 1, n):
                a[j, c] = a[j, c] + alpha * a[i, c]
            b[j] = b[j] + alpha * b[i]
    x = np.zeros(n, dtype=np.float64)
    for i in range(n - 1, -1, -1):
        s = b[i]
        for k in range(i + 1, n):
            s = s - a[i, k] * x[k]
        x[i] = s / a[i, i]
    return x.reshape(2, 3)


def affine_pair(center, scale, output_size, rot=0.0):
    """(trans, trans_inv) of ``get_affine_transform(center, scale, rot, output_size)``, float64 [2,3]."""
    src, dst = affine_triangles(center, scale, output_size, rot)
    return solve_affine_lu(src, dst), solve_affine_lu(dst, src)


def box_affines(boxes_xyxy, input_shape=(192, 256), output_shape=(48, 64), scale_mult=1.25):
    """``BasicTransform.__call__`` without the image warp (datasets/naive_data.py:44-56) for a list
    of detection boxes [x1, y1, x2, y2] (Python floats): centre, scale, area = scale_w * scale_h
    (float32 product) and the heatmap -> image affine ``trans_inv`` as the collate function ships
    it (``.float()``, :114-116). Returns float32 arrays center [P,2], scale [P,2], area [P],
    trans_inv [P,2,3]."""
    ratio = input_shape[0] / input_shape[1]
    n = len(boxes_xyxy)
    center = np.zeros((n, 2), np.float32)
    scale = np.zeros((n, 2), np.float32)
    area = np.zeros(n, np.float32)
    tinv = np.zeros((n, 2, 3), np.float32)
    for i, (x1, y1, x2, y2) in enumerate(boxes_xyxy):
        x1, y1, x2, y2 = float(x1), float(y1), float(x2), float(y2)
        c, s = box_center_scale(x1, y1, x2 - x1, y2 - y1, ratio, scale_mult)
        _, ti = affine_pair(c, s, output_shape)
        center[i], scale[i], area[i] = c, s, s[0] * s[1]
        tinv[i] = ti.astype(np.float32)
    return center, scale, area, tinv


# --------------------------------------------------------------------------- train-side caller of the encoder
def flip_joints_only(joints, width, joint_pairs=COCO_JOINT_PAIRS):
    """Joint half of ``flip_joints`` (commons/joint_utils.py:102-112): ``x -> width - x - 1`` in
    float32 (``width`` is a Python int, so both subtractions stay float32) for EVERY row, visible or
    not, then whole rows (x, y, vis) of each pair are swapped."""
    out = np.array(joints, dtype=np.float32, copy=True)
    out[:, 0] = np.float32(width) - out[:, 0] - np.float32(1)
    for a, b in joint_pairs:
        out[[a, b]] = out[[b, a]]
    return out


def affine_joints(joints, t):
    """``affine_transform_batch`` (commons/joint_utils.py:88-99): rows with vis > 0 are mapped by
    ``[x, y, 1] . t.T`` -- float32 operands promoted to float64, ``np.dot`` (OpenBLAS dgemm, which
    on FMA hardware accumulates ``fma(1, t2, fma(y, t1, x*t0))``; probe in DESIGN.md) -- and rounded
    back into the float32 joint array; the other rows are left alone."""
    out = np.array(joints, dtype=np.float32, copy=True)
    vis = out[:, 2] > 0
    homog = np.concatenate([out[vis, :2], np.ones_like(out[vis, 0:1])], axis=-1)
    out[vis, :2] = np.dot(homog, np.asarray(t).T)
    return out


def train_sample_geometry(box, img_w, joints, scale_ratio=1.0, rot=0.0, flip=False,
                          joint_pairs=COCO_JOINT_PAIRS, input_shape=(192, 256), output_shape=(48, 64),
                          sigma=2.0, basic=False):
    """``RefineSimpleTransform.__call__`` (commons/transforms.py:193-223) without the image work
    (``cv.warpAffine``, ``np.fliplr``) and with its random draws passed in: ``box`` is the box AFTER
    ``box_crop`` (four Python floats), ``scale_ratio`` / ``rot`` / ``flip`` are the three draws of
    :204-211. Returns a dict with the reference's per-sample products: ``center``, ``scale``
    (float32 [2], after augmentation), ``img_trans`` (float64 [2,3], what the image warp uses),
    ``trans_inv`` (float64 [2,3], ``joint_info.trans_inv``), ``joints_input`` (``joint_info.joints``),
    ``joints_hm`` (the encoder's input), ``heat_map`` [K,H,W], ``mask`` [K]."""
    x1, y1, x2, y2 = (float(v) for v in box)
    ratio = input_shape[0] / input_shape[1]
    center, scale = box_center_scale(x1, y1, x2 - x1, y2 - y1, ratio)
    scale = scale * np.float32(scale_ratio)                      # float32 array * Python float
    joints = np.array(joints, dtype=np.float32, copy=True)
    if flip:
        joints = flip_joints_only(joints, img_w, joint_pairs)
        center[0] = np.float32(img_w) - center[0] - np.float32(1)
    img_trans, _ = affine_pair(center, scale, input_shape, rot)
    joint_trans, trans_inv = affine_pair(center, scale, output_shape, rot)
    joints_input = affine_joints(joints, img_trans)
    joints_hm = affine_joints(joints, joint_trans)
    if basic:       # BasicSimpleTransform.__call__ (:118-148): quantised encoder on the INPUT-pixel joints, stride 4
        heat_map, mask = encode_person_basic(joints_input, sigma, output_shape, 4)
    else:
        heat_map, mask = encode_person(joints_hm, sigma, output_shape)
    return {"center": center, "scale": scale, "img_trans": img_trans, "joint_trans": joint_trans,
            "trans_inv": trans_inv, "joints_input": joints_input, "joints_hm": joints_hm,
            "heat_map": heat_map, "mask": mask}


def kps_to_dict(predicts, scores, img_ids, out_list):
    """``kps_to_dict_`` (metrics/pose_metrics.py:172-179): per person, score = mean + max of the joint peaks
    (float32 torch reductions over the [K,1] slice), keypoints = (x, y, peak) * K as Python floats."""
    for pd, sc, img_id in zip(predicts, scores, img_ids):
        out_list.append({"image_id": img_id, "score": float((sc.mean() + sc.max()).item()), "category_id": 1,
                         "keypoints": torch.cat([pd, sc], dim=-1).reshape(-1).cpu().tolist()})



def detie_scores(scores):
    """Distinct scores with the same ordering as ``scores`` where, among EQUAL values, the higher index ranks
    higher -- the visiting order ``argsort()[::-1]`` yields when the sort underneath is stable. Not part of the
    reference: ``oks_nms`` (datasets/naive_data.py:163) leaves the order of equal scores to ``numpy.argsort``'s
    default (unstable) sort, whose tie order depends on NumPy's SIMD dispatch for the host CPU (on AVX-512 /
    AVX2 builds even two equal scores among eight may swap). Feeding these scores to the reference removes
    that freedom; the CUDA kernel's documented rule is exactly this order."""
    scores = np.asarray(scores, dtype=np.float64)
    order = np.lexsort((np.arange(scores.shape[0]), scores))        # ascending score, then ascending index
    out = np.empty_like(scores)
    out[order] = (np.arange(scores.shape[0], dtype=np.float64) + 1.0) / (scores.shape[0] + 1.0)
    return out
