// A11: COCO keypoint evaluation, pycocotools' COCOeval(iouType='keypoints') with its keypoint defaults
// (eval.py:13-27, metrics/pose_metrics.py:182-209): evaluate() + accumulate() + the statistics of summarize().
// oracle/coco_eval_oracle.py restates the Python operation by operation; every float64 operation below keeps
// its order (__d*_rn, so that nvcc contracts nothing into an FMA).
//
// Six launches, no host synchronisation:
//   1. keys: each detection's image position (or "not evaluated") and its index;
//   2. CUB radix sort by image position -- stable, so an image's detections keep their input order;
//   3. one warp per image: rank the image's detections by score (stable) and keep the first 20, their
//      keypoint-extent areas, the [<= 20, G] OKS matrix (computeOks), then evaluateImg's greedy matching with
//      one lane per (area range, IoU threshold) pair; per detection slot (image * 20 + rank) a sort key and the
//      matched / ignored bit of each of the 30 lanes, per image the evaluated count and the non-ignored GT count
//      of each area range;
//   4. CUB radix sort of the slots by descending score. Slots are laid out by (image position, rank), and the
//      sort is stable, so the order is (score descending, image position, rank): accumulate()'s stable sort of
//      the detections concatenated in imgIds order;
//   5. one CTA per (threshold, area range): tp / fp counts, recall, precision made monotone from the right
//      (one backward pass that carries the suffix counts and the suffix maximum) and the 101 searchsorted
//      lookups;
//   6. the ten summary means in NumPy's pairwise summation order.
#include "sp_common.cuh"
#include "sp_numpy_sum.cuh"
#include <cfloat>
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <math_constants.h>

namespace {

constexpr int kK = 17, kT = 10, kR = 101, kA = 3, kMaxDets = 20;
constexpr int kLanes = kT * kA;                  // matching lanes of a warp: lane = area * kT + threshold
constexpr int kImgWarps = 4;
constexpr int kAccThreads = 512;
constexpr unsigned long long kNoDet = ~0ull;     // sort key of an unused slot: after every detection

__device__ __constant__ double kCocoSigmas[kK] = {.26, .25, .25, .35, .35, .79, .79, .72, .72,
                                                  .62, .62, 1.07, 1.07, .87, .87, .89, .89};

// GT flag bits (set on the host by _prepare's rule)
constexpr unsigned char kGtIgnore = 1;           // iscrowd or num_keypoints == 0
constexpr unsigned char kGtCrowd = 2;

// Sort key of a score: ascending key order = descending score order, +0.0 and -0.0 equal (as NumPy compares).
__device__ __forceinline__ unsigned long long desc_score_key(double s) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(__dadd_rn(s, 0.0));
    const unsigned long long ord = (u >> 63) ? ~u : (u | (1ull << 63));
    return ~ord;
}

__global__ void __launch_bounds__(256)
coco_det_keys_kernel(const int* __restrict__ det_img, const unsigned char* __restrict__ keep, int n, int images,
                     unsigned* __restrict__ keys, int* __restrict__ idx) {
    sp::grid_dep_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int im = det_img[i];
    const bool use = (keep == nullptr || keep[i] != 0) && im >= 0 && im < images;
    keys[i] = use ? (unsigned)im : (unsigned)images;
    idx[i] = i;
}

// computeOks for one (detection, GT) pair. d: the detection's row (x at 3k, y at 3k+1, float32); g: the GT's
// (x, y, v) * 17 in float64; bb: its (x, y, w, h).
__device__ __forceinline__ double coco_oks(const float* __restrict__ d, const double* __restrict__ g, double area,
                                        const double* __restrict__ bb) {
    int k1 = 0;
    for (int k = 0; k < kK; ++k) k1 += g[3 * k + 2] > 0.0;
    const double x0 = __dsub_rn(bb[0], bb[2]), x1 = __dadd_rn(bb[0], __dmul_rn(bb[2], 2.0));
    const double y0 = __dsub_rn(bb[1], bb[3]), y1 = __dadd_rn(bb[1], __dmul_rn(bb[3], 2.0));
    const double den = __dadd_rn(area, DBL_EPSILON);             // gt['area'] + np.spacing(1)
    const int cnt = k1 > 0 ? k1 : kK;
    sp::NumpySum acc;
    acc.begin(cnt);
    for (int k = 0; k < kK; ++k) {
        if (k1 > 0 && !(g[3 * k + 2] > 0.0)) continue;            // e = e[vg > 0]
        const double xd = (double)d[3 * k], yd = (double)d[3 * k + 1];
        double dx, dy;
        if (k1 > 0) {
            dx = __dsub_rn(xd, g[3 * k]);
            dy = __dsub_rn(yd, g[3 * k + 1]);
        } else {                                                   // distance to the grown GT box
            const double ax = __dsub_rn(x0, xd), bx = __dsub_rn(xd, x1);
            const double ay = __dsub_rn(y0, yd), by = __dsub_rn(yd, y1);
            dx = __dadd_rn(ax > 0.0 ? ax : 0.0, bx > 0.0 ? bx : 0.0);
            dy = __dadd_rn(ay > 0.0 ? ay : 0.0, by > 0.0 ? by : 0.0);
        }
        const double s = __ddiv_rn(kCocoSigmas[k], 10.0);
        const double t = __dmul_rn(s, 2.0);
        double e = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
        e = __ddiv_rn(__ddiv_rn(__ddiv_rn(e, __dmul_rn(t, t)), den), 2.0);
        acc.push(exp(-e));
    }
    return __ddiv_rn(acc.result(), (double)cnt);
}

__device__ __forceinline__ int lower_bound_u32(const unsigned* __restrict__ a, int n, unsigned v) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

struct GtView {
    const double* kps;      // [G, 51]
    const double* area;     // [G]
    const double* bbox;     // [G, 4]
    const unsigned char* flags;
    const int* seg;         // [I + 1]
};

// One warp per image: computeOks + evaluateImg for the three area ranges and ten thresholds.
__global__ void __launch_bounds__(kImgWarps * 32)
coco_image_kernel(const float* __restrict__ rows, int stride, const double* __restrict__ scores,
                  const unsigned* __restrict__ det_img_sorted, const int* __restrict__ det_sorted, int n_dets,
                  GtView gt, int images, const double* __restrict__ iou_thrs, const double* __restrict__ area_rng,
                  double* __restrict__ oks, unsigned char* __restrict__ gtm, int4* __restrict__ img_info,
                  unsigned long long* __restrict__ slot_key, unsigned long long* __restrict__ slot_flags,
                  int* __restrict__ slot_det) {
    __shared__ int s_det[kImgWarps][kMaxDets];
    __shared__ double s_area[kImgWarps][kMaxDets];
    sp::grid_dep_wait();
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int img = blockIdx.x * kImgWarps + w;
    if (img >= images) return;                                    // whole warps leave together

    // the image's detections, in input order (the sort by image position is stable)
    const int lo = lower_bound_u32(det_img_sorted, n_dets, (unsigned)img);
    const int n = lower_bound_u32(det_img_sorted, n_dets, (unsigned)img + 1u) - lo;
    // argsort(-score, kind='mergesort')[:20]: rank = #(higher score) + #(equal score earlier in the input)
    for (int j = lane; j < n; j += 32) {
        const int dj = det_sorted[lo + j];
        const double sj = scores[dj];
        int r = 0;
        for (int k = 0; k < n && r < kMaxDets; ++k) {
            const double sk = scores[det_sorted[lo + k]];
            r += (sk > sj) || (sk == sj && k < j);
        }
        if (r < kMaxDets) s_det[w][r] = dj;
    }
    __syncwarp();
    const int D = n < kMaxDets ? n : kMaxDets;
    if (lane < D) {                                               // loadRes: area of the keypoint extent
        const float* row = rows + (size_t)s_det[w][lane] * stride;
        double x0 = row[0], x1 = row[0], y0 = row[1], y1 = row[1];
        for (int k = 1; k < kK; ++k) {
            const double x = row[3 * k], y = row[3 * k + 1];
            x0 = x < x0 ? x : x0;
            x1 = x > x1 ? x : x1;
            y0 = y < y0 ? y : y0;
            y1 = y > y1 ? y : y1;
        }
        s_area[w][lane] = __dmul_rn(__dsub_rn(x1, x0), __dsub_rn(y1, y0));
    }
    if (lane < kMaxDets) {
        const size_t slot = (size_t)img * kMaxDets + lane;
        slot_key[slot] = lane < D ? desc_score_key(scores[s_det[w][lane]]) : kNoDet;
        if (slot_det) slot_det[slot] = lane < D ? s_det[w][lane] : -1;
    }
    __syncwarp();

    // the [D, G] OKS matrix, row-major, at oks + 20 * (first GT of the image)
    const int g0 = gt.seg[img], G = gt.seg[img + 1] - g0;
    double* O = oks + (size_t)kMaxDets * g0;
    for (int idx = lane; idx < D * G; idx += 32) {
        const int r = idx / G, g = idx - r * G;
        O[idx] = coco_oks(rows + (size_t)s_det[w][r] * stride, gt.kps + (size_t)(g0 + g) * 3 * kK, gt.area[g0 + g],
                          gt.bbox + (size_t)(g0 + g) * 4);
    }
    __syncwarp();

    // evaluateImg, one lane per (area range, threshold). A lane walks its GTs in mergesort(_ignore) order --
    // the non-ignored ones in file order, then the ignored ones in file order -- and keeps its own gtm row.
    const bool active = lane < kLanes;
    const int a = lane / kT, t = lane - a * kT;
    double a_lo = 0.0, a_hi = 0.0, thr = 0.0;
    unsigned char* M = gtm + (size_t)kLanes * g0 + (size_t)lane * G;
    int npig = 0;
    if (active) {
        a_lo = area_rng[2 * a];
        a_hi = area_rng[2 * a + 1];
        thr = iou_thrs[t];
        for (int g = 0; g < G; ++g) {
            M[g] = 0;
            const double ga = gt.area[g0 + g];
            npig += !((gt.flags[g0 + g] & kGtIgnore) || ga < a_lo || ga > a_hi);
        }
    }
    for (int d = 0; d < D; ++d) {
        bool matched = false, dt_ignored = false;
        if (active) {
            double iou = fmin(thr, 1.0 - 1e-10);
            int m = -1;
            bool m_ig = false;
            for (int pass = 0; pass < 2; ++pass) {
                // at the first ignored GT while holding a non-ignored match: stop
                if (pass == 1 && m > -1 && !m_ig) break;
                for (int g = 0; g < G; ++g) {
                    const unsigned char f = gt.flags[g0 + g];
                    const double ga = gt.area[g0 + g];
                    const bool ig = (f & kGtIgnore) || ga < a_lo || ga > a_hi;
                    if (ig != (pass == 1)) continue;
                    if (M[g] && !(f & kGtCrowd)) continue;        // already matched, not a crowd
                    const double o = O[d * G + g];
                    if (o < iou) continue;
                    iou = o;                                      // equal OKS: the later GT takes the match
                    m = g;
                    m_ig = ig;
                }
            }
            if (m > -1) {
                matched = true;
                dt_ignored = m_ig;
                M[m] = 1;
            } else {
                const double da = s_area[w][d];
                dt_ignored = da < a_lo || da > a_hi;
            }
        }
        const unsigned mb = __ballot_sync(SP_FULL, matched);
        const unsigned ib = __ballot_sync(SP_FULL, dt_ignored);
        if (lane == 0) slot_flags[(size_t)img * kMaxDets + d] = ((unsigned long long)ib << 32) | mb;
    }
    if (lane >= D && lane < kMaxDets) slot_flags[(size_t)img * kMaxDets + lane] = 0ull;
    const int n0 = __shfl_sync(SP_FULL, npig, 0), n1 = __shfl_sync(SP_FULL, npig, kT), n2 = __shfl_sync(SP_FULL, npig, 2 * kT);
    if (lane == 0) img_info[img] = make_int4(D, n0, n1, n2);
}

struct MaxOp {
    __device__ __forceinline__ double operator()(double x, double y) const { return x > y ? x : y; }
};

// accumulate() for one (threshold, area range): blockIdx.x = area * kT + threshold.
__global__ void __launch_bounds__(kAccThreads)
coco_accumulate_kernel(const int4* __restrict__ img_info, int images, const unsigned long long* __restrict__ flags,
                       const double* __restrict__ rec_thrs, double* __restrict__ precision, double* __restrict__ recall) {
    using ReduceI = cub::BlockReduce<int, kAccThreads>;
    using ScanI = cub::BlockScan<int, kAccThreads>;
    using ScanD = cub::BlockScan<double, kAccThreads>;
    __shared__ union {
        typename ReduceI::TempStorage reduce;
        typename ScanI::TempStorage scan_i;
        typename ScanD::TempStorage scan_d;
    } tmp;
    __shared__ double s_q[kR], s_thr[kR];
    __shared__ int s_tot[4];
    sp::grid_dep_wait();
    const int tid = threadIdx.x;
    const int lane_id = blockIdx.x, a = lane_id / kT, t = lane_id - a * kT;

    int nd = 0, np = 0;
    for (int i = tid; i < images; i += kAccThreads) {
        const int4 v = img_info[i];
        nd += v.x;
        np += a == 0 ? v.y : (a == 1 ? v.z : v.w);
    }
    nd = ReduceI(tmp.reduce).Sum(nd);
    __syncthreads();
    np = ReduceI(tmp.reduce).Sum(np);
    if (tid == 0) { s_tot[0] = nd; s_tot[1] = np; }
    for (int k = tid; k < kR; k += kAccThreads) { s_q[k] = 0.0; s_thr[k] = rec_thrs[k]; }
    __syncthreads();
    nd = s_tot[0];
    const int npig = s_tot[1];
    if (npig == 0) {                                              // precision and recall stay -1
        for (int k = tid; k < kR; k += kAccThreads) precision[(t * kR + k) * kA + a] = -1.0;
        if (tid == 0) recall[t * kA + a] = -1.0;
        return;
    }
    // totals: tps = dtm & ~dtIg, fps = ~dtm & ~dtIg
    int tpc = 0, fpc = 0;
    for (int p = tid; p < nd; p += kAccThreads) {
        const unsigned long long f = flags[p];
        const int m = (int)((f >> lane_id) & 1ull), ig = (int)((f >> (32 + lane_id)) & 1ull);
        tpc += m & (ig ^ 1);
        fpc += (m ^ 1) & (ig ^ 1);
    }
    __syncthreads();
    tpc = ReduceI(tmp.reduce).Sum(tpc);
    __syncthreads();
    fpc = ReduceI(tmp.reduce).Sum(fpc);
    if (tid == 0) { s_tot[2] = tpc; s_tot[3] = fpc; }
    __syncthreads();
    const int TP = s_tot[2], FP = s_tot[3];
    const double dnp = (double)npig;

    // backward over the sorted detections: tp[p] / fp[p] (cumulative through p) from the suffix counts, the
    // monotone precision as the suffix maximum, and searchsorted(rc, recThrs, 'left') answered at the p where rc
    // reaches each threshold first
    int carry_tp = 0, carry_fp = 0;
    double carry_max = -CUDART_INF;
    for (int end = nd; end > 0; end -= kAccThreads) {
        const int p = end - 1 - tid;
        int tpi = 0, fpi = 0;
        if (p >= 0) {
            const unsigned long long f = flags[p];
            const int m = (int)((f >> lane_id) & 1ull), ig = (int)((f >> (32 + lane_id)) & 1ull);
            tpi = m & (ig ^ 1);
            fpi = (m ^ 1) & (ig ^ 1);
        }
        int incl, agg;                                            // tp count in the high half, fp in the low
        ScanI(tmp.scan_i).InclusiveSum((tpi << 16) | fpi, incl, agg);
        __syncthreads();
        const int tp = TP - (carry_tp + (incl >> 16) - tpi);
        const int fp = FP - (carry_fp + (incl & 0xffff) - fpi);
        const double tpd = (double)tp, fpd = (double)fp;
        const double pr = p >= 0 ? __ddiv_rn(tpd, __dadd_rn(__dadd_rn(fpd, tpd), DBL_EPSILON)) : -CUDART_INF;
        double smax, cmax;
        ScanD(tmp.scan_d).InclusiveScan(pr, smax, MaxOp(), cmax);
        __syncthreads();
        const double q = smax > carry_max ? smax : carry_max;
        if (p >= 0 && (p == 0 || tpi)) {
            const double rc = __ddiv_rn(tpd, dnp);
            const double rc_prev = p == 0 ? -CUDART_INF : __ddiv_rn((double)(tp - tpi), dnp);
            int k = 0, hi = kR;                                   // first threshold above rc_prev
            while (k < hi) {
                const int mid = (k + hi) >> 1;
                if (s_thr[mid] > rc_prev) hi = mid; else k = mid + 1;
            }
            for (; k < kR && s_thr[k] <= rc; ++k) s_q[k] = q;
        }
        carry_tp += agg >> 16;
        carry_fp += agg & 0xffff;
        carry_max = cmax > carry_max ? cmax : carry_max;
    }
    __syncthreads();
    for (int k = tid; k < kR; k += kAccThreads) precision[(t * kR + k) * kA + a] = s_q[k];
    if (tid == 0) recall[t * kA + a] = nd ? __ddiv_rn((double)TP, dnp) : 0.0;
}

// _summarizeKps: stat s < 5 averages precision, s >= 5 recall; s % 5 selects all / IoU .5 / IoU .75 / medium /
// large. The kept values are gathered in C order into `buf` ([10][T * R]) and averaged as np.mean does.
__global__ void __launch_bounds__(32)
coco_stats_kernel(const double* __restrict__ precision, const double* __restrict__ recall,
                  const double* __restrict__ iou_thrs, double* __restrict__ stats, double* __restrict__ buf) {
    sp::grid_dep_wait();
    const int s = threadIdx.x;
    if (s >= 10) return;
    const bool ap = s < 5;
    const int v = s % 5;
    const int a = v == 3 ? 1 : (v == 4 ? 2 : 0);
    double* b = buf + (size_t)s * kT * kR;
    int n = 0;
    for (int t = 0; t < kT; ++t) {
        if ((v == 1 && !(iou_thrs[t] == 0.5)) || (v == 2 && !(iou_thrs[t] == 0.75))) continue;
        if (ap) {
            for (int r = 0; r < kR; ++r) {
                const double x = precision[(t * kR + r) * kA + a];
                if (x > -1.0) b[n++] = x;
            }
        } else {
            const double x = recall[t * kA + a];
            if (x > -1.0) b[n++] = x;
        }
    }
    stats[s] = n ? __ddiv_rn(sp::numpy_sum_array(b, n), (double)n) : -1.0;
}

inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

inline int key_bits(int images) {                                 // bits of the largest image key (= images)
    int b = 1;
    while (b < 31 && (1u << b) <= (unsigned)images) ++b;
    return b;
}

struct Layout {
    size_t keys1[2], idx1[2], keys2[2], vals2[2], info, oks, gtm, buf, temp, temp_bytes, total;
};

int layout(int n, int images, int gts, Layout* L) {
    size_t s1 = 0, s2 = 0;
    if (n > 0)
        SP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, s1, (const unsigned*)nullptr, (unsigned*)nullptr,
                                                (const int*)nullptr, (int*)nullptr, n, 0, key_bits(images)));
    const int slots = images * kMaxDets;
    if (slots > 0)
        SP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, s2, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                                (const unsigned long long*)nullptr, (unsigned long long*)nullptr, slots));
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = align_up(off + bytes); return o; };
    for (int i = 0; i < 2; ++i) { L->keys1[i] = take((size_t)n * 4); L->idx1[i] = take((size_t)n * 4); }
    for (int i = 0; i < 2; ++i) { L->keys2[i] = take((size_t)slots * 8); L->vals2[i] = take((size_t)slots * 8); }
    L->info = take((size_t)images * 16);
    L->oks = take((size_t)gts * kMaxDets * 8);
    L->gtm = take((size_t)gts * kLanes);
    L->buf = take((size_t)10 * kT * kR * 8);
    L->temp_bytes = s1 > s2 ? s1 : s2;
    L->temp = take(L->temp_bytes > 0 ? L->temp_bytes : 16);
    L->total = off;
    return 0;
}

}  // namespace

extern "C" size_t sp_coco_eval_workspace_bytes(int num_dets, int num_images, int num_gts) {
    if (num_dets < 0 || num_images < 0 || num_gts < 0) return 0;
    Layout L;
    if (layout(num_dets, num_images, num_gts, &L) != 0) return 0;
    return L.total;
}

extern "C" int sp_coco_eval_kps_f32(const float* det_rows, int det_stride, const double* det_scores, const int* det_img,
                                    const unsigned char* det_keep, int num_dets,
                                    const double* gt_kps, const double* gt_area, const double* gt_bbox,
                                    const unsigned char* gt_flags, const int* gt_seg, int num_images, int num_gts,
                                    const double* iou_thrs, const double* rec_thrs, const double* area_rng,
                                    int K, int T, int R, int A, int max_dets,
                                    double* precision, double* recall, double* stats,
                                    double* oks_out, unsigned long long* det_flags_out, int* det_order_out,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    SP_RETURN_IF(K != kK || T != kT || R != kR || A != kA || max_dets != kMaxDets, SP_ERR_UNSUPPORTED);
    SP_RETURN_IF(num_dets < 0 || num_images < 0 || num_gts < 0 || det_stride < 3 * kK, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(num_images > (1 << 24) || num_dets > (1 << 30) || num_gts > (1 << 26), SP_ERR_UNSUPPORTED);
    SP_RETURN_IF(!precision || !recall || !stats || !iou_thrs || !rec_thrs || !area_rng || !workspace, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(num_dets > 0 && (!det_rows || !det_scores || !det_img), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!gt_seg, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(num_gts > 0 && (!gt_kps || !gt_area || !gt_bbox || !gt_flags), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!sp_aligned16(workspace), SP_ERR_BAD_ALIGNMENT);
    Layout L;
    const int lerr = layout(num_dets, num_images, num_gts, &L);
    if (lerr != 0) return lerr;
    SP_RETURN_IF(workspace_bytes < L.total, SP_ERR_WORKSPACE);
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    auto at = [&](size_t off) { return static_cast<void*>(ws + off); };
    unsigned* keys1[2] = {static_cast<unsigned*>(at(L.keys1[0])), static_cast<unsigned*>(at(L.keys1[1]))};
    int* idx1[2] = {static_cast<int*>(at(L.idx1[0])), static_cast<int*>(at(L.idx1[1]))};
    unsigned long long* keys2[2] = {static_cast<unsigned long long*>(at(L.keys2[0])), static_cast<unsigned long long*>(at(L.keys2[1]))};
    unsigned long long* vals2[2] = {static_cast<unsigned long long*>(at(L.vals2[0])), static_cast<unsigned long long*>(at(L.vals2[1]))};
    int4* info = static_cast<int4*>(at(L.info));
    double* oks = oks_out ? oks_out : static_cast<double*>(at(L.oks));
    unsigned long long* slot_flags = det_flags_out ? det_flags_out : vals2[0];
    const int slots = num_images * kMaxDets;

    if (num_dets > 0) {
        SP_CUDA(sp_launch(coco_det_keys_kernel, dim3((num_dets + 255) / 256), dim3(256), 0, st,
                          det_img, det_keep, num_dets, num_images, keys1[0], idx1[0]));
        size_t tb = L.temp_bytes;
        SP_CUDA(cub::DeviceRadixSort::SortPairs(at(L.temp), tb, keys1[0], keys1[1], idx1[0], idx1[1], num_dets, 0,
                                                key_bits(num_images), st));
    }
    if (num_images > 0) {
        GtView gv{gt_kps, gt_area, gt_bbox, gt_flags, gt_seg};
        SP_CUDA(sp_launch(coco_image_kernel, dim3((num_images + kImgWarps - 1) / kImgWarps), dim3(kImgWarps * 32), 0, st,
                          det_rows, det_stride, det_scores, keys1[1], idx1[1], num_dets, gv, num_images, iou_thrs, area_rng,
                          oks, static_cast<unsigned char*>(at(L.gtm)), info, keys2[0], slot_flags, det_order_out));
        size_t tb = L.temp_bytes;
        SP_CUDA(cub::DeviceRadixSort::SortPairs(at(L.temp), tb, keys2[0], keys2[1], slot_flags, vals2[1], slots, 0, 64, st));
    }
    SP_CUDA(sp_launch(coco_accumulate_kernel, dim3(kLanes), dim3(kAccThreads), 0, st,
                      info, num_images, vals2[1], rec_thrs, precision, recall));
    SP_CUDA(sp_launch(coco_stats_kernel, dim3(1), dim3(32), 0, st,
                      precision, recall, iou_thrs, stats, static_cast<double*>(at(L.buf))));
    return 0;
}
