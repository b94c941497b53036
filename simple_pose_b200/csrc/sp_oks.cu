// A7/A8/A9: OKS similarity, greedy keypoint NMS per image, eval rescoring
// (reference datasets/naive_data.py:120-173 and eval.py:153-197). All float64.
//
// Latency-bound, not bandwidth-bound (408 B per person). One CTA owns one image (segment):
// persons are ranked by descending score with a counting rank (stable; ties -> higher index
// first, i.e. argsort()[::-1] of a stable sort). Images of up to 64 persons (every COCO image)
// then score all n(n-1)/2 ordered pairs at once, one thread per pair, into 64-bit suppression
// rows, and the greedy pass is n bit operations (cfg 5, 4952 images / 104 k persons: 0.26 ms
// instead of 1.09 ms). Larger images run the greedy loop itself: for each surviving pick the
// remaining candidates are scored in parallel, one thread per candidate. The per-pair arithmetic
// keeps the reference's operation order, including NumPy's 8-accumulator pairwise summation,
// so that the `oks > thresh` decisions agree.
#include "sp_common.cuh"
#include "sp_numpy_sum.cuh"
#include <math_constants.h>

namespace {

constexpr int kNmsThreads = 128;
constexpr int kMaxJoints = 64;

__device__ __constant__ double kCocoSigmas[17] = {.26, .25, .25, .35, .35, .79, .79, .72, .72,
                                                  .62, .62, 1.07, 1.07, .87, .87, .89, .89};

using sp::NumpySum;

struct OksParams {
    const double* sigmas;    // NULL -> COCO table
    int K;
    int use_vis;
    double vis_thresh;
};

__device__ __forceinline__ double joint_var(const OksParams& P, int k) {
    const double s = P.sigmas ? P.sigmas[k] : __ddiv_rn(kCocoSigmas[k], 10.0);
    const double t = __dmul_rn(s, 2.0);
    return __dmul_rn(t, t);
}

// oks_iou for one (pick, candidate) pair, naive_data.py:139-149. T = double (the reference's arrays) or
// float (decoder output rows; the JSON round trip of eval.py:138-160 widens exactly these floats).
template <typename T>
__device__ __noinline__ double oks_pair_generic(const OksParams& P, const T* __restrict__ pick, const T* __restrict__ cand,
                                   double pick_area, double cand_area) {
    const double denom_area = __dadd_rn(__ddiv_rn(__dadd_rn(pick_area, cand_area), 2.0), 1e-12);
    int nvis = P.K;
    if (P.use_vis) {
        nvis = 0;
        for (int k = 0; k < P.K; ++k)
            nvis += ((double)cand[3 * k + 2] > P.vis_thresh) && ((double)pick[3 * k + 2] > P.vis_thresh);
    }
    NumpySum acc;
    acc.begin(P.K);
    for (int k = 0; k < P.K; ++k) {
        const double dx = __dsub_rn((double)cand[3 * k + 0], (double)pick[3 * k + 0]);
        const double dy = __dsub_rn((double)cand[3 * k + 1], (double)pick[3 * k + 1]);
        double e = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
        e = __ddiv_rn(__ddiv_rn(__ddiv_rn(e, joint_var(P, k)), denom_area), 2.0);
        double v = exp(-e);
        if (P.use_vis) {
            const bool vis = ((double)cand[3 * k + 2] > P.vis_thresh) && ((double)pick[3 * k + 2] > P.vis_thresh);
            v = __dmul_rn(v, vis ? 1.0 : 0.0);
        }
        acc.push(v);
    }
    // (vd_vis.sum(-1) + 1e-12) is float32 arithmetic in the reference
    const float cnt = __fadd_rn((float)nvis, 1e-12f);
    return __ddiv_rn(acc.result(), (double)cnt);
}

// The COCO case (K = 17, in_vis_thresh=None, default sigmas), fully unrolled: the 17 per-joint chains
// (two float64 divisions and an exp each) are independent, so unrolled they overlap instead of running one
// after the other -- the NMS kernel is latency-bound (one image per CTA), and this chain is its critical
// path. Same operations in the same order per joint, and NumPy's pairwise sum written out for n = 17:
// r[j] = v[j] + v[j+8], ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), + v[16], 0 + that. Division by 2 is exact, so
// x * 0.5 == x / 2 bit for bit.
template <typename T>
__device__ __forceinline__ double oks_pair_coco17(const T* __restrict__ pick, const T* __restrict__ cand,
                                                  double pick_area, double cand_area) {
    const double denom_area = __dadd_rn(__dmul_rn(__dadd_rn(pick_area, cand_area), 0.5), 1e-12);
    double v[17];
#pragma unroll
    for (int k = 0; k < 17; ++k) {
        const double dx = __dsub_rn((double)cand[3 * k + 0], (double)pick[3 * k + 0]);
        const double dy = __dsub_rn((double)cand[3 * k + 1], (double)pick[3 * k + 1]);
        const double s = __ddiv_rn(kCocoSigmas[k], 10.0);
        const double t = __dmul_rn(s, 2.0);
        double e = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
        e = __dmul_rn(__ddiv_rn(__ddiv_rn(e, __dmul_rn(t, t)), denom_area), 0.5);
        v[k] = exp(-e);
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(v[j], v[j + 8]);
    double tail = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                            __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    tail = __dadd_rn(tail, v[16]);
    const float cnt = __fadd_rn(17.0f, 1e-12f);
    return __ddiv_rn(__dadd_rn(0.0, tail), (double)cnt);
}

template <typename T>
__device__ __forceinline__ double oks_pair(const OksParams& P, const T* __restrict__ pick, const T* __restrict__ cand,
                                           double pick_area, double cand_area) {
    if (P.K == 17 && !P.use_vis && P.sigmas == nullptr) return oks_pair_coco17(pick, cand, pick_area, cand_area);
    return oks_pair_generic(P, pick, cand, pick_area, cand_area);
}

// The NMS only needs the DECISION oks > thresh. The float64 chain above (two divisions and an exp per joint) made
// the NMS kernel float64-pipe bound: 221 us for the 104 k persons of BASELINE config 5, ~50 % of the FP64 issue
// rate. This float32 evaluation of the same expression costs an eighth of the instructions on a pipe twice as
// wide, and its error is bounded: the joint differences are formed exactly in float64 and rounded once, so the
// exponent e carries a relative error < 5e-7, each term exp(-e) an absolute error < 5e-7 (e * exp(-e) <= 1/e), the
// mean of 17 terms < 2e-6 in total. A pair is decided here when the result is further than kOksMargin = 1e-4 from
// the threshold -- 50 times the bound -- and re-evaluated with the exact chain otherwise (also when anything is
// NaN). The decisions, hence keep sets and pick order, are the float64 ones.
constexpr float kOksMargin = 1e-4f;
__device__ __constant__ float kCocoInvVar[17] = {
    // 1 / (2 * sigma_k / 10)^2
    1.0f / (0.052f * 0.052f), 1.0f / (0.050f * 0.050f), 1.0f / (0.050f * 0.050f), 1.0f / (0.070f * 0.070f), 1.0f / (0.070f * 0.070f),
    1.0f / (0.158f * 0.158f), 1.0f / (0.158f * 0.158f), 1.0f / (0.144f * 0.144f), 1.0f / (0.144f * 0.144f), 1.0f / (0.124f * 0.124f),
    1.0f / (0.124f * 0.124f), 1.0f / (0.214f * 0.214f), 1.0f / (0.214f * 0.214f), 1.0f / (0.174f * 0.174f), 1.0f / (0.174f * 0.174f),
    1.0f / (0.178f * 0.178f), 1.0f / (0.178f * 0.178f)};

template <typename T>
__device__ __forceinline__ float oks_pair_fast17(const T* __restrict__ pick, const T* __restrict__ cand, double pick_area,
                                                 double cand_area) {
    const float inv_area = 0.5f / (0.5f * ((float)pick_area + (float)cand_area) + 1e-12f);    // 1 / denom_area / 2
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 17; ++k) {
        const float dx = (float)((double)cand[3 * k + 0] - (double)pick[3 * k + 0]);
        const float dy = (float)((double)cand[3 * k + 1] - (double)pick[3 * k + 1]);
        const float e = (dx * dx + dy * dy) * kCocoInvVar[k] * inv_area;
        sum += expf(-e);
    }
    return sum * (1.0f / 17.0f);
}

// oks > thresh with the float64 chain's verdict
template <typename T>
__device__ __forceinline__ bool oks_exceeds(const OksParams& P, const T* __restrict__ pick, const T* __restrict__ cand,
                                            double pick_area, double cand_area, double thresh) {
    if (P.K == 17 && !P.use_vis && P.sigmas == nullptr) {
        const float v = oks_pair_fast17(pick, cand, pick_area, cand_area);
        const float gap = v - (float)thresh;
        if (fabsf(gap) > kOksMargin) return gap > 0.f;            // false for NaN: falls through to the exact chain
    }
    return oks_pair_generic(P, pick, cand, pick_area, cand_area) > thresh;    // rare: a rolled loop keeps the kernel's registers low
}

// eval.py:168-175 for one person: box_score * mean(conf[conf > thr]) (0 if none)
template <typename T>
__device__ double rescore_one(const T* __restrict__ k, int K, double thr, double box_score) {
    int cnt = 0;
    for (int j = 0; j < K; ++j) cnt += ((double)k[3 * j + 2] > thr);
    double mean = 0.0;
    if (cnt > 0) {
        NumpySum acc;
        acc.begin(cnt);
        for (int j = 0; j < K; ++j) {
            const double c = (double)k[3 * j + 2];
            if (c > thr) acc.push(c);
        }
        mean = __ddiv_rn(acc.result(), (double)cnt);
    }
    return __dmul_rn(box_score, mean);
}

__global__ void __launch_bounds__(128)
oks_iou_kernel(const double* __restrict__ pick_kps, const double* __restrict__ cand_kps,
               const double* __restrict__ pick_area, const double* __restrict__ cand_area,
               double* __restrict__ out, int n, OksParams P) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = oks_pair(P, pick_kps, cand_kps + (size_t)i * 3 * P.K, pick_area[0], cand_area[i]);
}

// dynamic shared memory of the NMS kernels, per image (max_seg = the largest image of the launch):
//   score[max_seg] f64 | area[max_seg] f64 | suppression rows[64] u64 | order[max_seg] i32 | alive[max_seg] u8
__host__ __device__ inline size_t nms_smem_bytes(int max_seg) {
    return (size_t)max_seg * 16 + 64 * 8 + (size_t)max_seg * 4 + (((size_t)max_seg + 15) & ~(size_t)15);
}

// Greedy OKS-NMS of one image whose scores and areas are already in shared memory. kps: person i's
// (x, y, conf) * K starts at kps + i * stride. Calls emit(i, kept) once per person and writes rank.
template <typename T, typename Emit>
__device__ __forceinline__ void nms_image(const T* __restrict__ kps, size_t stride, int n, const double* score,
                                          const double* area, unsigned long long* rows, int* order, unsigned char* alive,
                                          int* __restrict__ rank, double thresh, const OksParams& P, int force_serial,
                                          Emit&& emit) {
    const int tid = threadIdx.x;
    // descending-score visiting order; ties: higher index first
    for (int i = tid; i < n; i += kNmsThreads) {
        const double si = score[i];
        int r = 0;
        for (int j = 0; j < n; ++j) {
            const double sj = score[j];
            r += (sj > si) || (sj == si && j > i);
        }
        order[r] = i;
        if (rank) rank[i] = r;
        alive[i] = 1;
    }
    __syncthreads();

    if (n <= 64 && !force_serial) {
        // Small image (the COCO case: ~20 boxes): score ALL n(n-1)/2 (earlier, later) pairs of the
        // visiting order at once, one thread per pair, into 64-bit suppression rows; the greedy pass
        // is then n bit operations. Same decisions as the loop below (oks_pair is evaluated with the
        // earlier person as the pick, exactly as the loop would), but one exp-chain deep instead of
        // one per surviving pick.
        for (int i = tid; i < n; i += kNmsThreads) rows[i] = 0ull;
        __syncthreads();
        const int total = n * (n - 1) / 2;
        for (int idx = tid; idx < total; idx += kNmsThreads) {
            // row p of the strict upper triangle starts at S(p) = p*n - p*(p+1)/2
            const float b = (float)(2 * n - 1);
            int p = (int)((b - sqrtf(fmaxf(b * b - 8.0f * (float)idx, 0.0f))) * 0.5f);
            p = min(max(p, 0), n - 2);
            while (p + 1 <= n - 2 && (p + 1) * n - (p + 1) * (p + 2) / 2 <= idx) ++p;
            while (p > 0 && p * n - p * (p + 1) / 2 > idx) --p;
            const int c = p + 1 + (idx - (p * n - p * (p + 1) / 2));
            const int i = order[p], j = order[c];
            if (oks_exceeds(P, kps + (size_t)i * stride, kps + (size_t)j * stride, area[i], area[j], thresh))
                atomicOr(&rows[p], 1ull << c);
        }
        __syncthreads();
        if (tid == 0) {
            unsigned long long alive_bits = (n == 64) ? ~0ull : ((1ull << n) - 1ull);
            for (int p = 0; p < n; ++p) {
                if (!((alive_bits >> p) & 1ull)) { alive[p] = 0; continue; }
                alive_bits &= ~rows[p];
            }
        }
        __syncthreads();
    } else {
        for (int p = 0; p < n; ++p) {
            if (!alive[p]) continue;                   // uniform: everyone reads the same byte
            const int i = order[p];
            const T* pick = kps + (size_t)i * stride;
            const double pick_area = area[i];
            for (int c = p + 1 + tid; c < n; c += kNmsThreads) {
                if (!alive[c]) continue;
                const int j = order[c];
                if (oks_exceeds(P, pick, kps + (size_t)j * stride, pick_area, area[j], thresh)) alive[c] = 0;   // survivors: oks <= thresh
            }
            __syncthreads();
        }
    }
    // alive[p] now says whether the p-th person of the visiting order was picked
    for (int p = tid; p < n; p += kNmsThreads) emit(order[p], alive[p] != 0);
}

__global__ void __launch_bounds__(kNmsThreads)
oks_nms_kernel(const double* __restrict__ kps, const double* __restrict__ scores, const double* __restrict__ areas,
               const int* __restrict__ seg, unsigned char* __restrict__ keep, int* __restrict__ rank,
               int max_seg, double thresh, OksParams P, int force_serial) {
    extern __shared__ __align__(16) unsigned char nms_smem[];
    double* sc = reinterpret_cast<double*>(nms_smem);
    double* ar = sc + max_seg;
    unsigned long long* rows = reinterpret_cast<unsigned long long*>(ar + max_seg);
    int* order = reinterpret_cast<int*>(rows + 64);
    unsigned char* alive = reinterpret_cast<unsigned char*>(order + max_seg);
    const int lo = seg[blockIdx.x], hi = seg[blockIdx.x + 1];
    const int n = hi - lo;
    if (n <= 0) return;
    for (int i = threadIdx.x; i < n; i += kNmsThreads) {
        sc[i] = scores[lo + i];
        ar[i] = areas[lo + i];
    }
    __syncthreads();
    const size_t stride = (size_t)3 * P.K;
    nms_image(kps + (size_t)lo * stride, stride, n, sc, ar, rows, order, alive, rank + lo, thresh, P, force_serial,
              [&](int i, bool kept) { keep[lo + i] = kept ? 1 : 0; });
}

// The eval chain after the decoder in ONE launch (eval.py:153-197): the decoder has written
// (x, y, conf) * K into float32 result rows; per image this kernel rescores every person
// (box_score * mean(conf > thr)), runs the greedy OKS-NMS and completes the rows in place:
//   row[3K] = keep flag (0/1), row[3K+1], row[3K+2] = low / high 32 bits of the float64 score.
// No float64 keypoint copy (pack_kps), no separate rescoring pass, no pack_rows pass.
// Where the completed rows of an image go besides the local table: nowhere (world == 1), or into the same slot of
// every rank's copy of the gather buffer -- the all-gather of the multi-GPU evaluation done by this kernel's own
// stores over NVLink / NVSwitch instead of a collective after it. `mc_base` is the NVLS multicast mapping of the
// symmetric buffer (one multimem.st lands in all ranks' memories, replicated by the switch); without it the rows
// are stored to each peer's unicast mapping in turn. `slot` = float offset of this rank's slot in the buffer.
struct RowFanout {
    float* mc_base;
    float* const* peer_base;     // device array [world] of the buffer's address in each rank
    int world, me;
    long long slot;
};

__device__ __forceinline__ void multimem_st_v2(float2* mc_addr, float2 v) {
    asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1, %2};" ::"l"(mc_addr), "f"(v.x), "f"(v.y) : "memory");
}

__global__ void __launch_bounds__(kNmsThreads)
eval_rows_nms_kernel(float* __restrict__ rows_io, int row_stride, const double* __restrict__ box_scores,
                     const double* __restrict__ areas_f64, const float* __restrict__ areas_f32,
                     const int* __restrict__ seg, int* __restrict__ rank, int max_seg, double vis_thr, double thresh,
                     OksParams P, int force_serial, RowFanout out) {
    extern __shared__ __align__(16) unsigned char nms_smem[];
    double* sc = reinterpret_cast<double*>(nms_smem);
    double* ar = sc + max_seg;
    unsigned long long* rows = reinterpret_cast<unsigned long long*>(ar + max_seg);
    int* order = reinterpret_cast<int*>(rows + 64);
    unsigned char* alive = reinterpret_cast<unsigned char*>(order + max_seg);
    sp::grid_dep_wait();                // the rows come from the decode kernel just before on the stream
    const int lo = seg[blockIdx.x], hi = seg[blockIdx.x + 1];
    const int n = hi - lo;
    if (n <= 0) return;
    float* base = rows_io + (size_t)lo * row_stride;
    for (int i = threadIdx.x; i < n; i += kNmsThreads) {
        sc[i] = rescore_one(base + (size_t)i * row_stride, P.K, vis_thr, box_scores[lo + i]);
        ar[i] = areas_f64 ? areas_f64[lo + i] : (double)areas_f32[lo + i];
    }
    __syncthreads();
    const int K = P.K;
    nms_image(base, (size_t)row_stride, n, sc, ar, rows, order, alive, rank ? rank + lo : nullptr, thresh, P, force_serial,
              [&](int i, bool kept) {
                  float* r = base + (size_t)i * row_stride + 3 * K;
                  const unsigned long long bits = (unsigned long long)__double_as_longlong(sc[i]);
                  r[0] = kept ? 1.f : 0.f;
                  r[1] = __uint_as_float((unsigned)(bits & 0xffffffffull));
                  r[2] = __uint_as_float((unsigned)(bits >> 32));
              });
    if (out.world <= 1) return;
    // ---- fan the image's completed rows out to every rank (8-byte pieces; a row is 3K+3 floats, 8-byte aligned for
    // odd K and an even row_stride, which the host checks)
    __syncthreads();                                   // keep / score slots above were written by other threads
    const int pieces = n * row_stride / 2;
    const size_t off = (size_t)out.slot + (size_t)lo * row_stride;
    const float2* src = reinterpret_cast<const float2*>(base);
    if (out.mc_base != nullptr) {
        float2* dst = reinterpret_cast<float2*>(out.mc_base + off);
        for (int i = threadIdx.x; i < pieces; i += kNmsThreads) multimem_st_v2(dst + i, src[i]);
    } else {
        for (int p = 0; p < out.world; ++p) {
            if (p == out.me) continue;
            float2* dst = reinterpret_cast<float2*>(out.peer_base[p] + off);
            for (int i = threadIdx.x; i < pieces; i += kNmsThreads) dst[i] = src[i];
        }
    }
}

// eval.py:168-175
__global__ void __launch_bounds__(128)
rescore_kernel(const double* __restrict__ kps, const double* __restrict__ box_scores, double* __restrict__ scores,
               int N, int K, double thr) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    scores[i] = rescore_one(kps + (size_t)i * 3 * K, K, thr, box_scores[i]);
}

__global__ void __launch_bounds__(256)
pack_kps_kernel(const float* __restrict__ coords, const float* __restrict__ maxval, double* __restrict__ out, long long nk) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nk) return;
    const float2 c = reinterpret_cast<const float2*>(coords)[i];
    out[3 * i + 0] = (double)c.x;
    out[3 * i + 1] = (double)c.y;
    out[3 * i + 2] = (double)maxval[i];
}

// ShardedPoseEvaluator result rows: [n, 3K+2] f32 = (x, y, conf) * K, keep flag, rescored score
// (what eval.py:186-196 writes per kept person, kept as one table for the all-gather)
__global__ void __launch_bounds__(256)
pack_rows_kernel(const float* __restrict__ coords, const float* __restrict__ maxval, const unsigned char* __restrict__ keep,
                 const double* __restrict__ scores, float* __restrict__ rows, long long n, int K) {
    const int width = 3 * K + 2;
    const long long total = n * width;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long p = i / width;
        const int c = (int)(i - p * width);
        float v;
        if (c < 3 * K) {
            const int k = c / 3, e = c - 3 * k;
            v = (e < 2) ? coords[(p * K + k) * 2 + e] : maxval[p * K + k];
        } else if (c == 3 * K) {
            v = keep ? (float)keep[p] : 0.f;
        } else {
            v = scores ? (float)scores[p] : 0.f;
        }
        rows[i] = v;
    }
}

// kps_to_dict_ (metrics/pose_metrics.py:172-179) as one table: rows [N, 3K+1] f32 = (x, y, conf) * K, then the
// person score mean(conf) + max(conf) (sp::PersonScore, shared with the validation step kernel).
__global__ void __launch_bounds__(128)
person_rows_kernel(const float* __restrict__ coords, const float* __restrict__ maxval, float* __restrict__ rows, int N, int K) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= N) return;
    float* r = rows + (size_t)p * (3 * K + 1);
    sp::PersonScore score = sp::PersonScore::start();
    for (int k = 0; k < K; ++k) {
        const float2 c = reinterpret_cast<const float2*>(coords)[(size_t)p * K + k];
        const float v = maxval[(size_t)p * K + k];
        r[3 * k + 0] = c.x;
        r[3 * k + 1] = c.y;
        r[3 * k + 2] = v;
        score.add(v);
    }
    r[3 * K] = score.value(K);
}

}  // namespace

extern "C" int sp_person_rows_f32(const float* coords, const float* maxval, float* rows, int N, int K, void* stream) {
    SP_RETURN_IF(N < 0 || K <= 0, SP_ERR_BAD_ARGUMENT);
    if (N == 0) return 0;
    SP_RETURN_IF(!coords || !maxval || !rows, SP_ERR_BAD_ARGUMENT);
    SP_CUDA(sp_launch_plain(person_rows_kernel, dim3((N + 127) / 128), dim3(128), 0, static_cast<cudaStream_t>(stream),
                            coords, maxval, rows, N, K));
    return 0;
}

static int eval_rows_nms_launch(float* rows, int row_stride, const double* box_scores, const double* areas_f64,
                                const float* areas_f32, const int* seg, const double* sigmas, int* rank,
                                int N, int I, int K, int max_seg, double in_vis_thre, double oks_thre, RowFanout out, void* stream) {
    SP_RETURN_IF(N < 0 || I < 0 || K <= 0 || K > kMaxJoints || max_seg < 0 || row_stride < 3 * K + 3, SP_ERR_BAD_ARGUMENT);
    if (N == 0 || I == 0) return 0;
    SP_RETURN_IF(!rows || !box_scores || !seg || (!areas_f64 && !areas_f32), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!sigmas && K != 17, SP_ERR_BAD_ARGUMENT);
    const size_t smem = nms_smem_bytes(max_seg);
    SP_RETURN_IF(smem > 200 * 1024, SP_ERR_UNSUPPORTED);
    OksParams P{sigmas, K, 0, 0.0};
    SP_CUDA(sp_launch_smem(eval_rows_nms_kernel, dim3(I), dim3(kNmsThreads), smem, static_cast<cudaStream_t>(stream),
                           rows, row_stride, box_scores, areas_f64, areas_f32, seg, rank, max_seg, in_vis_thre, oks_thre, P,
                           sp_knob(sp_tuning().nms_serial, 0), out));
    return 0;
}

extern "C" int sp_eval_rows_nms_f32(float* rows, int row_stride, const double* box_scores, const double* areas_f64,
                                    const float* areas_f32, const int* seg, const double* sigmas, int* rank,
                                    int N, int I, int K, int max_seg, double in_vis_thre, double oks_thre, void* stream) {
    RowFanout out{nullptr, nullptr, 1, 0, 0};
    return eval_rows_nms_launch(rows, row_stride, box_scores, areas_f64, areas_f32, seg, sigmas, rank, N, I, K, max_seg,
                                in_vis_thre, oks_thre, out, stream);
}

extern "C" int sp_eval_rows_nms_fanout_f32(float* rows, int row_stride, const double* box_scores, const double* areas_f64,
                                           const float* areas_f32, const int* seg, const double* sigmas, int* rank,
                                           int N, int I, int K, int max_seg, double in_vis_thre, double oks_thre,
                                           void* multicast_base, const void* const* peer_bases, int world, int my_rank,
                                           long long slot_offset_floats, void* stream) {
    SP_RETURN_IF(world < 1 || my_rank < 0 || my_rank >= world || slot_offset_floats < 0, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(world > 1 && !multicast_base && !peer_bases, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(world > 1 && ((row_stride & 1) || (slot_offset_floats & 1) || (reinterpret_cast<uintptr_t>(rows) & 7u)), SP_ERR_BAD_ALIGNMENT);
    RowFanout out{static_cast<float*>(multicast_base), reinterpret_cast<float* const*>(const_cast<void* const*>(reinterpret_cast<const void* const*>(peer_bases))), world, my_rank, slot_offset_floats};
    return eval_rows_nms_launch(rows, row_stride, box_scores, areas_f64, areas_f32, seg, sigmas, rank, N, I, K, max_seg,
                                in_vis_thre, oks_thre, out, stream);
}

extern "C" int sp_pack_rows_f32(const float* coords, const float* maxval, const unsigned char* keep, const double* scores,
                                float* rows, int N, int K, void* stream) {
    SP_RETURN_IF(N < 0 || K <= 0, SP_ERR_BAD_ARGUMENT);
    if (N == 0) return 0;
    SP_RETURN_IF(!coords || !maxval || !rows, SP_ERR_BAD_ARGUMENT);
    const long long total = (long long)N * (3 * K + 2);
    long long blocks = (total + 255) / 256;
    const long long cap = (long long)sp_sm_count() * 16;
    if (blocks > cap) blocks = cap;
    SP_CUDA(sp_launch_plain(pack_rows_kernel, dim3((unsigned)blocks), dim3(256), 0, static_cast<cudaStream_t>(stream),
                            coords, maxval, keep, scores, rows, (long long)N, K));
    return 0;
}

extern "C" int sp_oks_iou_f64(const double* pick_kps, const double* cand_kps, const double* pick_area,
                              const double* cand_area, const double* sigmas, double* out,
                              int n, int K, int use_vis_thresh, double vis_thresh, void* stream) {
    SP_RETURN_IF(!pick_kps || !cand_kps || !pick_area || !cand_area || !out, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(n < 0 || K <= 0 || K > kMaxJoints, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!sigmas && K != 17, SP_ERR_BAD_ARGUMENT);
    if (n == 0) return 0;
    OksParams P{sigmas, K, use_vis_thresh ? 1 : 0, vis_thresh};
    SP_CUDA(sp_launch_plain(oks_iou_kernel, dim3((n + 127) / 128), dim3(128), 0, static_cast<cudaStream_t>(stream),
                            pick_kps, cand_kps, pick_area, cand_area, out, n, P));
    return 0;
}

extern "C" int sp_oks_nms_f64(const double* kps, const double* scores, const double* areas, const int* seg,
                              const double* sigmas, unsigned char* keep, int* rank,
                              int N, int I, int K, int max_seg, double thresh,
                              int use_vis_thresh, double vis_thresh, void* stream) {
    SP_RETURN_IF(!kps || !scores || !areas || !seg || !keep || !rank, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(N < 0 || I < 0 || K <= 0 || K > kMaxJoints || max_seg < 0, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!sigmas && K != 17, SP_ERR_BAD_ARGUMENT);
    if (N == 0 || I == 0) return 0;
    const size_t smem = nms_smem_bytes(max_seg);
    SP_RETURN_IF(smem > 200 * 1024, SP_ERR_UNSUPPORTED);
    if (smem > 48 * 1024) SP_CUDA(sp_ensure_dyn_smem(reinterpret_cast<const void*>(oks_nms_kernel), smem));
    OksParams P{sigmas, K, use_vis_thresh ? 1 : 0, vis_thresh};
    SP_CUDA(sp_launch_plain(oks_nms_kernel, dim3(I), dim3(kNmsThreads), smem, static_cast<cudaStream_t>(stream),
                            kps, scores, areas, seg, keep, rank, max_seg, thresh, P, sp_knob(sp_tuning().nms_serial, 0)));
    return 0;
}

extern "C" int sp_rescore_f64(const double* kps, const double* box_scores, double* scores,
                              int N, int K, double in_vis_thre, void* stream) {
    SP_RETURN_IF(!kps || !box_scores || !scores, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(N < 0 || K <= 0 || K > 128, SP_ERR_BAD_ARGUMENT);
    if (N == 0) return 0;
    SP_CUDA(sp_launch_plain(rescore_kernel, dim3((N + 127) / 128), dim3(128), 0, static_cast<cudaStream_t>(stream),
                            kps, box_scores, scores, N, K, in_vis_thre));
    return 0;
}

extern "C" int sp_pack_kps_f64(const float* coords, const float* maxval, double* out_kps, int N, int K, void* stream) {
    SP_RETURN_IF(!coords || !maxval || !out_kps, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(N < 0 || K <= 0, SP_ERR_BAD_ARGUMENT);
    const long long nk = (long long)N * K;
    if (nk == 0) return 0;
    SP_CUDA(sp_launch_plain(pack_kps_kernel, dim3((unsigned)((nk + 255) / 256)), dim3(256), 0, static_cast<cudaStream_t>(stream),
                            coords, maxval, out_kps, nk));
    return 0;
}
