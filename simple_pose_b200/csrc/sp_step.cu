// One launch per batch for the whole hot path over a predicted map (BASELINE configs 1 + 2 at their literal
// batch sizes, and the body of the solvers' val() loop, processors/dp_pose_hrnet_solver.py:150-161):
//
//   targets, mask = get_heat_map(joints)                          commons/transforms.py:167-191
//   loss = 0.5 * MSELoss(pred * mask, target * mask) (+ backward)    processors/dp_pose_hrnet_solver.py:106-107
//   acc inputs: argmax of pred * mask and target * mask             metrics/pose_metrics.py:223-224
//   pred_kps, scores = GaussTaylorKeyPointDecoder()(pred, trans_inv) metrics/pose_metrics.py:62-107
//
// Why: at batch 128 each of the three stand-alone kernels moves 27-80 MB (4-12 us of HBM time) and the step is
// bound by launch gaps and per-kernel ramp/tail, not bandwidth (30.6 us per step replayed from a CUDA graph,
// 47 us launched from Python, against 20 us of HBM time). Here every (person, joint) map is brought into shared
// memory ONCE by a 1-D TMA bulk copy and the owning warp does everything to it while it is there: argmax +
// 13-point blur + Taylor step + affine (the decode kernel's device code), then the float64 separable target, the
// masked difference, loss partial, gradient and -- on request -- the target map itself and the HeatMapAcc
// argmaxes (the fused training kernel's device code). pred is read once instead of twice and the targets are
// written but never read back: 3 map-sized HBM streams per person (read pred, write targets, write grad)
// instead of 5, in one launch instead of three. Results: coords / maxval / targets / weights / grad / acc axes
// are bit-identical to the stand-alone kernels; the loss differs only in the float64 summation order.
#include "sp_common.cuh"
#include "sp_argmax.cuh"
#include "sp_decode_dev.cuh"
#include "sp_train_dev.cuh"

namespace {

using sp_reduce::MseWorkspace;

constexpr int kHeadBytes = 1024;     // mbarriers (one per warp), claimed-map slots, CTA work counter
constexpr int kWtsBytes = 1024;      // 11 x 11 blur weights
constexpr int kPatchBytes = 1536;    // zero-padded 15 x 15 patch for peaks near the border

// dynamic shared memory: [head][blur weights] then per warp [patch][float64 factors][the map]
//
// Work distribution. static_maps == 0: CTA c owns the contiguous map range [c*nmaps/grid, (c+1)*nmaps/grid) and its
// warps claim maps from a shared-memory counter (small launches: nothing to balance, no global atomics).
// static_maps > 0: maps are dealt GRID-WIDE -- warp w of CTA c owns maps k*grid*nwarps + c*nwarps + w for
// k < static_maps, the rest come one at a time from the counter in the caller's workspace (claimed one map ahead, so
// the atomic's round trip is never waited for). The SMs do not drain HBM at equal rates once the memory system
// queues (profiles/r1f_fused_timeline.md), and with equal ranges the slowest SM is the critical path.
//
// The validation form (VAL, val_step_kernel) is the body of val() for both decoder families: no gradient, no target
// map, HeatMapAcc argmaxes always, the decoder MODE fixed at compile time (GaussTaylor or Basic; Basic reads no blur
// weights and needs no patch, but keeps the same shared-memory layout and so the same work distribution), and two
// results that need more than one map:
//   - the kps_to_dict_ row of a person: after a map's (x, y, conf) is in its row, lane 0 counts the map in the
//     person's arrival counter (release/acquire); the map that completes the person reads the K peaks back in joint
//     order, writes the score column and returns the counter to zero;
//   - the HeatMapAcc value: the last CTA of the loss reduction has acquired every CTA's argmax axes and runs the
//     stand-alone epilogue on them.
struct ValOut {
    unsigned int* arrivals;    // [B] per-person map counters in the caller's workspace, zero between launches
    float* acc;
    float norm_x, norm_y, thresh;
    int B;
};

template <bool WRITE_GRAD, bool WRITE_TARGETS, bool ACC, int MODE, bool VAL>
__device__ __forceinline__ void step_body(const sp_dec::DecodeArgs& A, const sp_trn::MapIo& io, float* __restrict__ loss,
                                          MseWorkspace* __restrict__ ws, double inv_count, int nwarps, int static_maps,
                                          const ValOut& V) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int KS = 11;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int hw = A.H * A.W;
    const uint32_t map_bytes = (uint32_t)hw * 4u;
    const int wpad = (A.W + 1) & ~1;
    const size_t fac_bytes = (size_t)(wpad + ((A.H + 1) & ~1)) * sizeof(double);
    const size_t per_warp = kPatchBytes + fac_bytes + map_bytes;

    uint64_t* bar = reinterpret_cast<uint64_t*>(smem) + warp;
    int& next_map = *reinterpret_cast<int*>(smem + kHeadBytes - 8);
    float* wts = reinterpret_cast<float*>(smem + kHeadBytes);
    unsigned char* mine = smem + kHeadBytes + kWtsBytes + (size_t)warp * per_warp;
    float* patch = reinterpret_cast<float*>(mine);
    double* ex = reinterpret_cast<double*>(mine + kPatchBytes);
    double* ey = ex + wpad;
    float* a = reinterpret_cast<float*>(mine + kPatchBytes + fac_bytes);

    const bool grid_wide = static_maps > 0;
    const int round = (int)gridDim.x * nwarps;
    const int range_lo = (int)((long long)blockIdx.x * A.nmaps / gridDim.x);
    const int range_hi = (int)((long long)(blockIdx.x + 1) * A.nmaps / gridDim.x);
    if (threadIdx.x == 0) next_map = range_lo + nwarps;      // per-CTA mode: the first nwarps maps are assigned statically
    if (lane == 0) {
        sp::mbar_init(bar, 1);
        sp::mbar_fence_init();
    }
    __syncthreads();
    sp::grid_dep_wait();            // everything above overlapped the previous kernel's tail

    auto issue = [&](int m) {       // lane 0: start the copy of map m
        sp::mbar_expect_tx(bar, map_bytes);
        sp::bulk_g2s(a, A.hm + (size_t)m * hw, map_bytes, bar);
    };
    long long static_next = (long long)blockIdx.x * nwarps + warp + round;      // grid-wide mode: this warp's second static map
    int static_left = static_maps - 1;
    auto claim = [&]() {            // lane 0: the map after the ones this warp already holds, or -1
        if (!grid_wide) {
            const int m = atomicAdd(&next_map, 1);
            return (m < range_hi) ? m : -1;
        }
        long long m;
        if (static_left > 0) {
            m = static_next;
            static_next += round;
            --static_left;
        } else {
            m = (long long)static_maps * round + (long long)atomicAdd(&ws->next_work, 1u);
        }
        return (m < A.nmaps) ? (int)m : -1;
    };
    int m = grid_wide ? (int)blockIdx.x * nwarps + warp : range_lo + warp;
    if (m >= (grid_wide ? A.nmaps : range_hi)) m = -1;
    if (lane == 0 && m >= 0) issue(m);
    if (MODE == SP_DECODE_GAUSS_TAYLOR)
        for (int t = threadIdx.x; t < KS * KS; t += blockDim.x) wts[t] = __ldg(A.blur_w + t);
    __syncthreads();
    sp_dec::LaneTaps<KS> taps;
    if (MODE == SP_DECODE_GAUSS_TAYLOR) taps.load(wts, lane);

    double sum_sq = 0.0;
    uint32_t parity = 0;
    while (m >= 0) {
        int ahead = -1;
        if (lane == 0) ahead = claim();                    // its latency hides behind this map's work
        const sp_dec::Affine T = sp_dec::load_affine(A, m);
        const sp_trn::Joint3 jc = sp_trn::load_joint(io, m);
        // float64 Gaussian factors of this map's target while its copy is in flight
        const sp_gauss::JointVerdict jv = sp_trn::prepare_map<0>(io, m, jc, ex, ey, lane);
        sp::mbar_wait(bar, parity);
        parity ^= 1u;
        // Two passes over the staged map, in an order that alternates between neighbouring warps: the loss pass is
        // where the bytes leave (two map-sized store streams), the decode pass is arithmetic only. If every warp
        // decoded first, HBM would idle for the first third of a small launch and be saturated by all the stores at
        // once afterwards.
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {
            if ((pass == 0) == ((warp & 1) != 0)) {
                // ---- target, masked difference, loss partial, gradient (+ target map, + HeatMapAcc argmaxes)
                sp_trn::MapState st;
                sp_trn::begin_map(io, jv, st, lane, ACC);
                sp_trn::run_quads<WRITE_GRAD, WRITE_TARGETS, ACC, true>(io, m, reinterpret_cast<const float4*>(a), 0, hw >> 2, jv,
                                                                        ex, ey, st, lane, io.half_scale);
                if (ACC) sp_trn::end_map_acc(io, m, jv, ex, ey, st, lane);
                sum_sq += (double)st.acc;
            } else if (VAL || A.coords != nullptr) {
                // ---- decode (argmax on the raw map, blur at the 13 stencil points, Taylor step, affine)
                const sp_arg::Peak pk = sp_dec::argmax_smem<false>(a, a, hw, A.W, lane);
                sp_arg::DirectView view{a};
                auto gauss_taylor = [&](int px, int py, float ori_max, float& ox, float& oy) {
                    return sp_dec::taylor_refine_smem<KS>(a, wts, patch, taps, A.H, A.W, px, py, ori_max, lane, ox, oy);
                };
                if constexpr (VAL) {
                    sp_dec::DecodeArgs D = A;
                    D.mode = MODE;                 // the branch of finish_map is chosen at compile time
                    if constexpr (MODE == SP_DECODE_BASIC) {
                        sp_dec::finish_map(D, view, m, pk, lane, T, [](int, int, float, float&, float&) { return false; });
                    } else {
                        sp_dec::finish_map(D, view, m, pk, lane, T, gauss_taylor);
                    }
                    // lane 0 stored this map's (x, y, conf) in the row; the warp that completes the person reads the K
                    // peaks in parallel (lane 0's acquire reaches the other lanes through __syncwarp), then every lane
                    // adds them up in joint order
                    const int person = m / A.K;
                    unsigned arrived = 0u;
                    if (lane == 0) arrived = sp::atomic_add_acq_rel(V.arrivals + person, 1u);
                    if (__shfl_sync(SP_FULL, arrived, 0) == (unsigned)A.K - 1u) {
                        __syncwarp();
                        float* r = A.rows + (size_t)person * A.row_stride;
                        sp::PersonScore score = sp::PersonScore::start();
                        for (int k0 = 0; k0 < A.K; k0 += 32) {
                            const float mine = (k0 + lane < A.K) ? __ldcg(r + 3 * (k0 + lane) + 2) : 0.f;
                            const int n = min(32, A.K - k0);
                            for (int j = 0; j < n; ++j) score.add(__shfl_sync(SP_FULL, mine, j));
                        }
                        if (lane == 0) {
                            r[3 * A.K] = score.value(A.K);
                            V.arrivals[person] = 0u;
                        }
                    }
                } else {
                    sp_dec::finish_map(A, view, m, pk, lane, T, gauss_taylor);
                }
            }
        }
        __syncwarp();               // every lane is done with the staged map and the factors
        if (lane == 0 && ahead >= 0) {
            sp::fence_proxy_async_smem();
            issue(ahead);
        }
        m = __shfl_sync(SP_FULL, ahead, 0);
    }
    // the last block also returns ws->next_work to zero
    const bool last = sp_reduce::finish_loss<512>(sum_sq, ws, loss, inv_count);
    if constexpr (VAL) {
        // every staged map is consumed: the counters go where the per-warp areas were
        if (last) sp_arg::heatmap_acc_block<true>(io.pred_xy, io.label_xy, V.acc, V.B, A.K, V.norm_x, V.norm_y, V.thresh,
                                                  reinterpret_cast<int*>(smem + kHeadBytes + kWtsBytes));
    }
}

template <bool WRITE_GRAD, bool WRITE_TARGETS, bool ACC>
__global__ void __launch_bounds__(512, 1)
step_kernel(const sp_dec::DecodeArgs A, const sp_trn::MapIo io, float* __restrict__ loss, MseWorkspace* __restrict__ ws,
            double inv_count, int nwarps, int static_maps) {
    step_body<WRITE_GRAD, WRITE_TARGETS, ACC, SP_DECODE_GAUSS_TAYLOR, false>(A, io, loss, ws, inv_count, nwarps, static_maps,
                                                                              ValOut{});
}

template <int MODE>
__global__ void __launch_bounds__(512, 1)
val_step_kernel(const sp_dec::DecodeArgs A, const sp_trn::MapIo io, float* __restrict__ loss, MseWorkspace* __restrict__ ws,
                double inv_count, int nwarps, int static_maps, const ValOut V) {
    step_body<false, false, true, MODE, true>(A, io, loss, ws, inv_count, nwarps, static_maps, V);
}

// Launch shape of step_kernel / val_step_kernel for B*K = nmaps maps of H x W. SP_ERR_UNSUPPORTED when not even one
// map fits in shared memory.
struct StepLayout {
    int nwarps, grid, static_maps;
    size_t smem;
};
int plan_step(int nmaps, int H, int W, StepLayout& L) {
    const size_t map_bytes = (size_t)H * W * 4;
    const int wpad = (W + 1) & ~1;
    const size_t fac_bytes = (size_t)(wpad + ((H + 1) & ~1)) * sizeof(double);
    const size_t budget = 226 * 1024 - kHeadBytes - kWtsBytes;      // 1 KB spare for static shared memory (loss reduction)
    const size_t per_warp1 = kPatchBytes + fac_bytes + map_bytes;
    int fit = (int)(budget / per_warp1);
    SP_RETURN_IF(fit < 1, SP_ERR_UNSUPPORTED);
    if (fit > 16) fit = 16;
    const int sms = sp_sm_count();
    // Small launches (at batch 128: 2176 maps on 148 SMs = 14.7 per SM, and 15 warps fit): one map per warp, as many
    // warps as fit, so that every map is resident at once and the launch is a single round (20.0 us at batch 128 with
    // 15 warps, 22-23 us with 8-12), maps taken from per-CTA ranges. Larger launches: FEWER warps (every warp reads one
    // stream and writes two; 9-12 warps per SM measure the same at 1024 x 64x48, 14 and more lose 1-4 %, 7 loses 7 %)
    // and maps dealt grid-wide, 80 % of a warp's share interleaved statically and the tail claimed dynamically:
    // 1024 x 64x48 113.0 -> 108.0 us, 2048: 212.5 -> 204.6 us (0.96 of the HBM peak), 512 x 96x72: 131 -> 125 us,
    // 384 x 64x48: 51.9 -> 47.3 us. A purely static interleaved assignment loses again (119.8 us with 10 warps).
    const SpTuning& tune = sp_tuning();
    const bool large = 2LL * nmaps >= 3LL * fit * sms;       // more than one and a half rounds of one map per warp
    int nwarps = large ? (fit >= 14 ? 9 : (fit + 1) / 2 + (fit >= 6 ? 2 : 0)) : fit;
    nwarps = sp_knob(tune.step_warps, nwarps);
    if (nwarps < 1) nwarps = 1;
    if (nwarps > fit) nwarps = fit;
    int grid = sms;
    const int need = (nmaps + nwarps - 1) / nwarps;
    if (grid > need) grid = need;
    // large launches: maps dealt grid-wide; SP_STEP_STATIC_PCT % of a warp's expected share is fixed up front (no atomic),
    // the rest is claimed dynamically. Tried and dropped for this kernel (numbers in DESIGN.md section 4): a second stage per
    // warp (123.5 vs 114.0 us at 1024 x 64x48) and the period-tiled loss pass of the fused training kernel (123 vs 113 us).
    int static_maps = 0;
    if (large || sp_knob(tune.step_static_pct, -1) >= 0) {
        const long long share = (long long)nmaps / ((long long)grid * nwarps);
        int pct = sp_knob(tune.step_static_pct, 80);
        if (pct > 100) pct = 100;
        long long dynamic = share * (100 - pct) / 100;
        if (dynamic > 8) dynamic = 8;              // the tail to even out is a few maps per warp whatever the launch size
        static_maps = (int)(share - dynamic);
        if (static_maps < 1) static_maps = 1;
    }
    L.nwarps = nwarps;
    L.grid = grid;
    L.static_maps = static_maps;
    L.smem = kHeadBytes + kWtsBytes + (size_t)nwarps * per_warp1;
    return 0;
}

sp_dec::DecodeArgs step_decode_args(const float* pred, const float* trans_inv, const float* blur_w, float* coords,
                                    float* maxval, float* rows, int B, int K, int H, int W, int mode) {
    sp_dec::DecodeArgs A;
    A.hm = pred; A.hm_flip = nullptr; A.perm = nullptr; A.trans_inv = trans_inv; A.blur_w = blur_w;
    A.coords = coords; A.maxval = maxval; A.argmax = nullptr; A.rows = rows; A.row_stride = rows ? 3 * K + 1 : 0;
    A.nmaps = B * K; A.K = K; A.H = H; A.W = W; A.ksize = 11; A.mode = mode; A.work = nullptr;
    return A;
}

sp_trn::MapIo step_io(const float* joints, const float* pred, float* grad, float* targets, float* weights, float* pred_xy,
                      float* label_xy, int B, int K, int H, int W, double sigma, float grad_scale) {
    const double count = (double)B * (double)K * (double)H * (double)W;
    sp_trn::MapIo io;
    io.joints = joints; io.pred = pred; io.grad = grad; io.targets = targets; io.weights = weights;
    io.pred_xy = reinterpret_cast<float2*>(pred_xy); io.label_xy = reinterpret_cast<float2*>(label_xy);
    io.nmaps = B * K; io.H = H; io.W = W; io.reach = (float)(sigma * 3.0); io.denom = 2.0 * (sigma * sigma);
    io.norm = (float)(2.0 / count); io.half_scale = 0.5f * grad_scale; io.scale_dev = nullptr;
    io.analytic_ok = (sigma >= 0.25 && sigma <= 64.0) ? 1 : 0;
    return io;
}

// validation workspace: the reduction workspace, then the per-person arrival counters, then room for the argmax axes
size_t val_arrivals_offset() { return (sizeof(MseWorkspace) + 15) & ~(size_t)15; }
size_t val_axes_offset(int B) { return val_arrivals_offset() + (((size_t)B * 4 + 15) & ~(size_t)15); }

}  // namespace

extern "C" int sp_step_f32(const float* joints, const float* pred, const float* trans_inv, const float* blur_w,
                           float* targets, float* weights, float* grad, float* loss, float* coords, float* maxval,
                           float* pred_xy, float* label_xy, void* workspace, size_t workspace_bytes,
                           int B, int K, int H, int W, double sigma, int ksize, float grad_scale, void* stream) {
    SP_RETURN_IF(!joints || !pred || !blur_w || !loss || !workspace, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((coords == nullptr) != (maxval == nullptr), SP_ERR_BAD_ARGUMENT);      // both NULL: no decode pass
    SP_RETURN_IF(B <= 0 || K <= 0 || H <= 0 || W <= 0 || !(sigma > 0.0), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((pred_xy == nullptr) != (label_xy == nullptr), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((long long)B * K > 0x7fffffffLL || (long long)H * W > (1 << 24), SP_ERR_UNSUPPORTED);
    SP_RETURN_IF(W % 4 != 0 || ksize != 11, SP_ERR_UNSUPPORTED);      // callers compose the stand-alone kernels instead
    SP_RETURN_IF(workspace_bytes < sizeof(MseWorkspace), SP_ERR_WORKSPACE);
    SP_RETURN_IF(!sp_aligned16(workspace) || !sp_aligned16(pred) || (grad && !sp_aligned16(grad)) || (targets && !sp_aligned16(targets)) ||
                 (coords && !sp_aligned16(coords)) || (pred_xy && (!sp_aligned16(pred_xy) || !sp_aligned16(label_xy))), SP_ERR_BAD_ALIGNMENT);
    StepLayout L;
    const int bad = plan_step(B * K, H, W, L);
    if (bad != 0) return bad;
    const sp_dec::DecodeArgs A = step_decode_args(pred, trans_inv, blur_w, coords, maxval, nullptr, B, K, H, W,
                                                  SP_DECODE_GAUSS_TAYLOR);
    const sp_trn::MapIo io = step_io(joints, pred, grad, targets, weights, pred_xy, label_xy, B, K, H, W, sigma, grad_scale);
    const double count = (double)B * (double)K * (double)H * (double)W;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MseWorkspace* ws = static_cast<MseWorkspace*>(workspace);
    const int sel = (grad ? 4 : 0) | (targets ? 2 : 0) | (pred_xy ? 1 : 0);
#define SP_LAUNCH_STEP(G, T, AC) \
    SP_CUDA(sp_launch_smem(step_kernel<G, T, AC>, dim3(L.grid), dim3(L.nwarps * 32), L.smem, st, A, io, loss, ws, 1.0 / count, L.nwarps, L.static_maps))
    switch (sel) {
        case 0: SP_LAUNCH_STEP(false, false, false); break;
        case 1: SP_LAUNCH_STEP(false, false, true); break;
        case 2: SP_LAUNCH_STEP(false, true, false); break;
        case 3: SP_LAUNCH_STEP(false, true, true); break;
        case 4: SP_LAUNCH_STEP(true, false, false); break;
        case 5: SP_LAUNCH_STEP(true, false, true); break;
        case 6: SP_LAUNCH_STEP(true, true, false); break;
        default: SP_LAUNCH_STEP(true, true, true); break;
    }
#undef SP_LAUNCH_STEP
    return 0;
}

extern "C" size_t sp_val_step_workspace_bytes(int B, int K) {
    if (B <= 0 || K <= 0) return val_arrivals_offset();
    return val_axes_offset(B) + 2 * (size_t)B * K * sizeof(float2);
}

extern "C" int sp_val_step_f32(const float* joints, const float* pred, const float* trans_inv, const float* blur_w, int mode,
                               float* weights, float* loss, float* acc, float* rows, float* coords, float* maxval,
                               float* pred_xy, float* label_xy, void* workspace, size_t workspace_bytes,
                               int B, int K, int H, int W, double sigma, int ksize, float distance_thresh, float norm_frac,
                               void* stream) {
    SP_RETURN_IF(mode != SP_DECODE_GAUSS_TAYLOR && mode != SP_DECODE_BASIC, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!joints || !pred || !loss || !acc || !rows || !workspace, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(mode == SP_DECODE_GAUSS_TAYLOR && !blur_w, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((coords == nullptr) != (maxval == nullptr), SP_ERR_BAD_ARGUMENT);      // both NULL: rows only
    SP_RETURN_IF((pred_xy == nullptr) != (label_xy == nullptr), SP_ERR_BAD_ARGUMENT);  // both NULL: in the workspace
    SP_RETURN_IF(B <= 0 || K <= 0 || H <= 0 || W <= 0 || !(sigma > 0.0) || !(norm_frac > 0.f), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((long long)B * K > 0x7fffffffLL / 3 || (long long)H * W > (1 << 24), SP_ERR_UNSUPPORTED);
    SP_RETURN_IF(W % 4 != 0 || (mode == SP_DECODE_GAUSS_TAYLOR && ksize != 11), SP_ERR_UNSUPPORTED);   // compose instead
    SP_RETURN_IF(workspace_bytes < sp_val_step_workspace_bytes(B, K), SP_ERR_WORKSPACE);
    SP_RETURN_IF(!sp_aligned16(workspace) || !sp_aligned16(pred) || (coords && !sp_aligned16(coords)) ||
                 (pred_xy && (!sp_aligned16(pred_xy) || !sp_aligned16(label_xy))), SP_ERR_BAD_ALIGNMENT);
    StepLayout L;
    const int bad = plan_step(B * K, H, W, L);
    if (bad != 0) return bad;
    // the HeatMapAcc counters reuse the per-warp areas of the last CTA
    SP_RETURN_IF((size_t)2 * K * sizeof(int) > L.smem - kHeadBytes - kWtsBytes, SP_ERR_UNSUPPORTED);
    unsigned char* wsb = static_cast<unsigned char*>(workspace);
    if (!pred_xy) {
        pred_xy = reinterpret_cast<float*>(wsb + val_axes_offset(B));
        label_xy = pred_xy + 2 * (size_t)B * K;
    }
    const sp_dec::DecodeArgs A = step_decode_args(pred, trans_inv, blur_w, coords, maxval, rows, B, K, H, W, mode);
    const sp_trn::MapIo io = step_io(joints, pred, nullptr, nullptr, weights, pred_xy, label_xy, B, K, H, W, sigma, 1.f);
    const double count = (double)B * (double)K * (double)H * (double)W;
    ValOut V;
    V.arrivals = reinterpret_cast<unsigned int*>(wsb + val_arrivals_offset());
    V.acc = acc;
    V.norm_x = (float)W / norm_frac;           // norm = tensor([W, H], float32) / norm_frac, as sp_heatmap_acc_f32
    V.norm_y = (float)H / norm_frac;
    V.thresh = distance_thresh;
    V.B = B;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MseWorkspace* ws = static_cast<MseWorkspace*>(workspace);
    if (mode == SP_DECODE_BASIC) {
        SP_CUDA(sp_launch_smem(val_step_kernel<SP_DECODE_BASIC>, dim3(L.grid), dim3(L.nwarps * 32), L.smem, st, A, io, loss, ws,
                               1.0 / count, L.nwarps, L.static_maps, V));
    } else {
        SP_CUDA(sp_launch_smem(val_step_kernel<SP_DECODE_GAUSS_TAYLOR>, dim3(L.grid), dim3(L.nwarps * 32), L.smem, st, A, io,
                               loss, ws, 1.0 / count, L.nwarps, L.static_maps, V));
    }
    return 0;
}
