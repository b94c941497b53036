// A2: masked joints-MSE, forward and backward in one pass
// (reference processors/dp_pose_hrnet_solver.py:86,106-107:
//  loss = 0.5 * MSELoss(pred * mask[..., None, None], target * mask[..., None, None]); loss.backward()).
//
// HBM-bound: reads pred and target once, writes grad once (3 streams; the ATen sequence makes
// ~6 passes and two temporaries).
//
// Main kernel (mse_ring_kernel): persistent, one CTA per SM. A CTA owns a contiguous range of
// fixed-size chunks (a chunk never straddles a map, so the mask is one scalar per chunk) and deals
// them round-robin to its warps, so at any moment the SM reads and writes ONE contiguous window of
// a few tens of KB -- HBM row-buffer friendly -- instead of one stream per warp. Every warp owns a
// small ring of shared-memory slots filled by 1-D TMA bulk copies (pred chunk + target chunk on one
// mbarrier); it consumes a slot with 16-byte shared loads, stores the gradient with coalesced
// 16-byte global stores and re-arms the slot at once. Measured on B200 (scratch/stream_bench.cu):
// for a 2-reads-1-write stream ~50-100 KB in flight per SM in few, large requests beats both the
// classic "many threads, one float4 each" loop (-8 %) and deeper rings (HBM read/write turnarounds).
// Plain-load kernel (mse_plain_kernel, every dtype of pred): float16 / bfloat16 pred, backward-only calls, a
// device-side upstream gradient, the SKIP_MASKED variant, any shape / alignment, and SP_LOSS_FORCE_LDG.
//
// The sum of squares is accumulated per thread in float32 over a few elements, then in float64;
// block partials go to the caller's workspace and the last block to finish adds them in a fixed
// order (deterministic, no floating-point atomics) and writes the scalar loss.
//
// Arithmetic follows ATen so that grad is bit-identical for finite inputs:
//   d = fl(m*p) - fl(m*t); grad = ((fl(2/N) * d) * 0.5) * m   (mse_loss_backward, then mul backward)
//
// ACC (forward calls of sp_mse_acc_fwd_bwd): the same pass also finds the argmax of both masked maps, m*p and m*t,
// which is what HeatMapAcc()(pred.mul(mask), target.mul(mask)) decodes (metrics/pose_metrics.py:223-224), and the
// last block runs the HeatMapAcc epilogue. A map may be split over lanes, warps and blocks (the ring kernel cuts its
// ranges by chunk count), so every partial argmax becomes a 64-bit key whose unsigned order is sp::better's and the
// partials meet in one atomicMax per (map, warp that scanned part of it) -- the result cannot depend on the split.
// The running argmax, its warp merge, the exact scan and the epilogue are those of sp_argmax.cuh, which the decode,
// fused training and step kernels use as well.
#include "sp_common.cuh"
#include "sp_reduce.cuh"
#include "sp_lowp.cuh"
#include "sp_argmax.cuh"

#ifdef SP_TRAIN_TRACE
__device__ long long* g_loss_trace_ptr = nullptr;     // scratch instrumentation, trace build only
extern "C" int sp_debug_set_loss_trace(void* p) { return (int)cudaMemcpyToSymbol(g_loss_trace_ptr, &p, sizeof(p)); }
__device__ __forceinline__ long long loss_gtime() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#endif

namespace {

using namespace sp_reduce;
constexpr int kThreads = 256;

__device__ __forceinline__ float sq_err_and_grad(float p, float t, float m, float norm, float half_scale, float& g) {
    const float d = __fsub_rn(__fmul_rn(m, p), __fmul_rn(m, t));
    g = __fmul_rn(__fmul_rn(__fmul_rn(norm, d), half_scale), m);
    return d;
}

// ---- HeatMapAcc riding along with the loss (ACC) ------------------------------------------------------------------
struct AccOut {
    unsigned long long* keys;    // [B*K][2] argmax keys of (m*p, m*t) in the caller's workspace, zero between launches
    float2* pred_xy;             // [B*K] heat_map_to_axis of m*p / m*t (the caller's buffers or the workspace's)
    float2* label_xy;
    float* acc;
    int B, K, W;
    float norm_x, norm_y, thresh;
};

// High word: the value in an order where NaN is above +inf and -0 == +0; low word: ~index, so the smaller index wins
// among equal values (and among NaNs). Key 0 is below every element: a map nobody scanned.
__device__ __forceinline__ unsigned long long argmax_key(float v, int i) {
    unsigned int o = 0xffffffffu;
    if (v == v) {
        const unsigned int b = __float_as_uint(v == 0.f ? 0.f : v);
        o = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
    }
    return ((unsigned long long)o << 32) | (unsigned int)~i;
}

// heat_map_to_axis of a merged key; key 0 (a map whose mask is 0: its products are 0 or NaN) gives (0, 0) as well
__device__ __forceinline__ float2 key_axis(unsigned long long key, int W) {
    const unsigned int o = (unsigned int)(key >> 32);
    const float v = (o == 0xffffffffu || o == 0u) ? CUDART_NAN_F : __uint_as_float((o & 0x80000000u) ? (o ^ 0x80000000u) : ~o);
    return sp_arg::axis_of(v, (int)~(unsigned int)key, W);
}

// One warp's share of a map seen through QuadBest (each lane visits its quads in increasing order; 4*bq + bsub is the
// flat index relative to `first`) merged into the map's key. A NaN or an infinity among them: the exact scan of the
// n elements at `src` (a superset of what the warp saw, starting at flat index `first`) decides instead.
template <typename PT>
__device__ __forceinline__ void merge_quads(const sp_arg::QuadBest& b, const PT* src, float mk, int n, int first, int lane,
                                            unsigned long long* key) {
    sp_arg::Peak pk;
    if (__any_sync(SP_FULL, b.poison != b.poison)) {
        pk = sp_arg::argmax_exact(sp_arg::MaskedPredView<PT>{src, mk}, n, lane);
    } else {
        pk = b.warp_peak();
        if (pk.value == -CUDART_INF_F) return;   // the warp had no element of this map (an infinity is poison)
    }
    if (lane == 0) atomicMax(key, argmax_key(pk.value, first + pk.index));
}

// Scalar paths: this lane's first maximal element by sp::better, merged over the warp, then into the map's key.
__device__ __forceinline__ void merge_scalar(float bv, int bi, int lane, unsigned long long* key) {
    const sp_arg::Peak pk = sp_arg::warp_best(bv, bi);
    if (lane == 0 && pk.index != 0x7fffffff) atomicMax(key, argmax_key(pk.value, pk.index));
}

// Run by ALL threads of the last block of the loss reduction (it has acquired every block's keys): the keys become
// heat_map_to_axis coordinates and return to zero, then the HeatMapAcc epilogue of heatmap_acc_kernel / val_step_kernel.
// counters: 2K ints of shared memory.
__device__ __forceinline__ void acc_epilogue(const AccOut& A, int* counters) {
    const int n = A.B * A.K;
    ulonglong2* keys = reinterpret_cast<ulonglong2*>(A.keys);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const ulonglong2 k = __ldcg(keys + i);
        keys[i] = make_ulonglong2(0ull, 0ull);
        A.pred_xy[i] = key_axis(k.x, A.W);
        A.label_xy[i] = key_axis(k.y, A.W);
    }
    __syncthreads();
    sp_arg::heatmap_acc_block<true>(A.pred_xy, A.label_xy, A.acc, A.B, A.K, A.norm_x, A.norm_y, A.thresh, counters);
}

// The plain-load kernel: one CTA per map at a time, grid-stride over the maps. It serves every call the ring kernel does
// not take: float16 / bfloat16 `pred`, backward-only calls, a device-side upstream gradient, SKIP_MASKED, any shape and
// alignment. `pred` arrives in PT (float32, or the autocast dtype float16 / bfloat16 of processors/dp_pose_hrnet_solver.py:
// 111-120) and the gradient leaves in PT. The arithmetic is what autocast runs: `pred.mul(mask)` promotes to float32,
// mse_loss is on autocast's float32 list, the backward of the promoted product casts d loss / d pred to PT once, AFTER
// the upstream gradient (GradScaler's scale, read here from device memory so that no host sync is needed) has been
// applied in float32 -- which is the whole point of loss scaling for float16.
// VEC (HW % E == 0, pred / target / grad 16-byte aligned): a step is one 16-byte load of pred, E = 16 / sizeof(PT)
// elements (4 floats or 8 halves), E / 4 float4 loads of target and one 16-byte grad store.
// loss == nullptr: backward only (no reduction); grad == nullptr: forward only. ACC only with loss != nullptr.
template <typename PT, bool VEC, bool ACC>
__global__ void __launch_bounds__(kThreads)
mse_plain_kernel(const PT* __restrict__ pred, const float* __restrict__ target, const float* __restrict__ mask,
                 PT* __restrict__ grad, float* __restrict__ loss, MseWorkspace* __restrict__ ws, int nmaps, int hw,
                 float norm, float half_scale_host, const float* __restrict__ scale_dev, double inv_count, int skip_masked,
                 const AccOut A) {
    constexpr int E = 16 / sizeof(PT);
    constexpr int kLogE = E == 4 ? 2 : 3;
    constexpr int Q = E / 4;                      // quads per step
    constexpr int kUnroll = Q == 1 ? 4 : 2;
    double block_sum = 0.0;
    sp::grid_dep_wait();
    const float half_scale = scale_dev ? __fmul_rn(half_scale_host, __ldg(scale_dev)) : half_scale_host;
    const bool write_grad = grad != nullptr;
    const int lane = threadIdx.x & 31;

    for (int m = blockIdx.x; m < nmaps; m += gridDim.x) {
        const float mk = __ldg(mask + m);
        const size_t base = (size_t)m * hw;
        float acc = 0.f;
        const bool track = ACC && mk != 0.f;      // a masked-out map's products are 0 or NaN: (0, 0) either way
        if (skip_masked && mk == 0.f) {
            if (write_grad) {
                if (VEC) {
                    uint4* g16 = reinterpret_cast<uint4*>(grad + base);
                    for (int o = threadIdx.x; o < (hw >> kLogE); o += kThreads) g16[o] = make_uint4(0u, 0u, 0u, 0u);
                } else {
                    for (int i = threadIdx.x; i < hw; i += kThreads) grad[base + i] = sp_lowp::from_float<PT>(0.f);
                }
            }
            continue;
        }
        if (VEC) {
            const float4* t4 = reinterpret_cast<const float4*>(target + base);
            const int nv = hw >> kLogE;
            sp_arg::QuadBest bp, bt;
            if (ACC) { bp.init(); bt.init(); }
#pragma unroll kUnroll
            for (int o = threadIdx.x; o < nv; o += kThreads) {
                float p[E], t[E], g[E];
                sp_lowp::load_group(pred + base + E * (size_t)o, p);
#pragma unroll
                for (int h = 0; h < Q; ++h) {
                    const float4 v = sp_lowp::ldg_stream4(t4 + Q * o + h);
                    t[4 * h] = v.x; t[4 * h + 1] = v.y; t[4 * h + 2] = v.z; t[4 * h + 3] = v.w;
                }
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const float d = sq_err_and_grad(p[e], t[e], mk, norm, half_scale, g[e]);
                    acc = fmaf(d, d, acc);
                }
                if (write_grad) sp_lowp::store_group(grad + base + E * (size_t)o, g);
                // float(p) * m: the float32 promotion autocast's pred.mul(mask) computes. Pushed for untracked maps too
                // (their state is never merged): a branch on `track` made the ACC calls 0.6-7 % slower.
                if (ACC) {
#pragma unroll
                    for (int h = 0; h < Q; ++h) {
                        bp.push(__fmul_rn(mk, p[4 * h]), __fmul_rn(mk, p[4 * h + 1]), __fmul_rn(mk, p[4 * h + 2]),
                                __fmul_rn(mk, p[4 * h + 3]), Q * o + h);
                        bt.push(__fmul_rn(mk, t[4 * h]), __fmul_rn(mk, t[4 * h + 1]), __fmul_rn(mk, t[4 * h + 2]),
                                __fmul_rn(mk, t[4 * h + 3]), Q * o + h);
                    }
                }
            }
            if (ACC && track) {
                merge_quads(bp, pred + base, mk, hw, 0, lane, A.keys + 2 * (size_t)m);
                merge_quads(bt, target + base, mk, hw, 0, lane, A.keys + 2 * (size_t)m + 1);
            }
        } else {
            float bvp = -CUDART_INF_F, bvt = -CUDART_INF_F;
            int bip = 0x7fffffff, bit = 0x7fffffff;
            for (int i = threadIdx.x; i < hw; i += kThreads) {
                float g;
                const float pv = sp_lowp::to_float(pred[base + i]), tv = target[base + i];
                const float d = sq_err_and_grad(pv, tv, mk, norm, half_scale, g);
                acc = fmaf(d, d, acc);
                if (write_grad) grad[base + i] = sp_lowp::from_float<PT>(g);
                if (ACC && track) {
                    const float mp = __fmul_rn(mk, pv), mt = __fmul_rn(mk, tv);
                    if (sp::better(mp, i, bvp, bip)) { bvp = mp; bip = i; }
                    if (sp::better(mt, i, bvt, bit)) { bvt = mt; bit = i; }
                }
            }
            if (ACC && track) {
                merge_scalar(bvp, bip, lane, A.keys + 2 * (size_t)m);
                merge_scalar(bvt, bit, lane, A.keys + 2 * (size_t)m + 1);
            }
        }
        block_sum += (double)acc;
    }
    if (loss != nullptr) {
        const bool last = finish_loss<kThreads>(block_sum, ws, loss, inv_count);
        if constexpr (ACC) {
            extern __shared__ int acc_counters[];     // 2K ints
            if (last) acc_epilogue(A, acc_counters);
        }
    }
}

// dynamic smem: [mbarriers 1024 B][per warp: ring x (pred chunk | target chunk)]
constexpr int kRingBarBytes = 1024;

// A variant that sent the gradient out through the TMA too (written into the drained slot, cp.async.bulk shared -> global)
// was within 1-2 % either way warm and 12 % slower from a cold cache, so the gradient stays on register stores (DESIGN.md, section 4).
// ACC: the argmax is taken over each staged chunk before its slot is re-armed (the exact scan of a chunk holding a NaN
// or an infinity reads the slot too); the last block's HeatMapAcc counters go where the slots were.
template <bool WRITE_GRAD, bool ACC>
__global__ void __launch_bounds__(1024, 1)
mse_ring_kernel(const float* __restrict__ pred, const float* __restrict__ target, const float* __restrict__ mask,
                float* __restrict__ grad, float* __restrict__ loss, MseWorkspace* __restrict__ ws,
                long long nchunks, int chunk_quads, int chunks_per_map, int nwarps, int ring,
                float norm, float half_scale, double inv_count, const AccOut A) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const uint32_t chunk_bytes = (uint32_t)chunk_quads * 16u;
    const size_t chunk_floats = (size_t)chunk_quads * 4;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw) + warp * ring;
    unsigned char* slots = smem_raw + kRingBarBytes + (size_t)warp * ring * 2 * chunk_bytes;
    if (lane == 0) {
        for (int r = 0; r < ring; ++r) sp::mbar_init(bars + r, 1);
        sp::mbar_fence_init();
    }
    __syncwarp();
    const long long lo = (long long)blockIdx.x * nchunks / gridDim.x;
    const long long hi = (long long)(blockIdx.x + 1) * nchunks / gridDim.x;
    sp::grid_dep_wait();            // the prologue above overlapped the previous kernel's tail
#ifdef SP_TRAIN_TRACE
    const long long trace_t0 = loss_gtime();
#endif

    long long pi = lo + warp;       // producer cursor (lane 0): next chunk to request, into slot ps
    int ps = 0;
    auto issue_next = [&]() {
        if (pi >= hi) return;
        unsigned char* dst = slots + (size_t)ps * 2 * chunk_bytes;
        sp::mbar_expect_tx(bars + ps, 2 * chunk_bytes);
        sp::bulk_g2s(dst, pred + pi * chunk_floats, chunk_bytes, bars + ps);
        sp::bulk_g2s(dst + chunk_bytes, target + pi * chunk_floats, chunk_bytes, bars + ps);
        pi += nwarps;
        if (++ps == ring) ps = 0;
    };
    if (lane == 0)
        for (int r = 0; r < ring; ++r) issue_next();

    double sum_sq = 0.0;
    int cs = 0;
    uint32_t parity = 0;
    for (long long i = lo + warp; i < hi; i += nwarps) {
        const float mk = __ldg(mask + i / chunks_per_map);          // latency hidden behind the wait below
        sp::mbar_wait(bars + cs, parity);
        const float4* p4 = reinterpret_cast<const float4*>(slots + (size_t)cs * 2 * chunk_bytes);
        const float4* t4 = reinterpret_cast<const float4*>(slots + (size_t)cs * 2 * chunk_bytes + chunk_bytes);
        float4* g4 = reinterpret_cast<float4*>(grad + i * chunk_floats);
        float acc = 0.f;
        const bool track = ACC && mk != 0.f;
        sp_arg::QuadBest bp, bt;
        if (ACC) { bp.init(); bt.init(); }
#pragma unroll 3
        for (int q = lane; q < chunk_quads; q += 32) {
            const float4 p = p4[q];
            const float4 t = t4[q];
            float4 g;
            float d;
            d = sq_err_and_grad(p.x, t.x, mk, norm, half_scale, g.x); acc = fmaf(d, d, acc);
            d = sq_err_and_grad(p.y, t.y, mk, norm, half_scale, g.y); acc = fmaf(d, d, acc);
            d = sq_err_and_grad(p.z, t.z, mk, norm, half_scale, g.z); acc = fmaf(d, d, acc);
            d = sq_err_and_grad(p.w, t.w, mk, norm, half_scale, g.w); acc = fmaf(d, d, acc);
            if (WRITE_GRAD) g4[q] = g;
            if (ACC && track) {
                bp.push(__fmul_rn(mk, p.x), __fmul_rn(mk, p.y), __fmul_rn(mk, p.z), __fmul_rn(mk, p.w), q);
                bt.push(__fmul_rn(mk, t.x), __fmul_rn(mk, t.y), __fmul_rn(mk, t.z), __fmul_rn(mk, t.w), q);
            }
        }
        sum_sq += (double)acc;
        if (ACC && track) {
            const long long map = i / chunks_per_map;
            const int first = (int)(i - map * chunks_per_map) * (int)chunk_floats;     // the chunk's place in its map
            merge_quads(bp, reinterpret_cast<const float*>(p4), mk, (int)chunk_floats, first, lane, A.keys + 2 * map);
            merge_quads(bt, reinterpret_cast<const float*>(t4), mk, (int)chunk_floats, first, lane, A.keys + 2 * map + 1);
        }
        __syncwarp();
        if (lane == 0) {
            sp::fence_proxy_async_smem();
            issue_next();                                           // refills the slot just drained
        }
        if (++cs == ring) { cs = 0; parity ^= 1u; }
    }
#ifdef SP_TRAIN_TRACE
    if (lane == 0 && g_loss_trace_ptr) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        long long* t = g_loss_trace_ptr + ((size_t)blockIdx.x * 32 + warp) * 4;
        t[0] = trace_t0; t[1] = loss_gtime(); t[2] = smid; t[3] = (long long)(hi - lo);
    }
#endif
    const bool last = finish_loss<1024>(sum_sq, ws, loss, inv_count);
    if constexpr (ACC) {
        if (last) acc_epilogue(A, reinterpret_cast<int*>(smem_raw + kRingBarBytes));
    }
}

__global__ void __launch_bounds__(256)
scale_inplace_kernel(float* __restrict__ data, long long n, const float* __restrict__ scale_dev) {
    sp::grid_dep_wait();
    const float s = __ldg(scale_dev);
    if (s == 1.0f) return;
    const long long n4 = n >> 2;
    float4* d4 = reinterpret_cast<float4*>(data);
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += stride) {
        float4 v = d4[q];
        v.x *= s; v.y *= s; v.z *= s; v.w *= s;
        d4[q] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) data[(n4 << 2) + threadIdx.x] *= s;
}

}  // namespace

extern "C" size_t sp_mse_workspace_bytes(void) { return sizeof(MseWorkspace); }

template <typename PT>
static auto plain_kernel(bool vec, bool acc) {
    return vec ? (acc ? mse_plain_kernel<PT, true, true> : mse_plain_kernel<PT, true, false>)
               : (acc ? mse_plain_kernel<PT, false, true> : mse_plain_kernel<PT, false, false>);
}

// Every entry point after its argument checks. A.acc != nullptr: with the HeatMapAcc argmaxes and epilogue (ACC).
static int mse_launch(const void* pred, int pred_dtype, const float* target, const float* mask, void* grad, float* loss,
                      MseWorkspace* ws, int B, int K, int HW, float grad_scale, const float* grad_scale_dev, int flags,
                      cudaStream_t st, const AccOut& A) {
    const int nmaps = B * K;
    const double count = (double)B * (double)K * (double)HW;
    const float norm = (float)(2.0 / count);       // ATen: norm = 2 / numel, applied in float32
    const float half_scale = 0.5f * grad_scale;    // the 0.5 of the loss expression times upstream grad
    const int per16 = pred_dtype == SP_DTYPE_F32 ? 4 : 8;           // elements of pred in 16 bytes
    const bool vec = (HW % per16 == 0) && sp_aligned16(pred) && sp_aligned16(target) && (!grad || sp_aligned16(grad));
    const int skip = (flags & SP_MSE_SKIP_MASKED) ? 1 : 0;
    const bool acc = A.acc != nullptr;
    const size_t counter_bytes = acc ? (size_t)2 * K * sizeof(int) : 0;      // HeatMapAcc epilogue of the last block

    // ring kernel: float32 forward calls with the upstream gradient on the host; needs 16-byte rows and a chunk size
    // (in quads) that divides the map
    const SpTuning& tune = sp_tuning();
    if (pred_dtype == SP_DTYPE_F32 && loss && !grad_scale_dev && vec && !skip && sp_knob(tune.loss_force_ldg, 0) == 0) {
        const int nq = HW >> 2;
        int want = sp_knob(tune.loss_chunk_quads, 192);           // 3 KB per stream
        if (want < 8) want = 8;
        if (want > 2048) want = 2048;
        int chunk_quads = 0;
        for (int d = want < nq ? want : nq; d >= 8; --d)
            if (nq % d == 0) { chunk_quads = d; break; }
        if (chunk_quads * 2 >= (want < nq ? want : nq)) {            // else: awkward map size, use the plain kernel
            int ring = sp_knob(tune.loss_ring, 3);
            if (ring < 1) ring = 1;
            if (ring > 8) ring = 8;
            int nwarps = sp_knob(tune.loss_warps, 4);   // 4 warps x 3 slots x 6 KB = 72 KB in flight per SM (sweep: profiles/)
            if (nwarps < 1) nwarps = 1;
            if (nwarps > 32) nwarps = 32;
            const size_t slot_bytes = (size_t)chunk_quads * 32;      // pred chunk + target chunk
            while (nwarps > 1 && (kRingBarBytes + (size_t)nwarps * ring * slot_bytes > 226 * 1024 || nwarps * ring * 8 > kRingBarBytes)) --nwarps;
            size_t smem = kRingBarBytes + (size_t)nwarps * ring * slot_bytes;
            if (smem <= 226 * 1024 && nwarps * ring * 8 <= kRingBarBytes) {    // 1 KB spare for static shared memory
                const long long nchunks = (long long)nmaps * (nq / chunk_quads);
                int grid = sp_sm_count();
                if ((long long)grid * nwarps > nchunks) grid = (int)((nchunks + nwarps - 1) / nwarps);
                if (acc && smem < kRingBarBytes + counter_bytes) smem = kRingBarBytes + counter_bytes;
#define SP_LAUNCH_RING(G, AC) \
    SP_CUDA(sp_launch_smem(mse_ring_kernel<G, AC>, dim3(grid), dim3(nwarps * 32), smem, st, pred, target, mask, grad, loss, ws, \
                           nchunks, chunk_quads, nq / chunk_quads, nwarps, ring, norm, half_scale, 1.0 / count, A))
                if (acc) { if (grad) SP_LAUNCH_RING(true, true); else SP_LAUNCH_RING(false, true); }
                else     { if (grad) SP_LAUNCH_RING(true, false); else SP_LAUNCH_RING(false, false); }
#undef SP_LAUNCH_RING
                return 0;
            }
        }
    }

    int grid = sp_sm_count() * 8;
    if (grid > nmaps) grid = nmaps;
    if (grid > kMaxPartials) grid = kMaxPartials;
    auto launch = [&](auto kernel) {
        SP_CUDA(sp_launch(kernel, dim3(grid), dim3(kThreads), counter_bytes, st, pred, target, mask, grad, loss, ws, nmaps, HW,
                          norm, half_scale, grad_scale_dev, 1.0 / count, skip, A));
        return 0;
    };
    if (pred_dtype == SP_DTYPE_F16) return launch(plain_kernel<__half>(vec, acc));
    if (pred_dtype == SP_DTYPE_BF16) return launch(plain_kernel<__nv_bfloat16>(vec, acc));
    return launch(plain_kernel<float>(vec, acc));
}

extern "C" int sp_mse_fwd_bwd_f32(const float* pred, const float* target, const float* mask,
                                  float* grad, float* loss, void* workspace, size_t workspace_bytes,
                                  int B, int K, int HW, float grad_scale, int flags, void* stream) {
    SP_RETURN_IF(!pred || !target || !mask || !loss || !workspace, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(B <= 0 || K <= 0 || HW <= 0, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((long long)B * K > 0x7fffffffLL, SP_ERR_UNSUPPORTED);
    SP_RETURN_IF(workspace_bytes < sizeof(MseWorkspace), SP_ERR_WORKSPACE);
    SP_RETURN_IF(!sp_aligned16(workspace), SP_ERR_BAD_ALIGNMENT);
    return mse_launch(pred, SP_DTYPE_F32, target, mask, grad, loss, static_cast<MseWorkspace*>(workspace), B, K, HW, grad_scale,
                      nullptr, flags, static_cast<cudaStream_t>(stream), AccOut{});
}

extern "C" int sp_mse_fwd_bwd(const void* pred, int pred_dtype, const float* target, const float* mask,
                              void* grad, float* loss, void* workspace, size_t workspace_bytes,
                              int B, int K, int HW, float grad_scale, const float* grad_scale_dev, int flags, void* stream) {
    SP_RETURN_IF(pred_dtype != SP_DTYPE_F32 && pred_dtype != SP_DTYPE_F16 && pred_dtype != SP_DTYPE_BF16, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!loss && !grad, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!pred || !target || !mask || (loss && !workspace), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(B <= 0 || K <= 0 || HW <= 0, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((long long)B * K > 0x7fffffffLL, SP_ERR_UNSUPPORTED);
    if (loss) {
        SP_RETURN_IF(workspace_bytes < sizeof(MseWorkspace), SP_ERR_WORKSPACE);
        SP_RETURN_IF(!sp_aligned16(workspace), SP_ERR_BAD_ALIGNMENT);
    }
    return mse_launch(pred, pred_dtype, target, mask, grad, loss, static_cast<MseWorkspace*>(workspace), B, K, HW, grad_scale,
                      grad_scale_dev, flags, static_cast<cudaStream_t>(stream), AccOut{});
}

// workspace of sp_mse_acc_fwd_bwd: the reduction workspace, the argmax keys (16 bytes per map), room for the axes (16 bytes
// per map, used when the caller passes no pred_xy / label_xy)
static size_t acc_keys_offset() { return (sizeof(MseWorkspace) + 15) & ~(size_t)15; }

extern "C" size_t sp_mse_acc_workspace_bytes(int B, int K) {
    if (B <= 0 || K <= 0 || (long long)B * K > 0x7fffffffLL) return 0;
    return acc_keys_offset() + 32 * (size_t)B * K;
}

extern "C" int sp_mse_acc_fwd_bwd(const void* pred, int pred_dtype, const float* target, const float* mask, void* grad,
                                  float* loss, float* acc, float* pred_xy, float* label_xy, void* workspace,
                                  size_t workspace_bytes, int B, int K, int H, int W, float grad_scale,
                                  const float* grad_scale_dev, float distance_thresh, float norm_frac, int flags, void* stream) {
    SP_RETURN_IF(pred_dtype != SP_DTYPE_F32 && pred_dtype != SP_DTYPE_F16 && pred_dtype != SP_DTYPE_BF16, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!pred || !target || !mask || !loss || !acc || !workspace, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((pred_xy == nullptr) != (label_xy == nullptr), SP_ERR_BAD_ARGUMENT);     // both NULL: kept in the workspace
    SP_RETURN_IF(B <= 0 || K <= 0 || H <= 0 || W <= 0 || !(norm_frac > 0.f), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((long long)B * K > 0x7fffffffLL || (long long)H * W > 0x7fffffffLL || K > 4096, SP_ERR_UNSUPPORTED);
    SP_RETURN_IF(workspace_bytes < sp_mse_acc_workspace_bytes(B, K), SP_ERR_WORKSPACE);
    SP_RETURN_IF(!sp_aligned16(workspace) || (pred_xy && (!sp_aligned16(pred_xy) || !sp_aligned16(label_xy))), SP_ERR_BAD_ALIGNMENT);
    unsigned char* wsb = static_cast<unsigned char*>(workspace);
    if (!pred_xy) {
        pred_xy = reinterpret_cast<float*>(wsb + acc_keys_offset() + 16 * (size_t)B * K);
        label_xy = pred_xy + 2 * (size_t)B * K;
    }
    AccOut A;
    A.keys = reinterpret_cast<unsigned long long*>(wsb + acc_keys_offset());
    A.pred_xy = reinterpret_cast<float2*>(pred_xy);
    A.label_xy = reinterpret_cast<float2*>(label_xy);
    A.acc = acc;
    A.B = B; A.K = K; A.W = W;
    A.norm_x = (float)W / norm_frac;           // norm = tensor([W, H], float32) / norm_frac, as sp_heatmap_acc_f32
    A.norm_y = (float)H / norm_frac;
    A.thresh = distance_thresh;
    return mse_launch(pred, pred_dtype, target, mask, grad, loss, static_cast<MseWorkspace*>(workspace), B, K, H * W, grad_scale,
                      grad_scale_dev, flags, static_cast<cudaStream_t>(stream), A);
}

extern "C" int sp_scale_inplace_f32(float* data, long long n, const float* scale_dev, void* stream) {
    SP_RETURN_IF(!data || !scale_dev || n < 0, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!sp_aligned16(data), SP_ERR_BAD_ALIGNMENT);
    if (n == 0) return 0;
    long long blocks = ((n >> 2) + 255) / 256;
    const long long cap = (long long)sp_sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    SP_CUDA(sp_launch(scale_inplace_kernel, dim3((int)blocks), dim3(256), 0, static_cast<cudaStream_t>(stream), data, n, scale_dev));
    return 0;
}
