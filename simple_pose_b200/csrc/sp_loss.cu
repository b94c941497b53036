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
// Fallback (mse_fwd_bwd_kernel): any shape / alignment, and the SKIP_MASKED variant.
//
// The sum of squares is accumulated per thread in float32 over a few elements, then in float64;
// block partials go to the caller's workspace and the last block to finish adds them in a fixed
// order (deterministic, no floating-point atomics) and writes the scalar loss.
//
// Arithmetic follows ATen so that grad is bit-identical for finite inputs:
//   d = fl(m*p) - fl(m*t); grad = ((fl(2/N) * d) * 0.5) * m   (mse_loss_backward, then mul backward)
#include "sp_common.cuh"
#include "sp_reduce.cuh"
#include "sp_lowp.cuh"

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

__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ float sq_err_and_grad(float p, float t, float m, float norm, float half_scale, float& g) {
    const float d = __fsub_rn(__fmul_rn(m, p), __fmul_rn(m, t));
    g = __fmul_rn(__fmul_rn(__fmul_rn(norm, d), half_scale), m);
    return d;
}

template <bool VEC4, bool WRITE_GRAD>
__global__ void __launch_bounds__(kThreads)
mse_fwd_bwd_kernel(const float* __restrict__ pred, const float* __restrict__ target,
                   const float* __restrict__ mask, float* __restrict__ grad, float* __restrict__ loss,
                   MseWorkspace* __restrict__ ws, int nmaps, int hw, float norm, float half_scale,
                   double inv_count, int skip_masked) {
    double block_sum = 0.0;
    sp::grid_dep_wait();

    for (int m = blockIdx.x; m < nmaps; m += gridDim.x) {
        const float mk = __ldg(mask + m);
        const size_t base = (size_t)m * hw;
        float acc = 0.f;
        if (skip_masked && mk == 0.f) {
            if (WRITE_GRAD) {
                if (VEC4) {
                    float4* g4 = reinterpret_cast<float4*>(grad + base);
                    for (int q = threadIdx.x; q < (hw >> 2); q += kThreads) g4[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                } else {
                    for (int i = threadIdx.x; i < hw; i += kThreads) grad[base + i] = 0.f;
                }
            }
            continue;
        }
        if (VEC4) {
            const float4* p4 = reinterpret_cast<const float4*>(pred + base);
            const float4* t4 = reinterpret_cast<const float4*>(target + base);
            float4* g4 = reinterpret_cast<float4*>(grad + base);
            const int nq = hw >> 2;
#pragma unroll 4
            for (int q = threadIdx.x; q < nq; q += kThreads) {
                const float4 p = ldg_stream(p4 + q);
                const float4 t = ldg_stream(t4 + q);
                float4 g;
                float d;
                d = sq_err_and_grad(p.x, t.x, mk, norm, half_scale, g.x); acc = fmaf(d, d, acc);
                d = sq_err_and_grad(p.y, t.y, mk, norm, half_scale, g.y); acc = fmaf(d, d, acc);
                d = sq_err_and_grad(p.z, t.z, mk, norm, half_scale, g.z); acc = fmaf(d, d, acc);
                d = sq_err_and_grad(p.w, t.w, mk, norm, half_scale, g.w); acc = fmaf(d, d, acc);
                if (WRITE_GRAD) g4[q] = g;
            }
        } else {
            for (int i = threadIdx.x; i < hw; i += kThreads) {
                float g;
                const float d = sq_err_and_grad(pred[base + i], target[base + i], mk, norm, half_scale, g);
                acc = fmaf(d, d, acc);
                if (WRITE_GRAD) grad[base + i] = g;
            }
        }
        block_sum += (double)acc;
    }

    finish_loss<kThreads>(block_sum, ws, loss, inv_count);
}

// Mixed-precision variant (torch.cuda.amp, processors/dp_pose_hrnet_solver.py:111-120): `pred` arrives in the
// autocast dtype PT (float16 / bfloat16; float32 also instantiated) and the gradient leaves in PT. The
// arithmetic is what autocast runs: `pred.mul(mask)` promotes to float32, mse_loss is on autocast's float32
// list, the backward of the promoted product casts d loss / d pred to PT once, AFTER the upstream gradient
// (GradScaler's scale, read here from device memory so that no host sync is needed) has been applied in
// float32 -- which is the whole point of loss scaling for float16. Eight elements per thread per step:
// one 16-byte load of pred (8 x PT; 2 x float4 for float32), two of target, one 16-byte grad store.
// loss == nullptr: backward only (no reduction); grad == nullptr: forward only.
template <typename PT, bool VEC8>
__global__ void __launch_bounds__(kThreads)
mse_mixed_kernel(const PT* __restrict__ pred, const float* __restrict__ target, const float* __restrict__ mask,
                 PT* __restrict__ grad, float* __restrict__ loss, MseWorkspace* __restrict__ ws, int nmaps, int hw,
                 float norm, float half_scale_host, const float* __restrict__ scale_dev, double inv_count, int skip_masked) {
    double block_sum = 0.0;
    sp::grid_dep_wait();
    const float half_scale = scale_dev ? __fmul_rn(half_scale_host, __ldg(scale_dev)) : half_scale_host;
    const bool write_grad = grad != nullptr;

    for (int m = blockIdx.x; m < nmaps; m += gridDim.x) {
        const float mk = __ldg(mask + m);
        const size_t base = (size_t)m * hw;
        float acc = 0.f;
        if (skip_masked && mk == 0.f) {
            if (write_grad)
                for (int i = threadIdx.x; i < hw; i += kThreads) grad[base + i] = sp_lowp::from_float<PT>(0.f);
            continue;
        }
        if (VEC8) {
            const int n8 = hw >> 3;
#pragma unroll 2
            for (int o = threadIdx.x; o < n8; o += kThreads) {
                float p[8], g[8];
                sp_lowp::load8(pred + base + 8 * (size_t)o, p);
                const float4 t0 = ldg_stream(reinterpret_cast<const float4*>(target + base) + 2 * o);
                const float4 t1 = ldg_stream(reinterpret_cast<const float4*>(target + base) + 2 * o + 1);
                const float t[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const float d = sq_err_and_grad(p[e], t[e], mk, norm, half_scale, g[e]);
                    acc = fmaf(d, d, acc);
                }
                if (write_grad) sp_lowp::store8(grad + base + 8 * (size_t)o, g);
            }
        } else {
            for (int i = threadIdx.x; i < hw; i += kThreads) {
                float g;
                const float d = sq_err_and_grad(sp_lowp::to_float(pred[base + i]), target[base + i], mk, norm, half_scale, g);
                acc = fmaf(d, d, acc);
                if (write_grad) grad[base + i] = sp_lowp::from_float<PT>(g);
            }
        }
        block_sum += (double)acc;
    }
    if (loss != nullptr) finish_loss<kThreads>(block_sum, ws, loss, inv_count);
}

// dynamic smem: [mbarriers 1024 B][per warp: ring x (pred chunk | target chunk)]
constexpr int kRingBarBytes = 1024;

// A variant that sent the gradient out through the TMA too (written into the drained slot, cp.async.bulk shared -> global)
// was within 1-2 % either way warm and 12 % slower from a cold cache, so the gradient stays on register stores (DESIGN.md, section 4).
template <bool WRITE_GRAD>
__global__ void __launch_bounds__(1024, 1)
mse_ring_kernel(const float* __restrict__ pred, const float* __restrict__ target, const float* __restrict__ mask,
                float* __restrict__ grad, float* __restrict__ loss, MseWorkspace* __restrict__ ws,
                long long nchunks, int chunk_quads, int chunks_per_map, int nwarps, int ring,
                float norm, float half_scale, double inv_count) {
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
        }
        sum_sq += (double)acc;
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
    finish_loss<1024>(sum_sq, ws, loss, inv_count);
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

extern "C" int sp_mse_fwd_bwd_f32(const float* pred, const float* target, const float* mask,
                                  float* grad, float* loss, void* workspace, size_t workspace_bytes,
                                  int B, int K, int HW, float grad_scale, int flags, void* stream) {
    SP_RETURN_IF(!pred || !target || !mask || !loss || !workspace, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(B <= 0 || K <= 0 || HW <= 0, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((long long)B * K > 0x7fffffffLL, SP_ERR_UNSUPPORTED);
    SP_RETURN_IF(workspace_bytes < sizeof(MseWorkspace), SP_ERR_WORKSPACE);
    SP_RETURN_IF(!sp_aligned16(workspace), SP_ERR_BAD_ALIGNMENT);
    const int nmaps = B * K;
    const double count = (double)B * (double)K * (double)HW;
    const float norm = (float)(2.0 / count);       // ATen: norm = 2 / numel, applied in float32
    const float half_scale = 0.5f * grad_scale;    // the 0.5 of the loss expression times upstream grad
    const bool vec4 = (HW % 4 == 0) && sp_aligned16(pred) && sp_aligned16(target) && (!grad || sp_aligned16(grad));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MseWorkspace* ws = static_cast<MseWorkspace*>(workspace);
    const int skip = (flags & SP_MSE_SKIP_MASKED) ? 1 : 0;

    // ring kernel: needs 16-byte rows and a chunk size (in quads) that divides the map
    const SpTuning& tune = sp_tuning();
    if (vec4 && !skip && sp_knob(tune.loss_force_ldg, 0) == 0) {
        const int nq = HW >> 2;
        int want = sp_knob(tune.loss_chunk_quads, 192);           // 3 KB per stream
        if (want < 8) want = 8;
        if (want > 2048) want = 2048;
        int chunk_quads = 0;
        for (int d = want < nq ? want : nq; d >= 8; --d)
            if (nq % d == 0) { chunk_quads = d; break; }
        if (chunk_quads * 2 >= (want < nq ? want : nq)) {            // else: awkward map size, use the fallback
            int ring = sp_knob(tune.loss_ring, 3);
            if (ring < 1) ring = 1;
            if (ring > 8) ring = 8;
            int nwarps = sp_knob(tune.loss_warps, 4);   // 4 warps x 3 slots x 6 KB = 72 KB in flight per SM (sweep: profiles/)
            if (nwarps < 1) nwarps = 1;
            if (nwarps > 32) nwarps = 32;
            const size_t slot_bytes = (size_t)chunk_quads * 32;      // pred chunk + target chunk
            while (nwarps > 1 && (kRingBarBytes + (size_t)nwarps * ring * slot_bytes > 226 * 1024 || nwarps * ring * 8 > kRingBarBytes)) --nwarps;
            const size_t smem = kRingBarBytes + (size_t)nwarps * ring * slot_bytes;
            if (smem <= 226 * 1024 && nwarps * ring * 8 <= kRingBarBytes) {    // 1 KB spare for static shared memory
                const long long nchunks = (long long)nmaps * (nq / chunk_quads);
                int grid = sp_sm_count();
                if ((long long)grid * nwarps > nchunks) grid = (int)((nchunks + nwarps - 1) / nwarps);
                if (grad) {
                    SP_CUDA(sp_launch_smem(mse_ring_kernel<true>, dim3(grid), dim3(nwarps * 32), smem, st, pred, target, mask, grad, loss, ws,
                                      nchunks, chunk_quads, nq / chunk_quads, nwarps, ring, norm, half_scale, 1.0 / count));
                } else {
                    SP_CUDA(sp_launch_smem(mse_ring_kernel<false>, dim3(grid), dim3(nwarps * 32), smem, st, pred, target, mask, grad, loss, ws,
                                      nchunks, chunk_quads, nq / chunk_quads, nwarps, ring, norm, half_scale, 1.0 / count));
                }
                return 0;
            }
        }
    }

    int grid = sp_sm_count() * 8;
    if (grid > nmaps) grid = nmaps;
    if (grid > kMaxPartials) grid = kMaxPartials;
#define SP_LAUNCH_MSE(V, G) \
    SP_CUDA(sp_launch(mse_fwd_bwd_kernel<V, G>, dim3(grid), dim3(kThreads), 0, st, pred, target, mask, grad, loss, ws, nmaps, HW, norm, half_scale, 1.0 / count, skip))
    if (vec4) { if (grad) SP_LAUNCH_MSE(true, true); else SP_LAUNCH_MSE(true, false); }
    else      { if (grad) SP_LAUNCH_MSE(false, true); else SP_LAUNCH_MSE(false, false); }
#undef SP_LAUNCH_MSE
    return 0;
}

template <typename PT>
static int launch_mixed(const void* pred, const float* target, const float* mask, void* grad, float* loss, MseWorkspace* ws,
                        int nmaps, int HW, float norm, float half_scale, const float* scale_dev, double inv_count, int skip,
                        cudaStream_t st) {
    const bool vec8 = (HW % 8 == 0) && sp_aligned16(pred) && sp_aligned16(target) && (!grad || sp_aligned16(grad));
    int grid = sp_sm_count() * 8;
    if (grid > nmaps) grid = nmaps;
    if (grid > kMaxPartials) grid = kMaxPartials;
    const PT* p = static_cast<const PT*>(pred);
    PT* g = static_cast<PT*>(grad);
    if (vec8) SP_CUDA(sp_launch(mse_mixed_kernel<PT, true>, dim3(grid), dim3(kThreads), 0, st, p, target, mask, g, loss, ws, nmaps, HW, norm, half_scale, scale_dev, inv_count, skip));
    else      SP_CUDA(sp_launch(mse_mixed_kernel<PT, false>, dim3(grid), dim3(kThreads), 0, st, p, target, mask, g, loss, ws, nmaps, HW, norm, half_scale, scale_dev, inv_count, skip));
    return 0;
}

extern "C" int sp_mse_fwd_bwd(const void* pred, int pred_dtype, const float* target, const float* mask,
                              void* grad, float* loss, void* workspace, size_t workspace_bytes,
                              int B, int K, int HW, float grad_scale, const float* grad_scale_dev, int flags, void* stream) {
    SP_RETURN_IF(pred_dtype != SP_DTYPE_F32 && pred_dtype != SP_DTYPE_F16 && pred_dtype != SP_DTYPE_BF16, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!loss && !grad, SP_ERR_BAD_ARGUMENT);
    if (pred_dtype == SP_DTYPE_F32 && loss && !grad_scale_dev)        // the float32 fast path (TMA ring kernel)
        return sp_mse_fwd_bwd_f32(static_cast<const float*>(pred), target, mask, static_cast<float*>(grad), loss, workspace,
                                  workspace_bytes, B, K, HW, grad_scale, flags, stream);
    SP_RETURN_IF(!pred || !target || !mask, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(B <= 0 || K <= 0 || HW <= 0, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((long long)B * K > 0x7fffffffLL, SP_ERR_UNSUPPORTED);
    if (loss) {
        SP_RETURN_IF(!workspace, SP_ERR_BAD_ARGUMENT);
        SP_RETURN_IF(workspace_bytes < sizeof(MseWorkspace), SP_ERR_WORKSPACE);
        SP_RETURN_IF(!sp_aligned16(workspace), SP_ERR_BAD_ALIGNMENT);
    }
    const double count = (double)B * (double)K * (double)HW;
    const float norm = (float)(2.0 / count);
    const float half_scale = 0.5f * grad_scale;
    const int skip = (flags & SP_MSE_SKIP_MASKED) ? 1 : 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MseWorkspace* ws = static_cast<MseWorkspace*>(workspace);
    if (pred_dtype == SP_DTYPE_F16)
        return launch_mixed<__half>(pred, target, mask, grad, loss, ws, B * K, HW, norm, half_scale, grad_scale_dev, 1.0 / count, skip, st);
    if (pred_dtype == SP_DTYPE_BF16)
        return launch_mixed<__nv_bfloat16>(pred, target, mask, grad, loss, ws, B * K, HW, norm, half_scale, grad_scale_dev, 1.0 / count, skip, st);
    return launch_mixed<float>(pred, target, mask, grad, loss, ws, B * K, HW, norm, half_scale, grad_scale_dev, 1.0 / count, skip, st);
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
