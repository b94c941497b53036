// Shared device helpers for the sm_100a heatmap kernels: launch checks, warp reductions and
// the PTX wrappers for mbarrier + cp.async.bulk (the 1-D TMA bulk copy, SASS: UBLKCP).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdlib.h>
#include "../../include/simple_pose_b200.h"

#define SP_WARP 32
#define SP_FULL 0xffffffffu

#define SP_RETURN_IF(cond, code) do { if (cond) return (code); } while (0)
#define SP_CUDA(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) return (int)e__; } while (0)

static inline bool sp_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static inline int sp_sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// ---- tuning knobs ------------------------------------------------------------------------------
// Read from the environment ONCE per process (first library call) into this table; a launch never
// calls getenv. sp_reload_tuning() re-reads it (tests and scratch/ubench.py sweep a knob by setting
// the variable and reloading). SP_UNSET = variable absent -> the launch code's own default.
#define SP_UNSET (-2147483647 - 1)
struct SpTuning {
    int no_pdl;
    int encode_warps, encode_parts;
    int loss_force_ldg, loss_chunk_quads, loss_ring, loss_warps;
    int train_force_ldg, train_chunk_quads, train_no_tile, train_static_pct, train_warps, train_ring;
    int decode_force_generic, decode_warps, decode_stages, decode_grid_wide, decode_runtime_ksize, decode_static_pct;
    int step_warps, step_static_pct;
    int nms_serial;
};
const SpTuning& sp_tuning();                                     // sp_abi.cu
static inline int sp_knob(int value, int fallback) { return value == SP_UNSET ? fallback : value; }

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device, size high-water mark)
// instead of a driver call on every launch (sp_abi.cu).
cudaError_t sp_ensure_dyn_smem(const void* func, size_t bytes);

// Launch status of the triple-chevron launches: peek (do not clear errors that belong to other
// users of the context, e.g. PyTorch kernels on the same device).
static inline int sp_launch_status() { return (int)cudaPeekAtLastError(); }

// Every kernel of the library is launched with programmatic dependent launch (PDL) allowed: its
// CTAs may be scheduled as soon as CTAs of the previous kernel on the stream exit, which hides the
// launch latency and the prologue (mbarrier init, index setup) behind the predecessor's tail. The
// contract inside the kernels: sp::grid_dep_wait() before the first global-memory access (it returns
// once the predecessor has completed and its writes are visible). No kernel triggers its
// dependents early (griddepcontrol.launch_dependents): the implicit trigger at CTA exit is what
// is wanted here. An early trigger was measured to cost 6-17 us per transition whenever two
// DIFFERENT kernels alternate on a stream (encode+loss+decode step: 1535 us with it, 1455 us
// without; scratch/seq_step.py), and to gain < 1 % for back-to-back launches of one kernel.
// SP_NO_PDL=1 in the environment restores plain stream-ordered launches.
template <typename... KArgs, typename... Args>
static inline cudaError_t sp_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                    Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = sp_tuning().no_pdl == 1 ? 0 : 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Same, raising the kernel's dynamic shared-memory limit first when it needs more than 48 KB.
template <typename... KArgs, typename... Args>
static inline cudaError_t sp_launch_smem(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                         Args... args) {
    if (smem > 48 * 1024) {
        const cudaError_t e = sp_ensure_dyn_smem(reinterpret_cast<const void*>(kernel), smem);
        if (e != cudaSuccess) return e;
    }
    return sp_launch(kernel, grid, block, smem, st, args...);
}

// Plain stream-ordered launch (kernels that do not call griddepcontrol.wait).
template <typename... KArgs, typename... Args>
static inline cudaError_t sp_launch_plain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                          Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = nullptr;
    cfg.numAttrs = 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

namespace sp {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- programmatic dependent launch ----------------------------------------------------------
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- mbarrier (shared::cta) ---------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// generic-proxy accesses to shared memory are ordered before later async-proxy (TMA) accesses
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- 1-D bulk copy global -> shared, completion counted on an mbarrier ----------------------
// bytes % 16 == 0, both addresses 16-byte aligned.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---- NaN-propagating max (max.NaN.f32) ------------------------------------------------------
__device__ __forceinline__ float fmax_nan(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}

// ---- warp reductions --------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(SP_FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(SP_FULL, v, o);
    return v;
}

// torch.max ordering on (value, index): larger value wins, NaN beats every number, equal
// values (and NaN vs NaN) are decided by the smaller index.
__device__ __forceinline__ bool better(float v, int i, float bv, int bi) {
    const bool vn = (v != v), bn = (bv != bv);
    if (vn != bn) return vn;
    if (vn) return i < bi;
    return (v > bv) || (v == bv && i < bi);
}

// ---- global counter with release (this thread's earlier writes) and acquire (later reads) semantics, device scope
__device__ __forceinline__ unsigned int atomic_add_acq_rel(unsigned int* p, unsigned int v) {
    unsigned int old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
    return old;
}

// Person score of kps_to_dict_ (metrics/pose_metrics.py:176): mean(conf) + max(conf) over the K joint peaks, fed in
// joint order. The mean is accumulated in float64 and rounded once (torch's float32 reduction order differs between
// its CPU and CUDA kernels; this is within 1 ulp of either); a NaN peak makes the score NaN.
struct PersonScore {
    double sum;
    float mx;
    bool nan;
    static __device__ __forceinline__ PersonScore start() {
        PersonScore s;
        s.sum = 0.0;
        s.mx = -CUDART_INF_F;
        s.nan = false;
        return s;
    }
    __device__ __forceinline__ void add(float v) {
        sum += (double)v;
        nan |= (v != v);
        mx = fmaxf(mx, v);
    }
    __device__ __forceinline__ float value(int K) const {
        const float mean = (float)(sum / (double)K);
        return nan ? CUDART_NAN_F : __fadd_rn(mean, mx);
    }
};

}  // namespace sp
