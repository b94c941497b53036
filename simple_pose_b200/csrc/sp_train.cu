// SURVEY section 8f ranks 1+2: the training-step half of the path as ONE pass.
//
//   targets, mask = get_heat_map(joints)                      commons/transforms.py:167-191
//   loss = 0.5 * MSELoss(pred * mask, target * mask); backward   processors/dp_pose_hrnet_solver.py:106-107
//   acc  = HeatMapAcc()(pred * mask, target * mask)              metrics/pose_metrics.py:212-245, solver :123-124
//
// The targets are never materialised: each warp owns one (person, joint) map, evaluates the
// separable float64 Gaussian factors exactly like the stand-alone encoder, and while the predicted
// map streams by (one 16-byte load per lane per step) forms target, masked difference, squared
// error, gradient and -- for HeatMapAcc -- the running argmax of both masked maps. HBM traffic per
// person drops from 209 168 (encode) + 626 756 (loss) + 2 x 208 896 (two argmax passes) bytes to
// read pred + write grad = 417 860 bytes. Per-element arithmetic is the same as in the separate
// kernels, so grad/targets/weights are bit-identical to sp_encode_f32 + sp_mse_fwd_bwd_f32 and the
// loss differs only by the float64 summation order.
#include "sp_common.cuh"
#include "sp_gauss.cuh"
#include "sp_reduce.cuh"
#include "sp_lowp.cuh"
#include "sp_train_dev.cuh"
#include <math_constants.h>
#include <stdlib.h>

#ifdef SP_TRAIN_TRACE
// scratch instrumentation (never compiled into the product library): per-warp timestamps of the
// period-tiled kernel, 8 x int64 per warp: [globaltimer at entry, after griddepcontrol.wait, first
// chunk landed, last map done, after the loss reduction, maps processed, clock64 span of the map loop, 0]
__device__ long long* g_trace_ptr = nullptr;
extern "C" int sp_debug_set_trace(void* p) {
    return (int)cudaMemcpyToSymbol(g_trace_ptr, &p, sizeof(p));
}
__device__ __forceinline__ long long gtime() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#endif

namespace {

using namespace sp_gauss;
using namespace sp_reduce;
using namespace sp_trn;

// Variant A: predicted maps read straight from global memory (any map size).
// PT = storage type of pred and grad (float32, or float16 / bfloat16 under torch.cuda.amp: the arithmetic stays
// float32 as autocast runs it, the gradient is cast to PT once, after the upstream scale has been applied).
template <bool WRITE_GRAD, bool WRITE_TARGETS, bool ACC, typename PT = float>
__global__ void __launch_bounds__(kThreads)
encode_mse_kernel(const MapIo io, float* __restrict__ loss, MseWorkspace* __restrict__ ws, double inv_count) {
    extern __shared__ __align__(16) double factors[];   // per warp: ex[Wpad] then ey[H]
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int wpad = (io.W + 1) & ~1;
    double* ex = factors + (size_t)warp * (wpad + ((io.H + 1) & ~1));   // even stride: 16-byte aligned ex for every warp (odd H)
    double* ey = ex + wpad;
    const int hw = io.H * io.W;
    const int total_warps = gridDim.x * kWarps;
    double sum_sq = 0.0;
    sp::grid_dep_wait();
    const float half_scale = io.scale_dev ? __fmul_rn(io.half_scale, __ldg(io.scale_dev)) : io.half_scale;
    Joint3 jn = load_joint(io, blockIdx.x * kWarps + warp);
    for (int m = blockIdx.x * kWarps + warp; m < io.nmaps; m += total_warps) {
        const Joint3 jc = jn;
        jn = load_joint(io, m + total_warps);               // next map's joint: latency hidden behind this map
        const JointVerdict jv = prepare_map(io, m, jc, ex, ey, lane);
        MapState st;
        begin_map(io, jv, st, lane, ACC);
        run_quads<WRITE_GRAD, WRITE_TARGETS, ACC, false, PT>(
            io, m, reinterpret_cast<const float4*>(reinterpret_cast<const PT*>(io.pred) + (size_t)m * hw), 0, hw >> 2, jv, ex, ey,
            st, lane, half_scale);
        if (ACC) end_map_acc<PT>(io, m, jv, ex, ey, st, lane);
        sum_sq += (double)st.acc;
    }
    if (loss != nullptr) finish_loss<512>(sum_sq, ws, loss, inv_count);     // every lane carries the quads it visited
}

// Variant B (default): persistent, one CTA per SM, up to 32 warps. Every warp streams its predicted
// maps through a private ring of small shared-memory slots (1-D TMA bulk copies of `chunk_quads`
// quads each, mbarrier complete_tx). The map is consumed strictly in order, so a slot is re-armed
// with the chunk `ring` positions ahead -- possibly of the warp's NEXT map -- the moment it has been
// read: the copy engine runs a full ring ahead of the arithmetic, nothing stalls on individual
// global loads, and a 6 KB ring per warp leaves room for 32 resident warps to hide the float64
// and shared-memory latencies.
// Work distribution: CTA c owns the contiguous map range [c*nmaps/grid, (c+1)*nmaps/grid); its warps
// claim maps from a shared-memory counter (lane 0, one map ahead of the copies it is issuing) and
// pass the claimed indices to the consuming lanes through a small per-warp FIFO.
// dynamic smem: [mbarriers 1024 B][claim FIFOs + work counter 2048 B][factors per warp][ring slots per warp]

template <bool WRITE_GRAD, bool WRITE_TARGETS, bool ACC>
__global__ void __launch_bounds__(512, 1)
encode_mse_ring_kernel(const MapIo io, float* __restrict__ loss, MseWorkspace* __restrict__ ws, double inv_count,
                       int nwarps, int ring, int chunk_quads) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int hw = io.H * io.W;
    const int nq = hw >> 2;
    const int chunks_per_map = nq / chunk_quads;                 // host guarantees divisibility
    const uint32_t chunk_bytes = (uint32_t)chunk_quads * 16u;
    const int wpad = (io.W + 1) & ~1;
    const size_t fac_bytes = (size_t)(wpad + ((io.H + 1) & ~1)) * sizeof(double);   // multiple of 16 (odd H too)
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw) + warp * ring;
    volatile int* fifo = reinterpret_cast<int*>(smem_raw + 1024) + warp * kFifo;
    int& next_map = *reinterpret_cast<int*>(smem_raw + 1024 + 2048);
    double* ex = reinterpret_cast<double*>(smem_raw + kRingHeader + warp * fac_bytes);
    double* ey = ex + wpad;
    unsigned char* slots = smem_raw + kRingHeader + (size_t)nwarps * fac_bytes + (size_t)warp * ring * chunk_bytes;
    const int range_lo = (int)((long long)blockIdx.x * io.nmaps / gridDim.x);
    const int range_hi = (int)((long long)(blockIdx.x + 1) * io.nmaps / gridDim.x);
    if (threadIdx.x == 0) next_map = range_lo;
    if (lane == 0) {
        for (int r = 0; r < ring; ++r) sp::mbar_init(bars + r, 1);
        sp::mbar_fence_init();
    }
    __syncthreads();
    sp::grid_dep_wait();            // the prologue above overlapped the previous kernel's tail

    // producer (lane 0 only): copies chunk pc of map pm into slot ps; pnext = the map claimed after pm
    int pm = -1, pnext = -1, pc = 0, ps = 0, tail = 0;
    auto claim = [&]() {
        const int m = atomicAdd(&next_map, 1);
        const int got = (m < range_hi) ? m : -1;
        fifo[tail & (kFifo - 1)] = got;
        ++tail;
        return got;
    };
    auto issue_next = [&]() {
        if (pm < 0) return;
        sp::mbar_expect_tx(bars + ps, chunk_bytes);
        sp::bulk_g2s(slots + (size_t)ps * chunk_bytes, io.pred + (size_t)pm * hw + (size_t)pc * chunk_quads * 4,
                     chunk_bytes, bars + ps);
        if (++pc == chunks_per_map) {
            pc = 0;
            pm = pnext;
            pnext = (pm >= 0) ? claim() : -1;
        }
        if (++ps == ring) ps = 0;
    };
    if (lane == 0) {
        pm = claim();
        pnext = (pm >= 0) ? claim() : -1;
        for (int r = 0; r < ring; ++r) issue_next();
    }
    __syncwarp();

    double sum_sq = 0.0;
    int cs = 0;                 // consumer slot
    uint32_t parity = 0;
    int head = 0;
    int m = fifo[0];
    Joint3 jn = load_joint(io, m >= 0 ? m : io.nmaps);
    while (m >= 0) {
        const Joint3 jc = jn;
        // the producer claimed this map's successor before it issued this map's first chunk
        const int m_next = fifo[(head + 1) & (kFifo - 1)];
        jn = load_joint(io, m_next >= 0 ? m_next : io.nmaps);           // next map's joint, a whole map ahead
        const JointVerdict jv = prepare_map(io, m, jc, ex, ey, lane);   // overlaps the copies in flight
        MapState st;
        begin_map(io, jv, st, lane, ACC);
        for (int c = 0; c < chunks_per_map; ++c) {
            sp::mbar_wait(bars + cs, parity);
            const float4* chunk = reinterpret_cast<const float4*>(slots + (size_t)cs * chunk_bytes);
            run_quads<WRITE_GRAD, WRITE_TARGETS, ACC, true>(io, m, chunk, c * chunk_quads, (c + 1) * chunk_quads,
                                                            jv, ex, ey, st, lane, io.half_scale);
            __syncwarp();
            if (lane == 0) {
                sp::fence_proxy_async_smem();
                issue_next();                                           // refills the slot just drained
            }
            if (++cs == ring) { cs = 0; parity ^= 1u; }
        }
        if (ACC) end_map_acc(io, m, jv, ex, ey, st, lane);
        sum_sq += (double)st.acc;
        __syncwarp();
        ++head;
        m = m_next;
    }
    finish_loss<512>(sum_sq, ws, loss, inv_count);
}

// Variant C (default for W = 48 and W = 72 when grad is wanted and targets are not): the ring of
// variant B with the per-quad and per-chunk bookkeeping compiled away. With QPR quads per row, the
// (row, quad-in-row) pattern a lane sees repeats every PERIOD = QPR / gcd(32, QPR) warp steps and
// advances by ROWS = 32 / gcd(32, QPR) rows, so the chunk body is fully unrolled over PPC periods
// with per-lane constants: no index arithmetic, for PERIOD <= 3 the lane's x factors live in
// registers (one shared-memory load per quad left: the row factor), ring depth and chunk size are
// template parameters, shared memory is addressed with 32-bit offsets, the draw / unit-mask /
// tracking decisions are made once per map (three specialisations of the map body), and the running
// argmax keeps only (value, quad) -- the position inside the winning quad is recovered at the end
// of the NEXT map from a 16-byte re-read that has had a whole map to complete.
// Why it matters: with 16 warps per SM each warp issues about one instruction every 8 cycles, so
// the kernel's time is (instructions per quad) x latency until the copy engine becomes the limit.
// dynamic smem: same layout as variant B
template <int QPR, int PPC, int RING, bool ACC>
__global__ void __launch_bounds__(512, 1)
encode_mse_tile_kernel(const MapIo io, float* __restrict__ loss, MseWorkspace* __restrict__ ws, double inv_count, int nwarps,
                       int depth,   // == RING; making it compile-time reschedules the kernel, a change to measure on its own
                       int static_maps) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int CHUNK_BYTES = PPC * 32 * Tile<QPR>::PERIOD * 16;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
#ifdef SP_TRAIN_TRACE
    long long tr[8] = {gtime(), 0, 0, 0, 0, 0, 0, 0};
#endif
    const int hw = io.H * io.W;
    const int wpad = (io.W + 1) & ~1;
    const size_t fac_bytes = (size_t)(wpad + ((io.H + 1) & ~1)) * sizeof(double);   // multiple of 16 (odd H too)
    volatile int* fifo = reinterpret_cast<int*>(smem_raw + 1024) + warp * kFifo;
    double* ex = reinterpret_cast<double*>(smem_raw + kRingHeader + warp * fac_bytes);
    double* ey = ex + wpad;
    TileRing<RING, CHUNK_BYTES> rg;
    const uint32_t base = sp::smem_u32(smem_raw);
    rg.bar0 = base + (uint32_t)(warp * RING * 8);
    rg.slot0 = base + (uint32_t)(kRingHeader + (size_t)nwarps * fac_bytes + (size_t)warp * RING * CHUNK_BYTES);
    rg.cs = 0; rg.parity = 0; rg.ps = 0; rg.tail = 0; rg.left = 0; rg.pnext = -1; rg.src = nullptr;
    rg.inflight = 0; rg.depth = depth;
    rg.fifo = fifo; rg.next_work = &ws->next_work;
    rg.nmaps = io.nmaps;
    rg.static_stride = (int)gridDim.x * nwarps;
    rg.static_next = (int)blockIdx.x * nwarps + warp;
    rg.static_left = static_maps;
    rg.dyn_base = static_maps * rg.static_stride;
    rg.pred = reinterpret_cast<const char*>(io.pred);
    rg.map_bytes = (size_t)hw * 4;
    rg.chunks_per_map = hw * 4 / CHUNK_BYTES;
    if (lane == 0) {
        for (int r = 0; r < RING; ++r) sp::mbar_init(reinterpret_cast<uint64_t*>(smem_raw) + warp * RING + r, 1);
        sp::mbar_fence_init();
    }
    __syncthreads();
    sp::grid_dep_wait();            // the prologue above overlapped the previous kernel's tail
#ifdef SP_TRAIN_TRACE
    tr[1] = gtime();
#endif

    if (lane == 0) {
        rg.start(rg.claim());
        rg.top_up();
    }
    __syncwarp();
#ifdef SP_TRAIN_TRACE
    if (fifo[0] >= 0) { while (!mbar_try_wait_a(rg.bar0, 0)) { } }
    tr[2] = gtime();
    const long long c0 = clock64();
#endif

    double sum_sq = 0.0;
    PendingAxis pd;
    pd.m = -1; pd.quad = 0; pd.gmax = 0.f; pd.mk = 0.f; pd.v = make_float4(0.f, 0.f, 0.f, 0.f);
    int head = 0;
    int m = fifo[0];
    Joint3 jn = load_joint(io, m >= 0 ? m : io.nmaps);
    while (m >= 0) {
        const Joint3 jc = jn;
        const int m_next = fifo[(head + 1) & (kFifo - 1)];   // claimed before this map's first chunk was issued
        jn = load_joint(io, m_next >= 0 ? m_next : io.nmaps);
        const JointVerdict jv = prepare_map<QPR>(io, m, jc, ex, ey, lane);
        float acc;
        if (jv.draw && jv.weight == 1.0f && (!ACC || io.analytic_ok))
            acc = tile_map<QPR, PPC, ACC, 0>(io, m, jv, ex, ey, rg, pd, lane);
        else if (!jv.draw && jv.weight == 0.0f)
            acc = tile_map<QPR, PPC, ACC, 1>(io, m, jv, ex, ey, rg, pd, lane);
        else
            acc = tile_map<QPR, PPC, ACC, 2>(io, m, jv, ex, ey, rg, pd, lane);
        sum_sq += (double)acc;
        __syncwarp();
        ++head;
        m = m_next;
    }
    if (ACC) flush_pending(io, pd, lane);
#ifdef SP_TRAIN_TRACE
    tr[3] = gtime(); tr[5] = head; tr[6] = clock64() - c0;
    { unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); tr[7] = smid; }
#endif
    finish_loss<512>(sum_sq, ws, loss, inv_count);
#ifdef SP_TRAIN_TRACE
    tr[4] = gtime();
    if (lane == 0 && g_trace_ptr) {
        long long* t = g_trace_ptr + ((size_t)blockIdx.x * 16 + warp) * 8;
        for (int i = 0; i < 8; ++i) t[i] = tr[i];
    }
#endif
}

// HeatMapAcc epilogue (metrics/pose_metrics.py:227-245) on the [B,K] argmax coordinates.
__global__ void __launch_bounds__(256)
heatmap_acc_kernel(const float2* __restrict__ pred_xy, const float2* __restrict__ label_xy, float* __restrict__ acc,
                   int B, int K, float norm_x, float norm_y, float thresh) {
    extern __shared__ int counters[];        // hit[K], valid[K]
    sp::grid_dep_wait();
    int* hit = counters;
    int* valid = counters + K;
    for (int k = threadIdx.x; k < 2 * K; k += blockDim.x) counters[k] = 0;
    __syncthreads();
    const int n = B * K;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float2 l = label_xy[i];
        if (l.x > 1.f && l.y > 1.f) {
            const float2 p = pred_xy[i];
            const float dx = __fsub_rn(__fdiv_rn(p.x, norm_x), __fdiv_rn(l.x, norm_x));
            const float dy = __fsub_rn(__fdiv_rn(p.y, norm_y), __fdiv_rn(l.y, norm_y));
            // torch.norm accumulates float inputs in double on CPU (the pinned oracle); no (dx, dy)
            // pair of the supported map sizes lands on the threshold, so float vs double is moot
            const float dist = (float)sqrt((double)dx * (double)dx + (double)dy * (double)dy);
            const int k = i % K;
            atomicAdd(&valid[k], 1);
            if (dist < thresh) atomicAdd(&hit[k], 1);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float sum = 0.f;
        int used = 0;
        for (int k = 0; k < K; ++k) {
            if (valid[k] < 1) continue;
            sum = __fadd_rn(sum, __fdiv_rn((float)hit[k], (float)valid[k]));
            ++used;
        }
        acc[0] = used > 0 ? __fdiv_rn(sum, (float)used) : 0.f;
    }
}

}  // namespace

static int encode_mse_launch(const float* joints, const void* pred_raw, int pred_dtype, void* grad_raw, float* targets,
                             float* weights, float* loss, float* pred_xy, float* label_xy,
                             void* workspace, size_t workspace_bytes,
                             int B, int K, int H, int W, double sigma, float grad_scale, const float* scale_dev, void* stream) {
    const float* pred = static_cast<const float*>(pred_raw);      // reinterpreted per dtype inside the generic kernel
    float* grad = static_cast<float*>(grad_raw);
    const bool plain_f32 = (pred_dtype == SP_DTYPE_F32) && !scale_dev && loss;
    SP_RETURN_IF(pred_dtype != SP_DTYPE_F32 && pred_dtype != SP_DTYPE_F16 && pred_dtype != SP_DTYPE_BF16, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(!joints || !pred || (!loss && !grad) || !workspace, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(B <= 0 || K <= 0 || H <= 0 || W <= 0 || !(sigma > 0.0), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((pred_xy == nullptr) != (label_xy == nullptr), SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((long long)B * K > 0x7fffffffLL || (long long)H * W > (1 << 24), SP_ERR_UNSUPPORTED);
    SP_RETURN_IF(W % 4 != 0, SP_ERR_UNSUPPORTED);          // callers compose sp_encode_f32 + sp_mse_fwd_bwd_f32 instead
    SP_RETURN_IF(workspace_bytes < sizeof(MseWorkspace), SP_ERR_WORKSPACE);
    SP_RETURN_IF(!sp_aligned16(workspace) || !sp_aligned16(pred) || (grad && !sp_aligned16(grad)) ||
                 (targets && !sp_aligned16(targets)) || (pred_xy && (!sp_aligned16(pred_xy) || !sp_aligned16(label_xy))),
                 SP_ERR_BAD_ALIGNMENT);
    const int nmaps = B * K;
    const float reach = (float)(sigma * 3.0);
    const double denom = 2.0 * (sigma * sigma);
    const double count = (double)B * (double)K * (double)H * (double)W;
    const float norm = (float)(2.0 / count);
    const float half_scale = 0.5f * grad_scale;
    const int wpad = (W + 1) & ~1;
    const size_t fac_bytes = (size_t)(wpad + ((H + 1) & ~1)) * sizeof(double);          // multiple of 16 (odd H too)
    MapIo io;
    io.joints = joints; io.pred = pred; io.grad = grad; io.targets = targets; io.weights = weights;
    io.pred_xy = reinterpret_cast<float2*>(pred_xy); io.label_xy = reinterpret_cast<float2*>(label_xy);
    io.nmaps = nmaps; io.H = H; io.W = W; io.reach = reach; io.denom = denom; io.norm = norm; io.half_scale = half_scale;
    io.scale_dev = scale_dev;
    io.analytic_ok = (sigma >= 0.25 && sigma <= 64.0) ? 1 : 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MseWorkspace* ws = static_cast<MseWorkspace*>(workspace);
    const int sel = (grad ? 4 : 0) | (targets ? 2 : 0) | (pred_xy ? 1 : 0);

    // Ring variant: needs the map to split into equal chunks of a multiple of 32 quads (<= 4 KB)
    const int nq = (H * W) >> 2;
    const SpTuning& tune = sp_tuning();
    const bool force_ldg = sp_knob(tune.train_force_ldg, 0) == 1;
    int chunk_quads = 0;
    if ((H * W) % 4 == 0 && nq % 32 == 0) {
        int want = sp_knob(tune.train_chunk_quads, 192);  // 3 KB
        if (want < 32) want = 32;
        for (int d = want - want % 32; d >= 32; d -= 32)
            if (nq % d == 0) { chunk_quads = d; break; }
    }
    // Variant C: W = 48 / 72 (12 / 18 quads per row), whole periods per map, grad wanted, targets not
    const int qpr = W >> 2;
    if (plain_f32 && (qpr == 12 || qpr == 18) && grad && !targets && !force_ldg && sp_knob(tune.train_no_tile, 0) == 0) {
        const int period = (qpr == 12) ? Tile<12>::PERIOD : Tile<18>::PERIOD;
        const int rows = (qpr == 12) ? Tile<12>::ROWS : Tile<18>::ROWS;
        // the tuned layouts (PPC periods per chunk, RING slots per warp): (2, 1) at W = 48, (1, 2) at W = 72
        const int ppc = (qpr == 12) ? 2 : 1, ring = (qpr == 12) ? 1 : 2;
        const int periods = nq / (32 * period);
        if (H % rows == 0 && periods % ppc == 0) {
            const size_t chunk_bytes = (size_t)ppc * 32 * period * 16;
            const size_t budget = 226 * 1024 - kRingHeader;
            int nwarps = (int)(budget / (fac_bytes + ring * chunk_bytes));
            if (nwarps > 16) nwarps = 16;
            // 96x72 maps are 27 KB: with 16 warps a map takes ~20 us and the launch ends with a long,
            // thin tail; 8 warps (74 KB in flight per SM) halve it (512 persons: 88 -> 83 us) once there
            // are enough maps to keep the warps fed. Small launches keep 16 warps (more maps in flight).
            int want_warps = (qpr == 18 && nmaps >= 2 * 16 * sp_sm_count()) ? 8 : 16;
            want_warps = sp_knob(tune.train_warps, want_warps);
            if (want_warps < nwarps) nwarps = want_warps;
            if (nwarps >= 1) {
                const size_t smem = kRingHeader + (size_t)nwarps * (fac_bytes + ring * chunk_bytes);
                int grid = sp_sm_count();
                const int need = (nmaps + nwarps - 1) / nwarps;
                if (grid > need) grid = need;
                // maps per warp that are assigned up front (no atomic); the rest are dealt from the grid-wide
                // counter. All atomics hit one address (~3.5 ns each on B200), so the dynamic share is kept to
                // what the spread of SM speeds needs: half of a warp's expected maps, at least 2 fixed.
                int static_maps = (int)((long long)nmaps * sp_knob(tune.train_static_pct, 50) / 100 / ((long long)grid * nwarps));
                if (static_maps < 2) static_maps = 2;
#define SP_LAUNCH_TILE(Q, P, R)                                                                                              \
    do {                                                                                                                     \
        if (pred_xy) {                                                                                                       \
            SP_CUDA(sp_launch_smem(encode_mse_tile_kernel<Q, P, R, true>, dim3(grid), dim3(nwarps * 32), smem, st, io, loss, ws, 1.0 / count, nwarps, ring, static_maps)); \
        } else {                                                                                                             \
            SP_CUDA(sp_launch_smem(encode_mse_tile_kernel<Q, P, R, false>, dim3(grid), dim3(nwarps * 32), smem, st, io, loss, ws, 1.0 / count, nwarps, ring, static_maps)); \
        }                                                                                                                    \
    } while (0)
                if (qpr == 12) SP_LAUNCH_TILE(12, 2, 1);
                else           SP_LAUNCH_TILE(18, 1, 2);
#undef SP_LAUNCH_TILE
                return 0;
            }
        }
    }
    if (plain_f32 && chunk_quads > 0 && !force_ldg) {
        const size_t chunk_bytes = (size_t)chunk_quads * 16;
        const size_t budget = 226 * 1024 - kRingHeader;        // 1 KB spare for static shared memory
        int ring = sp_knob(tune.train_ring, 2);
        if (ring < 1) ring = 1;
        if (ring > 8) ring = 8;
        int nwarps = (int)(budget / (fac_bytes + ring * chunk_bytes));
        if (nwarps > 16) nwarps = 16;      // 16 x 2 x 3 KB = 96 KB in flight per SM; more warps = more HBM streams = slower
        { const int w = sp_knob(tune.train_warps, 16); if (w < nwarps) nwarps = w; }
        if (nwarps < 1) nwarps = 1;
        SP_RETURN_IF((size_t)nwarps * ring * 8 > 1024, SP_ERR_UNSUPPORTED);
        const size_t smem = kRingHeader + (size_t)nwarps * (fac_bytes + ring * chunk_bytes);
        int grid = sp_sm_count();
        const int need = (nmaps + nwarps - 1) / nwarps;
        if (grid > need) grid = need;
#define SP_LAUNCH_RING(G, T, A)                                                                                              \
    do {                                                                                                                     \
        SP_CUDA(sp_launch_smem(encode_mse_ring_kernel<G, T, A>, dim3(grid), dim3(nwarps * 32), smem, st, io, loss, ws, 1.0 / count, nwarps, ring, chunk_quads)); \
    } while (0)
        switch (sel) {
            case 0: SP_LAUNCH_RING(false, false, false); break;
            case 1: SP_LAUNCH_RING(false, false, true); break;
            case 2: SP_LAUNCH_RING(false, true, false); break;
            case 3: SP_LAUNCH_RING(false, true, true); break;
            case 4: SP_LAUNCH_RING(true, false, false); break;
            case 5: SP_LAUNCH_RING(true, false, true); break;
            case 6: SP_LAUNCH_RING(true, true, false); break;
            default: SP_LAUNCH_RING(true, true, true); break;
        }
#undef SP_LAUNCH_RING
        return 0;
    }

    const size_t smem = (size_t)kWarps * fac_bytes;
    SP_RETURN_IF(smem > 200 * 1024, SP_ERR_UNSUPPORTED);
    int grid = (nmaps + kWarps - 1) / kWarps;
    if (grid > kMaxPartials) grid = kMaxPartials;
#define SP_LAUNCH_TRAIN(G, T, A)                                                                                         \
    do {                                                                                                                 \
        if (pred_dtype == SP_DTYPE_F16)                                                                                  \
            SP_CUDA(sp_launch_smem(encode_mse_kernel<G, T, A, __half>, dim3(grid), dim3(kThreads), smem, st, io, loss, ws, 1.0 / count)); \
        else if (pred_dtype == SP_DTYPE_BF16)                                                                            \
            SP_CUDA(sp_launch_smem(encode_mse_kernel<G, T, A, __nv_bfloat16>, dim3(grid), dim3(kThreads), smem, st, io, loss, ws, 1.0 / count)); \
        else                                                                                                             \
            SP_CUDA(sp_launch_smem(encode_mse_kernel<G, T, A, float>, dim3(grid), dim3(kThreads), smem, st, io, loss, ws, 1.0 / count)); \
    } while (0)
    switch (sel) {
        case 0: SP_LAUNCH_TRAIN(false, false, false); break;
        case 1: SP_LAUNCH_TRAIN(false, false, true); break;
        case 2: SP_LAUNCH_TRAIN(false, true, false); break;
        case 3: SP_LAUNCH_TRAIN(false, true, true); break;
        case 4: SP_LAUNCH_TRAIN(true, false, false); break;
        case 5: SP_LAUNCH_TRAIN(true, false, true); break;
        case 6: SP_LAUNCH_TRAIN(true, true, false); break;
        default: SP_LAUNCH_TRAIN(true, true, true); break;
    }
#undef SP_LAUNCH_TRAIN
    return 0;
}

extern "C" int sp_encode_mse_fwd_bwd_f32(const float* joints, const float* pred, float* grad, float* targets,
                                         float* weights, float* loss, float* pred_xy, float* label_xy,
                                         void* workspace, size_t workspace_bytes,
                                         int B, int K, int H, int W, double sigma, float grad_scale, void* stream) {
    SP_RETURN_IF(!loss, SP_ERR_BAD_ARGUMENT);
    return encode_mse_launch(joints, pred, SP_DTYPE_F32, grad, targets, weights, loss, pred_xy, label_xy, workspace, workspace_bytes,
                             B, K, H, W, sigma, grad_scale, nullptr, stream);
}

extern "C" int sp_encode_mse_fwd_bwd(const float* joints, const void* pred, int pred_dtype, void* grad, float* targets,
                                     float* weights, float* loss, float* pred_xy, float* label_xy,
                                     void* workspace, size_t workspace_bytes,
                                     int B, int K, int H, int W, double sigma, float grad_scale, const float* grad_scale_dev,
                                     void* stream) {
    return encode_mse_launch(joints, pred, pred_dtype, grad, targets, weights, loss, pred_xy, label_xy, workspace, workspace_bytes,
                             B, K, H, W, sigma, grad_scale, grad_scale_dev, stream);
}

extern "C" int sp_heatmap_acc_f32(const float* pred_xy, const float* label_xy, float* acc,
                                  int B, int K, int H, int W, float distance_thresh, float norm_frac, void* stream) {
    SP_RETURN_IF(!pred_xy || !label_xy || !acc, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF(B <= 0 || K <= 0 || H <= 0 || W <= 0 || K > 4096, SP_ERR_BAD_ARGUMENT);
    SP_RETURN_IF((long long)B * K > 0x7fffffffLL, SP_ERR_UNSUPPORTED);
    SP_RETURN_IF(!sp_aligned16(pred_xy) || !sp_aligned16(label_xy), SP_ERR_BAD_ALIGNMENT);
    // norm = tensor([W, H], float32) / norm_frac
    const float nx = (float)W / norm_frac, ny = (float)H / norm_frac;
    SP_CUDA(sp_launch(heatmap_acc_kernel, dim3(1), dim3(256), (size_t)2 * K * sizeof(int), static_cast<cudaStream_t>(stream),
                      reinterpret_cast<const float2*>(pred_xy), reinterpret_cast<const float2*>(label_xy), acc, B, K, nx, ny,
                      distance_thresh));
    return 0;
}
