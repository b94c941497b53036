// Device-side building blocks of the fused encode + masked-MSE (+ HeatMapAcc) pass over a predicted map,
// shared by the training kernels (sp_train.cu) and the one-launch step kernel (sp_step.cu). The argmax rule and the
// HeatMapAcc epilogue are in sp_argmax.cuh. See sp_train.cu.
#pragma once
#include "sp_common.cuh"
#include "sp_gauss.cuh"
#include "sp_reduce.cuh"
#include "sp_lowp.cuh"
#include "sp_argmax.cuh"
#include <math_constants.h>

namespace sp_trn {

using namespace sp_gauss;
using namespace sp_reduce;
using namespace sp_arg;

constexpr int kWarps = 8;
constexpr int kThreads = kWarps * SP_WARP;

// quad q (4 consecutive elements) of a map stored as float32 / float16 / bfloat16
__device__ __forceinline__ float4 load_quad(const float* map, int q) { return sp_lowp::ldg_stream4(reinterpret_cast<const float4*>(map) + q); }
__device__ __forceinline__ float4 load_quad(const __half* map, int q) {
    const uint2 w = __ldg(reinterpret_cast<const uint2*>(map) + q);
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&w.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&w.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float4 load_quad(const __nv_bfloat16* map, int q) {
    const uint2 w = __ldg(reinterpret_cast<const uint2*>(map) + q);
    return make_float4(__uint_as_float(w.x << 16), __uint_as_float(w.x & 0xffff0000u), __uint_as_float(w.y << 16),
                       __uint_as_float(w.y & 0xffff0000u));
}
__device__ __forceinline__ void store_quad(float* map, int q, float4 v) { reinterpret_cast<float4*>(map)[q] = v; }
__device__ __forceinline__ void store_quad(__half* map, int q, float4 v) {
    const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    reinterpret_cast<uint2*>(map)[q] = make_uint2(*reinterpret_cast<const unsigned*>(&a), *reinterpret_cast<const unsigned*>(&b));
}
__device__ __forceinline__ void store_quad(__nv_bfloat16* map, int q, float4 v) {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    reinterpret_cast<uint2*>(map)[q] = make_uint2(*reinterpret_cast<const unsigned*>(&a), *reinterpret_cast<const unsigned*>(&b));
}

struct MapIo {                 // per-launch constants of the fused kernel
    const float* joints;
    const float* pred;
    float* grad;
    float* targets;
    float* weights;
    float2* pred_xy;
    float2* label_xy;
    int nmaps, H, W;
    float reach;
    double denom;
    float norm, half_scale;
    const float* scale_dev;   // optional device scalar multiplied into half_scale (upstream gradient); generic kernel only
    int analytic_ok;          // sigma in the range where the target argmax can be found analytically
};

// One (person, joint) map, one warp. `src` = the predicted map, in shared memory (SMEM_PRED, staged
// by TMA) or in global memory. Returns this lane's share of sum((m*p - m*t)^2).
// Per-map running state of one warp while the predicted map streams by (possibly in chunks).
struct MapState {
    float acc;                   // this lane's share of sum((m*p - m*t)^2)
    QuadBest bp, bt;             // running argmax of the masked predicted / target map
    int y, xq;                   // row and quad-in-row of this lane's next quad
    bool track, analytic_t, track_t;
};

__device__ __forceinline__ void begin_map(const MapIo& io, const JointVerdict& jv, MapState& st, int lane, bool acc_on) {
    const int qpr = io.W >> 2;
    st.acc = 0.f;
    st.bp.init();
    st.bt.init();
    st.y = lane / qpr;
    st.xq = lane - st.y * qpr;
    st.track = acc_on && (jv.weight != 0.f);
    // The target's argmax is found analytically (3x3 block around the rounded centre) when the
    // mask and sigma are in the range where float32 rounding cannot create far-away ties.
    st.analytic_t = st.track && jv.draw && io.analytic_ok && jv.weight >= 0.5f && jv.weight <= 4.f;
    st.track_t = st.track && jv.draw && !st.analytic_t;
}

// Quads q = q_begin + lane, +32, ... < q_end of map m; `chunk` points at quad q_begin of the
// predicted map (shared memory when SMEM_PRED, else global). q_begin is a multiple of 32.
// UNIT: the mask is exactly 1.0f (the common case), so m*p == p, m*t == t and (...)*m is dropped;
// the results are bit-identical to the general expressions.
template <bool WRITE_GRAD, bool WRITE_TARGETS, bool ACC, bool SMEM_PRED, bool UNIT, typename PT = float>
__device__ __forceinline__ void run_quads_impl(const MapIo& io, int m, const float4* chunk, int q_begin, int q_end,
                                               const JointVerdict& jv, const double* ex, const double* ey,
                                               MapState& st, int lane, float half_scale) {
    const int W = io.W, hw = io.H * io.W, qpr = W >> 2;
    const int step_y = 32 / qpr, step_x = 32 - step_y * qpr;
    const float mk = jv.weight, norm = io.norm;
    PT* gmap = reinterpret_cast<PT*>(io.grad) + (size_t)m * hw;                 // PT == float unless SMEM_PRED is false
    const PT* pmap = reinterpret_cast<const PT*>(chunk);                        // global path: chunk is the map base
    float4* t4 = reinterpret_cast<float4*>(io.targets + (size_t)m * hw);
    int y = st.y, xq = st.xq;
    float acc = st.acc;
    QuadBest bp = st.bp, bt = st.bt;
    const bool draw = jv.draw, track = st.track, track_t = st.track_t;
#pragma unroll 3
    for (int q = q_begin + lane; q < q_end; q += 32) {
        const float4 p = SMEM_PRED ? chunk[q - q_begin] : load_quad(pmap, q - q_begin);
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        if (draw) {
            const double2 a = *reinterpret_cast<const double2*>(ex + 4 * xq);
            const double2 b = *reinterpret_cast<const double2*>(ex + 4 * xq + 2);
            const double fy = ey[y];
            t.x = __double2float_rn(__dmul_rn(a.x, fy));
            t.y = __double2float_rn(__dmul_rn(a.y, fy));
            t.z = __double2float_rn(__dmul_rn(b.x, fy));
            t.w = __double2float_rn(__dmul_rn(b.y, fy));
        }
        const float px = UNIT ? p.x : __fmul_rn(mk, p.x), py = UNIT ? p.y : __fmul_rn(mk, p.y);
        const float pz = UNIT ? p.z : __fmul_rn(mk, p.z), pw = UNIT ? p.w : __fmul_rn(mk, p.w);
        const float tx = UNIT ? t.x : __fmul_rn(mk, t.x), ty = UNIT ? t.y : __fmul_rn(mk, t.y);
        const float tz = UNIT ? t.z : __fmul_rn(mk, t.z), tw = UNIT ? t.w : __fmul_rn(mk, t.w);
        const float dx = __fsub_rn(px, tx), dy = __fsub_rn(py, ty), dz = __fsub_rn(pz, tz), dw = __fsub_rn(pw, tw);
        acc = fmaf(dx, dx, acc);
        acc = fmaf(dy, dy, acc);
        acc = fmaf(dz, dz, acc);
        acc = fmaf(dw, dw, acc);
        if (WRITE_GRAD) {
            float4 g;
            g.x = __fmul_rn(__fmul_rn(norm, dx), half_scale);
            g.y = __fmul_rn(__fmul_rn(norm, dy), half_scale);
            g.z = __fmul_rn(__fmul_rn(norm, dz), half_scale);
            g.w = __fmul_rn(__fmul_rn(norm, dw), half_scale);
            if (!UNIT) {
                g.x = __fmul_rn(g.x, mk); g.y = __fmul_rn(g.y, mk); g.z = __fmul_rn(g.z, mk); g.w = __fmul_rn(g.w, mk);
            }
            store_quad(gmap, q, g);
        }
        if (WRITE_TARGETS) t4[q] = t;
        if (ACC && track) bp.push(px, py, pz, pw, q);
        if (ACC && track_t) bt.push(tx, ty, tz, tw, q);
        xq += step_x;
        y += step_y;
        if (xq >= qpr) { xq -= qpr; ++y; }
    }
    st.y = y; st.xq = xq; st.acc = acc; st.bp = bp; st.bt = bt;
}

template <bool WRITE_GRAD, bool WRITE_TARGETS, bool ACC, bool SMEM_PRED, typename PT = float>
__device__ __forceinline__ void run_quads(const MapIo& io, int m, const float4* chunk, int q_begin, int q_end,
                                          const JointVerdict& jv, const double* ex, const double* ey, MapState& st, int lane,
                                          float half_scale) {
    if (jv.weight == 1.0f) run_quads_impl<WRITE_GRAD, WRITE_TARGETS, ACC, SMEM_PRED, true, PT>(io, m, chunk, q_begin, q_end, jv, ex, ey, st, lane, half_scale);
    else                   run_quads_impl<WRITE_GRAD, WRITE_TARGETS, ACC, SMEM_PRED, false, PT>(io, m, chunk, q_begin, q_end, jv, ex, ey, st, lane, half_scale);
}

// Position of x factor i in the period-tiled kernel's layout: the four factors of a quad are split
// into two planes of (e0, e1) and (e2, e3) pairs, so that the 16-byte shared loads of eight
// consecutive lanes (consecutive quads of a row) cover 128 contiguous bytes. With the four doubles
// of a quad contiguous (32-byte lane stride) every such load was a 2-way bank conflict.
template <int QPR>
__device__ __forceinline__ int ex_slot(int i) {
    return QPR > 0 ? (((i >> 2) << 1) + (i & 1) + ((i & 2) ? 2 * QPR : 0)) : i;
}

// heat_map_to_axis of the masked target fl(mk * t) of a drawn map, found analytically: the factors decrease
// monotonically away from the centre, so every maximiser of the rounded products lies in the 3x3 block around
// the nearest in-map pixel. ex is laid out as ex_slot<QPR>.
template <int QPR>
__device__ __forceinline__ float2 analytic_target_axis(const MapIo& io, const JointVerdict& jv, float mk, const double* ex,
                                                       const double* ey, int lane) {
    const int W = io.W;
    const int xn = min(max(__float2int_rn(jv.mx), 0), W - 1), yn = min(max(__float2int_rn(jv.my), 0), io.H - 1);
    const int yy = yn - 1 + lane / 3, xx = xn - 1 + lane % 3;
    const bool in = lane < 9 && yy >= 0 && yy < io.H && xx >= 0 && xx < W;
    float v = -CUDART_INF_F;
    if (in) v = __fmul_rn(mk, __double2float_rn(__dmul_rn(ex[ex_slot<QPR>(xx)], ey[yy])));
    const Peak pk = warp_first_max(v, in ? (unsigned)(yy * W + xx) : 0x7fffffffu);
    return axis_of(pk.value, pk.index, W);
}

// HeatMapAcc coordinates of both masked maps (heat_map_to_axis). The winning quad of the predicted
// map is re-read from global memory (L2-resident: it has just streamed through), so the staged
// copy may already have been recycled.
template <typename PT = float>
__device__ __forceinline__ void end_map_acc(const MapIo& io, int m, const JointVerdict& jv, const double* ex,
                                            const double* ey, const MapState& st, int lane) {
    const int W = io.W, hw = io.H * io.W;
    const float mk = jv.weight;
    float2 pxy = make_float2(0.f, 0.f), lxy = make_float2(0.f, 0.f);
    if (st.track) {
        const PT* src = reinterpret_cast<const PT*>(io.pred) + (size_t)m * hw;
        const Peak pp = __any_sync(SP_FULL, st.bp.poison != st.bp.poison) ? argmax_exact(MaskedPredView<PT>{src, mk}, hw, lane)
                                                                            : st.bp.warp_peak();
        pxy = axis_of(pp.value, pp.index, W);
        // target map: fl(m * t); always finite
        if (st.analytic_t) {
            lxy = analytic_target_axis<0>(io, jv, mk, ex, ey, lane);
        } else if (jv.draw) {
            const Peak pt = st.bt.warp_peak();
            lxy = axis_of(pt.value, pt.index, W);
        }
    }
    if (lane == 0) {
        io.pred_xy[m] = pxy;
        io.label_xy[m] = lxy;
    }
}

struct Joint3 {
    float x, y, v;
};
__device__ __forceinline__ Joint3 load_joint(const MapIo& io, int m) {
    Joint3 j;
    j.x = j.y = j.v = 0.f;
    if (m < io.nmaps) {
        j.x = __ldg(io.joints + 3 * (size_t)m + 0);
        j.y = __ldg(io.joints + 3 * (size_t)m + 1);
        j.v = __ldg(io.joints + 3 * (size_t)m + 2);
    }
    return j;
}

// joint -> verdict, weight store, float64 factors into this warp's shared-memory slice
template <int QPR = 0>
__device__ __forceinline__ JointVerdict prepare_map(const MapIo& io, int m, const Joint3 j, double* ex, double* ey, int lane) {
    const float mx = j.x, my = j.y, vis = j.v;
    const JointVerdict jv = judge_joint(mx, my, vis, io.reach, io.H, io.W);
    if (lane == 0 && io.weights) io.weights[m] = jv.weight;
    __syncwarp();
    if (jv.draw) {
        for (int i = lane; i < io.W + io.H; i += 32) {
            if (i < io.W) ex[ex_slot<QPR>(i)] = gauss_factor(i, mx, io.denom);
            else          ey[i - io.W] = gauss_factor(i - io.W, my, io.denom);
        }
    }
    __syncwarp();
    return jv;
}


// ---- period-tiled map body (variant C of sp_train.cu) ----------------------------------------------------------------
constexpr int kFifo = 16;          // entries per warp; the producer is never more than ring+2 <= 10 maps ahead
constexpr int kRingHeader = 1024 + 2048 + 64;

constexpr int cgcd(int a, int b) { return b == 0 ? a : cgcd(b, a % b); }

template <int QPR>
struct Tile {
    static constexpr int G = cgcd(32, QPR);
    static constexpr int PERIOD = QPR / G;
    static constexpr int ROWS = 32 / G;
    static constexpr bool EX_IN_REGS = PERIOD <= 3;
};

__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ double lds64f(uint32_t addr) {
    double r;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(r) : "r"(addr));
    return r;
}
__device__ __forceinline__ double2 lds128d(uint32_t addr) {
    double2 r;
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(r.x), "=d"(r.y) : "r"(addr));
    return r;
}
__device__ __forceinline__ bool mbar_try_wait_a(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}

// Per-warp ring of RING slots of CHUNK_BYTES, all shared-memory addresses 32-bit.
template <int RING, int CHUNK_BYTES>
struct TileRing {
    uint32_t bar0, slot0;        // shared addresses of this warp's first barrier / slot
    uint32_t cs, parity;         // consumer slot and phase
    // producer side (lane 0): next chunk to request
    const char* src;             // global address of the next chunk
    int left;                    // chunks of the current map still to request (0: no map)
    int pnext;                   // map claimed after the current one (-1: none)
    uint32_t ps;
    int tail, nmaps;
    int inflight, depth;         // copies in flight / copies kept in flight while there are unclaimed maps
    int static_next, static_left, static_stride, dyn_base;
    volatile int* fifo;
    unsigned int* next_work;     // grid-wide counter in the caller's workspace
    const char* pred;
    size_t map_bytes;
    int chunks_per_map;

    // Maps are dealt GRID-WIDE: the first two of every warp are fixed (no atomic storm at launch), the
    // rest come from one counter in the caller's workspace, one map ahead of the copies being issued.
    // A per-CTA range would make the slowest SM the critical path, and the SMs are far from equal once
    // the memory system queues: at 96x72 half the TPCs finished equal ranges in ~58 us and the other
    // half in ~86 us (per-warp timestamps, profiles/r1f_fused_timeline.md).
    __device__ __forceinline__ int claim() {
        int m;
        if (static_left > 0) {
            m = static_next;
            static_next += static_stride;
            --static_left;
        } else {
            m = dyn_base + (int)atomicAdd(next_work, 1u);
        }
        const int got = (m >= 0 && m < nmaps) ? m : -1;
        fifo[tail & (kFifo - 1)] = got;
        ++tail;
        return got;
    }
    __device__ __forceinline__ void start(int m) {           // lane 0
        left = 0;
        pnext = -1;
        if (m >= 0) {
            src = pred + (size_t)m * map_bytes;
            left = chunks_per_map;
            pnext = claim();
        }
    }
    __device__ __forceinline__ void issue_next() {           // lane 0
        if (left == 0) return;
        const uint32_t bar = bar0 + ps * 8u, dst = slot0 + ps * (uint32_t)CHUNK_BYTES;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "n"(CHUNK_BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(dst), "l"(src), "n"(CHUNK_BYTES), "r"(bar) : "memory");
        src += CHUNK_BYTES;
        ++inflight;
        if (--left == 0 && pnext >= 0) {
            src = pred + (size_t)pnext * map_bytes;
            left = chunks_per_map;
            pnext = claim();
        }
        if (RING > 1) ps = (ps + 1 == RING) ? 0u : ps + 1;
    }
    // Keep `depth` copies in flight while the CTA has maps left to hand out; once this warp is on its
    // last map (nothing claimed behind it) use every slot: the SM's other warps are running dry, a
    // lone warp at depth 1 pulls ~1.3 KB/us of the SM's 22 KB/us, and the deeper ring that is slower
    // under full load (HBM read/write turnarounds) is what shortens the launch tail.
    __device__ __forceinline__ void top_up() {               // lane 0
        const int want = (pnext < 0) ? RING : depth;
        while (inflight < want && left > 0) issue_next();
    }
    __device__ __forceinline__ uint32_t wait() {             // returns the shared address of the chunk
        const uint32_t bar = bar0 + cs * 8u;
        while (!mbar_try_wait_a(bar, parity)) {
        }
        return slot0 + cs * (uint32_t)CHUNK_BYTES;
    }
    __device__ __forceinline__ void release(int lane) {
        __syncwarp();
        if (lane == 0) {
            sp::fence_proxy_async_smem();
            --inflight;
            top_up();                                        // refills the slot just drained (and more in the tail)
        }
        if (RING > 1) {
            if (++cs == RING) { cs = 0; parity ^= 1u; }
        } else {
            parity ^= 1u;
        }
    }
};

// The predicted-map argmax of one map whose winning quad is still on its way back from L2.
struct PendingAxis {
    int m;              // < 0: nothing pending
    int quad;
    float gmax, mk;
    float4 v;
};

__device__ __forceinline__ void flush_pending(const MapIo& io, PendingAxis& pd, int lane) {
    if (pd.m < 0) return;
    const float a = __fmul_rn(pd.mk, pd.v.x), b = __fmul_rn(pd.mk, pd.v.y), c = __fmul_rn(pd.mk, pd.v.z);
    const int sub = (a == pd.gmax) ? 0 : (b == pd.gmax) ? 1 : (c == pd.gmax) ? 2 : 3;
    if (lane == 0) io.pred_xy[pd.m] = axis_of(pd.gmax, 4 * pd.quad + sub, io.W);
    pd.m = -1;
}

// One map, its chunks arriving through the warp's TileRing: writes the gradient (never the targets), returns this
// lane's share of sum((m*p - m*t)^2) and, with ACC, the HeatMapAcc coordinates.
// MODE 0: Gaussian drawn, mask == 1, argmax tracked iff ACC (the common case);
// MODE 1: nothing drawn and mask == 0 (invisible / culled joint): target 0, no tracking;
// MODE 2: anything else (odd mask values, sigma outside the analytic range): run-time flags.
template <int QPR, int PPC, bool ACC, int MODE, int RING, int CHUNK_BYTES>
__device__ __forceinline__ float tile_map(const MapIo& io, int m, const JointVerdict& jv, const double* ex, const double* ey,
                                          TileRing<RING, CHUNK_BYTES>& rg, PendingAxis& pd, int lane) {
    using T = Tile<QPR>;
    constexpr int PERIOD = T::PERIOD, ROWS = T::ROWS;
    constexpr int CHUNK_QUADS = PPC * 32 * PERIOD;
    const int hw = io.H * io.W;
    const bool draw = (MODE == 0) ? true : (MODE == 1) ? false : jv.draw;
    const bool unit = (MODE == 0);
    const bool track = ACC && ((MODE == 0) ? true : (MODE == 1) ? false : (jv.weight != 0.f));
    const bool analytic_t = track && draw && io.analytic_ok && jv.weight >= 0.5f && jv.weight <= 4.f;
    const bool track_t = (MODE == 2) && track && draw && !analytic_t;
    const float mk = unit ? 1.0f : jv.weight, norm = io.norm, half_scale = io.half_scale;

    // per-lane constants of one period: shared addresses of the row factor and of the x factors
    const uint32_t ex_a = sp::smem_u32(ex), ey_a = sp::smem_u32(ey);
    uint32_t eya[PERIOD], exa[PERIOD];
#pragma unroll
    for (int j = 0; j < PERIOD; ++j) {
        const int q = lane + 32 * j;
        const int y = q / QPR;
        eya[j] = ey_a + 8u * (uint32_t)y;
        exa[j] = ex_a + 16u * (uint32_t)(q - y * QPR);           // (e0, e1) plane; (e2, e3) is 16*QPR bytes further
    }
    double exr[T::EX_IN_REGS ? PERIOD : 1][4];
    if (T::EX_IN_REGS && draw) {
#pragma unroll
        for (int j = 0; j < PERIOD; ++j) {
            const double2 a = lds128d(exa[j]), b = lds128d(exa[j] + 16u * QPR);
            exr[j][0] = a.x; exr[j][1] = a.y; exr[j][2] = b.x; exr[j][3] = b.y;
        }
    }

    float acc = 0.f;
    float best = -CUDART_INF_F, tbest = -CUDART_INF_F;
    int bq = lane, tbq = lane;
    int qlane = lane;                                   // this lane's quad at step 0 of the current chunk
    float4* g4 = reinterpret_cast<float4*>(io.grad + (size_t)m * hw) + lane;
    const int chunks = (hw >> 2) / CHUNK_QUADS;

#pragma unroll 1
    for (int c = 0; c < chunks; ++c) {
        const uint32_t chunk = rg.wait() + 16u * (uint32_t)lane;
#pragma unroll
        for (int it = 0; it < PPC; ++it) {
#pragma unroll
            for (int j = 0; j < PERIOD; ++j) {
                const int step = it * PERIOD + j;
                const float4 p = lds128(chunk + 512u * step);
                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                if (draw) {
                    const double fy = lds64f(eya[j] + 8u * (uint32_t)(it * ROWS));
                    double e0, e1, e2, e3;
                    if (T::EX_IN_REGS) {
                        e0 = exr[j][0]; e1 = exr[j][1]; e2 = exr[j][2]; e3 = exr[j][3];
                    } else {
                        const double2 a = lds128d(exa[j]), b = lds128d(exa[j] + 16u * QPR);
                        e0 = a.x; e1 = a.y; e2 = b.x; e3 = b.y;
                    }
                    t.x = __double2float_rn(__dmul_rn(e0, fy));
                    t.y = __double2float_rn(__dmul_rn(e1, fy));
                    t.z = __double2float_rn(__dmul_rn(e2, fy));
                    t.w = __double2float_rn(__dmul_rn(e3, fy));
                }
                const float px = unit ? p.x : __fmul_rn(mk, p.x), py = unit ? p.y : __fmul_rn(mk, p.y);
                const float pz = unit ? p.z : __fmul_rn(mk, p.z), pw = unit ? p.w : __fmul_rn(mk, p.w);
                const float tx = unit ? t.x : __fmul_rn(mk, t.x), ty = unit ? t.y : __fmul_rn(mk, t.y);
                const float tz = unit ? t.z : __fmul_rn(mk, t.z), tw = unit ? t.w : __fmul_rn(mk, t.w);
                const float dx = __fsub_rn(px, tx), dy = __fsub_rn(py, ty), dz = __fsub_rn(pz, tz), dw = __fsub_rn(pw, tw);
                acc = fmaf(dx, dx, acc);
                acc = fmaf(dy, dy, acc);
                acc = fmaf(dz, dz, acc);
                acc = fmaf(dw, dw, acc);
                float4 g;
                g.x = __fmul_rn(__fmul_rn(norm, dx), half_scale);
                g.y = __fmul_rn(__fmul_rn(norm, dy), half_scale);
                g.z = __fmul_rn(__fmul_rn(norm, dz), half_scale);
                g.w = __fmul_rn(__fmul_rn(norm, dw), half_scale);
                if (!unit) {
                    g.x = __fmul_rn(g.x, mk); g.y = __fmul_rn(g.y, mk); g.z = __fmul_rn(g.z, mk); g.w = __fmul_rn(g.w, mk);
                }
                g4[32 * step] = g;
                if (track) {
                    const float m4 = sp::fmax_nan(sp::fmax_nan(px, py), sp::fmax_nan(pz, pw));
                    if (m4 > best) bq = qlane + 32 * step;
                    best = sp::fmax_nan(best, m4);          // NaN sticks: resolved by the exact scan below
                }
                if (track_t) {
                    const float m4 = fmaxf(fmaxf(tx, ty), fmaxf(tz, tw));
                    if (m4 > tbest) { tbest = m4; tbq = qlane + 32 * step; }
                }
            }
        }
        rg.release(lane);
        g4 += CHUNK_QUADS;
        qlane += CHUNK_QUADS;
#pragma unroll
        for (int j = 0; j < PERIOD; ++j) eya[j] += 8u * (uint32_t)(PPC * ROWS);
    }

    if (ACC) {
        flush_pending(io, pd, lane);                 // the previous map's quad arrived long ago
        float2 lxy = make_float2(0.f, 0.f);
        if (track) {
            const float* src = io.pred + (size_t)m * hw;
            if (__any_sync(SP_FULL, best != best)) {
                const Peak pk = argmax_exact(MaskedPredView<float>{src, mk}, hw, lane);
                if (lane == 0) io.pred_xy[m] = axis_of(pk.value, pk.index, io.W);
            } else {
                // every lane kept the first quad holding its own maximum: the smallest quad among
                // the lanes that hold the warp-wide maximum contains torch.max's answer
                const Peak g = warp_first_max(best, (unsigned)bq);
                pd.m = m;
                pd.quad = g.index;
                pd.gmax = g.value;
                pd.mk = mk;
                pd.v = __ldg(reinterpret_cast<const float4*>(src) + g.index);
            }
            if (analytic_t) {
                lxy = analytic_target_axis<QPR>(io, jv, mk, ex, ey, lane);
            } else if (track_t) {
                const Peak g = warp_first_max(tbest, (unsigned)tbq);
                const float gmax = g.value;
                const int gq = g.index;
                const int y = gq / QPR, x4 = 4 * (gq - y * QPR);
                int sub = 3;
#pragma unroll
                for (int e = 2; e >= 0; --e)
                    if (__fmul_rn(mk, __double2float_rn(__dmul_rn(ex[ex_slot<QPR>(x4 + e)], ey[y]))) == gmax) sub = e;
                lxy = axis_of(gmax, 4 * gq + sub, io.W);
            }
        } else if (lane == 0) {
            io.pred_xy[m] = make_float2(0.f, 0.f);
        }
        if (lane == 0) io.label_xy[m] = lxy;
    }
    return acc;
}

}  // namespace sp_trn
