// The argmax of a map with torch.max semantics (NaN beats every number, -0 equals +0, the smaller index wins a
// tie) and the HeatMapAcc epilogue on the argmax axes, shared by the decode (sp_decode_dev.cuh), masked-MSE loss
// (sp_loss.cu), fused training (sp_train_dev.cuh) and step (sp_step.cu) kernels. Each kernel keeps its own running
// argmax loop; what it does after the loop -- the warp merge, the exact scan when a NaN or an infinity was seen, the
// axes and the epilogue -- is here.
#pragma once
#include "sp_common.cuh"
#include "sp_lowp.cuh"
#include <math_constants.h>

namespace sp_arg {

struct Peak {
    float value;
    int index;
};

// warp-wide max in one instruction (redux.sync.max.f32, sm_100a; SASS CREDUX)
__device__ __forceinline__ float warp_max_f32(float v) {
    float r;
    asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
    return r;
}

// Every value of the warp finite (or -inf): the warp-wide maximum and the smallest `index` among the lanes that hold
// it. A lane that holds nothing passes -inf, or 0x7fffffff as its index.
__device__ __forceinline__ Peak warp_first_max(float v, unsigned index) {
    Peak p;
    p.value = warp_max_f32(v);
    p.index = (int)__reduce_min_sync(SP_FULL, (v == p.value) ? index : 0x7fffffffu);
    return p;
}

// (value, index) butterfly with sp::better: any values, NaN included
__device__ __forceinline__ Peak warp_best(float v, int i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(SP_FULL, v, o);
        const int oi = __shfl_xor_sync(SP_FULL, i, o);
        if (sp::better(ov, oi, v, i)) { v = ov; i = oi; }
    }
    Peak p;
    p.value = v;
    p.index = i;
    return p;
}

struct DirectView {
    const float* p;
    __device__ __forceinline__ float at(int i) const { return p[i]; }
};

template <typename PT = float>
struct MaskedPredView {          // m * pred[i] (float(pred[i]) * m for float16 / bfloat16 pred)
    const PT* p;
    float m;
    __device__ __forceinline__ float at(int i) const { return __fmul_rn(m, sp_lowp::to_float(p[i])); }
};

// exact scalar scan of map.at(0 .. hw-1); the fallback of every vector scan that met a NaN or an infinity
template <typename View>
__device__ __noinline__ Peak argmax_exact(const View map, int hw, int lane) {
    float bv = -CUDART_INF_F;
    int bi = 0x7fffffff;
    for (int i = lane; i < hw; i += 32) {
        const float v = map.at(i);
        if (sp::better(v, i, bv, bi)) { bv = v; bi = i; }
    }
    return warp_best(bv, bi);
}

// running (value, quad) argmax over the quads a lane visits in increasing order
struct QuadBest {
    float best;
    int bq;
    int bsub;          // first element of quad bq that equals best
    float poison;      // NaN once a quad held a NaN or an infinity
    __device__ __forceinline__ void init() { best = -CUDART_INF_F; bq = 0x0fffffff; bsub = 0; poison = 0.f; }
    __device__ __forceinline__ void push(float a, float b, float c, float d, int q) {
        const float m4 = sp::fmax_nan(sp::fmax_nan(a, b), sp::fmax_nan(c, d));
        poison = fmaf(m4, 0.f, poison);
        if (m4 > best) {
            best = m4;
            bq = q;
            bsub = (a == m4) ? 0 : (b == m4) ? 1 : (c == m4) ? 2 : 3;
        }
    }
    // No lane of the warp poisoned: every lane holds the first maximal element of its own quads, so the smallest
    // flat index among the lanes that hold the warp-wide maximum is torch.max's answer.
    __device__ __forceinline__ Peak warp_peak() const { return warp_first_max(best, (unsigned)(4 * bq + bsub)); }
};

// heat_map_to_axis on an index/value pair: (x, y) as floats, zeroed when the max is not > 0
__device__ __forceinline__ float2 axis_of(float val, int idx, int W) {
    if (!(val > 0.f)) return make_float2(0.f, 0.f);
    const int y = idx / W;
    return make_float2((float)(idx - y * W), (float)y);
}

// HeatMapAcc epilogue (metrics/pose_metrics.py:227-245) on the [B,K] argmax coordinates, run by ALL threads of one
// block; counters = 2K ints of shared memory. Every step is a correctly rounded float32 operation in the oracle's order
// (divide, subtract, the distance below, compare), so each verdict is the oracle's. The per-joint counts do not depend
// on the order the threads add them in and one thread sums the joints in order, so every block size gives the same bits. COHERENT: read the axes through L2
// (ld.global.cg) because other CTAs of the same launch wrote them (the caller has acquired their writes).
template <bool COHERENT>
__device__ __forceinline__ void heatmap_acc_block(const float2* __restrict__ pred_xy, const float2* __restrict__ label_xy,
                                                  float* __restrict__ acc, int B, int K, float norm_x, float norm_y,
                                                  float thresh, int* counters) {
    int* hit = counters;
    int* valid = counters + K;
    for (int k = threadIdx.x; k < 2 * K; k += blockDim.x) counters[k] = 0;
    __syncthreads();
    const int n = B * K;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float2 l = COHERENT ? __ldcg(label_xy + i) : label_xy[i];
        if (l.x > 1.f && l.y > 1.f) {
            const float2 p = COHERENT ? __ldcg(pred_xy + i) : pred_xy[i];
            const float dx = __fsub_rn(__fdiv_rn(p.x, norm_x), __fdiv_rn(l.x, norm_x));
            const float dy = __fsub_rn(__fdiv_rn(p.y, norm_y), __fdiv_rn(l.y, norm_y));
            // torch.norm(d, dim=-1) of a float32 pair on the CPU (the pinned oracle) is sqrtf(fmaf(dy, dy, dx * dx)),
            // in float32 (tests/test_heatmap_acc_norm_cpu.py pins it). A double sum rounded once differs in the last
            // bit for about one offset in nine, and some of those lie on the threshold: at 100 x 100 with the defaults,
            // pred (0, 3) and label (3, 7) are 0.49999997 apart, a hit, where the double form gives 0.5, a miss.
            const float dist = __fsqrt_rn(__fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
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

}  // namespace sp_arg
