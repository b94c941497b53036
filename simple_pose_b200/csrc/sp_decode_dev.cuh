// Device-side building blocks of the heatmap decoders (the vector argmax scan of a staged map, the 13-point blur +
// Taylor refinement, the epilogue with the affine back-projection), shared by the decode kernels (sp_decode.cu) and
// the one-launch step kernel (sp_step.cu). The argmax rule itself is in sp_argmax.cuh. See sp_decode.cu for the
// design notes.
#pragma once
#include "sp_common.cuh"
#include "sp_argmax.cuh"
#include <math_constants.h>

namespace sp_dec {

using namespace sp_arg;

constexpr int kMaxKsize = 15;
constexpr int kStencil = 13;
constexpr int kPatchMax = kMaxKsize + 4;               // 19
constexpr int kPatchFloats = kPatchMax * kPatchMax;    // 361

struct DecodeArgs {
    const float* hm;
    const float* hm_flip;
    const int* perm;
    const float* trans_inv;
    const float* blur_w;
    float* coords;
    float* maxval;
    int* argmax;
    float* rows;               // optional result table: rows[person * row_stride + 3*joint + {0,1,2}] = x, y, peak value
    int row_stride;
    int nmaps, K, H, W, ksize, mode;
    unsigned int* work;        // caller's workspace {next map, CTAs finished}; nullptr = equal per-CTA ranges
};

// 13 stencil points (dy, dx): centre, x+-1, y+-1, x+-2, y+-2, four diagonals.
#define SP_STENCIL_DY {0, 0, 0, 1, -1, 0, 0, 2, -2, 1, -1, 1, -1}
#define SP_STENCIL_DX {0, 1, -1, 0, 0, 2, -2, 0, 0, 1, 1, -1, -1}
enum { S_C = 0, S_XP1, S_XM1, S_YP1, S_YM1, S_XP2, S_XM2, S_YP2, S_YM2, S_PP, S_MP, S_PM, S_MM };
// S_PP = (y+1,x+1), S_MP = (y-1,x+1), S_PM = (y+1,x-1), S_MM = (y-1,x-1)

// warp-wide min in one instruction (redux.sync.min.f32, sm_100a; SASS CREDUX)
__device__ __forceinline__ float warp_min_f32(float v) {
    float r;
    asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
    return r;
}

// 0.5*(a[y,x] + b[y,W-1-x]) evaluated on the fly (generic path of the flip test)
struct FlipAvgView {
    const float* a;
    const float* b;
    int W;
    __device__ __forceinline__ float at(int i) const {
        const int y = i / W, x = i - y * W;
        return __fmul_rn(0.5f, __fadd_rn(a[i], b[y * W + (W - 1 - x)]));
    }
};

// ---------------------------------------------------------------------------------------------
// argmax of a map that is resident in shared memory (the generic path runs argmax_exact on the map in place)
// ---------------------------------------------------------------------------------------------
// Vector scan over a shared-memory map (hw % 4 == 0). If FLIP, first folds the mirrored partner
// map into `a` in place (W % 4 == 0 so the mirror of an aligned quad is an aligned quad).
template <bool FLIP>
__device__ __forceinline__ Peak argmax_smem(float* a, const float* b, int hw, int W, int lane) {
    const int nq = hw >> 2;
    float best = -CUDART_INF_F;
    int bq = 0x3fffffff;
    float poison = 0.f;                 // becomes NaN if any quad max is NaN or +-Inf
    float4* a4 = reinterpret_cast<float4*>(a);
    const int qpr = W >> 2;
    int y = 0, xq = 0, step_y = 0, step_x = 0;
    if (FLIP) {
        y = lane / qpr;
        xq = lane - y * qpr;
        step_y = 32 / qpr;
        step_x = 32 - step_y * qpr;
    }
#pragma unroll 4
    for (int q = lane; q < nq; q += 32) {
        float4 v = a4[q];
        if (FLIP) {
            const float4 m = *reinterpret_cast<const float4*>(b + y * W + (W - 4 - 4 * xq));
            v.x = __fmul_rn(0.5f, __fadd_rn(v.x, m.w));
            v.y = __fmul_rn(0.5f, __fadd_rn(v.y, m.z));
            v.z = __fmul_rn(0.5f, __fadd_rn(v.z, m.y));
            v.w = __fmul_rn(0.5f, __fadd_rn(v.w, m.x));
            a4[q] = v;
            xq += step_x;
            y += step_y;
            if (xq >= qpr) { xq -= qpr; ++y; }
        }
        const float m4 = sp::fmax_nan(sp::fmax_nan(v.x, v.y), sp::fmax_nan(v.z, v.w));
        poison = fmaf(m4, 0.f, poison);
        if (m4 > best) { best = m4; bq = q; }
    }
    if (FLIP) __syncwarp();             // folded values visible to the whole warp
    const bool weird = __any_sync(SP_FULL, poison != poison);
    if (weird) {
        DirectView view{a};
        return argmax_exact(view, hw, lane);
    }
    // all values finite: warp max in one CREDUX, then the smallest quad index that attains it
    const Peak g = warp_first_max(best, (unsigned)bq);
    const float gmax = g.value;
    const unsigned gq = (unsigned)g.index;
    const float4 w = a4[gq];            // broadcast read; first element of the quad equal to the max
    const int sub = (w.x == gmax) ? 0 : (w.y == gmax) ? 1 : (w.z == gmax) ? 2 : 3;
    Peak p;
    p.value = (sub == 0) ? w.x : (sub == 1) ? w.y : (sub == 2) ? w.z : w.w;   // keeps the sign of a zero
    p.index = 4 * (int)gq + sub;
    return p;
}

// ---------------------------------------------------------------------------------------------
// Taylor refinement around an interior peak. All lanes return the same values.
// ---------------------------------------------------------------------------------------------
// exact slow path: max over the whole zero-padded blurred map of this joint
template <typename View>
__device__ __noinline__ float full_blur_max(const View map, const float* w, int H, int W, int ks, int lane) {
    const int r = ks >> 1;
    float best = -CUDART_INF_F;
    bool seen_nan = false;
    for (int i = lane; i < H * W; i += 32) {
        const int y = i / W, x = i - y * W;
        float acc = 0.f;
        for (int ty = 0; ty < ks; ++ty) {
            const int yy = y + ty - r;
            if (yy < 0 || yy >= H) continue;
            for (int tx = 0; tx < ks; ++tx) {
                const int xx = x + tx - r;
                if (xx < 0 || xx >= W) continue;
                acc = fmaf(w[ty * ks + tx], map.at(yy * W + xx), acc);
            }
        }
        if (acc != acc) seen_nan = true;
        best = fmaxf(best, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = fmaxf(best, __shfl_xor_sync(SP_FULL, best, o));
    if (__any_sync(SP_FULL, seen_nan)) best = CUDART_NAN_F;   // torch.max propagates NaN
    return best;
}

// log of one blurred stencil value on the exact path: log(clamp(blur * ori_max / blur_max, 1e-10))
__device__ __forceinline__ float exact_log(float blur, float ori_max, float bmax) {
    const float v = __fdiv_rn(__fmul_rn(blur, ori_max), bmax);
    return logf((v != v) ? v : fmaxf(v, 1e-10f));            // torch.clamp(min=) keeps NaN
}

// finite differences + 2x2 solve, same operation order as pose_metrics.py:80-100
__device__ __forceinline__ bool taylor_step(const float (&L)[kStencil], float& ox, float& oy) {
    const float dx = __fmul_rn(0.5f, __fsub_rn(L[S_XP1], L[S_XM1]));
    const float dy = __fmul_rn(0.5f, __fsub_rn(L[S_YP1], L[S_YM1]));
    const float c2 = __fmul_rn(2.f, L[S_C]);
    const float dxx = __fmul_rn(0.25f, __fadd_rn(__fsub_rn(L[S_XP2], c2), L[S_XM2]));
    const float dyy = __fmul_rn(0.25f, __fadd_rn(__fsub_rn(L[S_YP2], c2), L[S_YM2]));
    const float dxy = __fmul_rn(0.25f, __fadd_rn(__fsub_rn(__fsub_rn(L[S_PP], L[S_MP]), L[S_PM]), L[S_MM]));
    const float det = __fsub_rn(__fmul_rn(dxx, dyy), __fmul_rn(dxy, dxy));
    if (!(det != 0.f)) return false;                          // det == 0 -> skip; NaN != 0 is true, as in torch
    const float inv = __fdiv_rn(1.f, det);                    // offset = -H^-1 g, H = [[dxx, dxy], [dxy, dyy]]
    ox = -__fmul_rn(__fsub_rn(__fmul_rn(dyy, dx), __fmul_rn(dxy, dy)), inv);
    oy = -__fmul_rn(__fsub_rn(__fmul_rn(dxx, dy), __fmul_rn(dxy, dx)), inv);
    return true;
}

// Which of the three cases of the file header applies. Returns 0 = clamp cannot fire (drop the
// common factor), 1 = exact path with blur_max, 2 = every log equals log(1e-10) -> not refined.
template <typename View>
__device__ __forceinline__ int clamp_case(const View& map, const float* wts, int H, int W, int ks, int lane,
                                          float lo, float hi, bool any_nan, float ori_max, float& bmax) {
    if (!any_nan && lo >= 2e-10f) return 0;
    bmax = full_blur_max(map, wts, H, W, ks, lane);
    if (!any_nan && hi <= 0.f && ori_max > 0.f && bmax > 0.f) return 2;
    return 1;
}

// ---- generic kernel size (runtime ks), any memory space -------------------------------------
template <typename View>
__device__ __noinline__ bool taylor_refine_generic(const View map, const float* wts, float* patch, int H, int W,
                                                   int ks, int px, int py, float ori_max, int lane, float& ox, float& oy) {
    const int r = ks >> 1;
    const int P = ks + 4;               // patch side: blur radius + stencil radius 2 on each side
    const int pr = r + 2;
    __syncwarp();
    for (int e = lane; e < P * P; e += 32) {   // zero-padded patch of the raw map around the peak
        const int ry = e / P, rx = e - ry * P;
        const int yy = py + ry - pr, xx = px + rx - pr;
        patch[e] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? map.at(yy * W + xx) : 0.f;
    }
    __syncwarp();
    constexpr int kStencilDy[kStencil] = SP_STENCIL_DY;
    constexpr int kStencilDx[kStencil] = SP_STENCIL_DX;
    float acc[kStencil];
#pragma unroll
    for (int s = 0; s < kStencil; ++s) acc[s] = 0.f;
    for (int t = lane; t < ks * ks; t += 32) {
        const int ty = t / ks, tx = t - ty * ks;
        const float wv = wts[t];
        const float* base = patch + (ty + 2) * P + (tx + 2);
#pragma unroll
        for (int s = 0; s < kStencil; ++s) acc[s] = fmaf(wv, base[kStencilDy[s] * P + kStencilDx[s]], acc[s]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int s = 0; s < kStencil; ++s) acc[s] += __shfl_xor_sync(SP_FULL, acc[s], o);
    }
    float lo = acc[0], hi = acc[0];
    bool any_nan = false;
#pragma unroll
    for (int s = 0; s < kStencil; ++s) {
        lo = fminf(lo, acc[s]);
        hi = fmaxf(hi, acc[s]);
        any_nan |= (acc[s] != acc[s]);
    }
    float bmax = 1.f;
    const int which = clamp_case(map, wts, H, W, ks, lane, lo, hi, any_nan, ori_max, bmax);
    if (which == 2) return false;
    float L[kStencil];
#pragma unroll
    for (int s = 0; s < kStencil; ++s) L[s] = (which == 0) ? logf(acc[s]) : exact_log(acc[s], ori_max, bmax);
    return taylor_step(L, ox, oy);
}

// ---- KS x KS kernel known at compile time, map in shared memory ------------------------------
// Per-lane share of the KS*KS taps: weights and (row+2, col+2) offsets, set up once per kernel.
template <int KS>
struct LaneTaps {
    static constexpr int N = (KS * KS + 31) / 32;
    float w[N];
    int ty2[N], tx2[N];
    __device__ __forceinline__ void load(const float* wts, int lane) {
#pragma unroll
        for (int j = 0; j < N; ++j) {
            const int t = lane + 32 * j;
            const bool real = t < KS * KS;
            const int tt = real ? t : 0;
            w[j] = real ? wts[tt] : 0.f;
            ty2[j] = tt / KS + 2;
            tx2[j] = tt % KS + 2;
        }
    }
};

// Sum 13 per-lane partials across the warp so that lane 16*b4 + 2*local (+1) ends up holding the
// total of slot s = 7*b4 + local: recursive halving, 7+4+2+1+1 = 15 shuffles instead of 65.
__device__ __forceinline__ float reduce_scatter13(float (&v)[kStencil], int lane) {
    const bool up16 = lane & 16, up8 = lane & 8, up4 = lane & 4, up2 = lane & 2;
    float a[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) {
        const float hi = (j + 7 < kStencil) ? v[j + 7] : 0.f;
        const float send = up16 ? v[j] : hi;
        const float keep = up16 ? hi : v[j];
        a[j] = keep + __shfl_xor_sync(SP_FULL, send, 16);
    }
    float b[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float hi = (j + 4 < 7) ? a[j + 4] : 0.f;
        const float send = up8 ? a[j] : hi;
        const float keep = up8 ? hi : a[j];
        b[j] = keep + __shfl_xor_sync(SP_FULL, send, 8);
    }
    float c[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float send = up4 ? b[j] : b[j + 2];
        const float keep = up4 ? b[j + 2] : b[j];
        c[j] = keep + __shfl_xor_sync(SP_FULL, send, 4);
    }
    const float send = up2 ? c[0] : c[1];
    const float keep = up2 ? c[1] : c[0];
    float d = keep + __shfl_xor_sync(SP_FULL, send, 2);
    d += __shfl_xor_sync(SP_FULL, d, 1);
    return d;
}
__device__ __forceinline__ bool lane_has_slot(int lane) { return ((lane >> 1) & 7) < ((lane & 16) ? 6 : 7); }
__device__ __forceinline__ constexpr int lane_of_slot(int s) { return (s >= 7) ? 16 + 2 * (s - 7) : 2 * s; }

template <int KS>
__device__ __forceinline__ bool taylor_refine_smem(const float* map, const float* wts, float* patch,
                                                   const LaneTaps<KS>& taps, int H, int W, int px, int py,
                                                   float ori_max, int lane, float& ox, float& oy) {
    constexpr int R = KS / 2, P = KS + 4, PR = R + 2;
    // All 13 windows inside the map (the common case): read the map in place. Otherwise build a
    // zero-padded P x P patch of the raw map around the peak and read that.
    const float* org;
    int stride;
    if (px >= PR && px + PR < W && py >= PR && py + PR < H) {
        org = map + (py - PR) * W + (px - PR);
        stride = W;
    } else {
        __syncwarp();
        for (int e = lane; e < P * P; e += 32) {
            const int ry = e / P, rx = e - ry * P;
            const int yy = py + ry - PR, xx = px + rx - PR;
            patch[e] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? map[yy * W + xx] : 0.f;
        }
        __syncwarp();
        org = patch;
        stride = P;
    }
    constexpr int kStencilDy[kStencil] = SP_STENCIL_DY;
    constexpr int kStencilDx[kStencil] = SP_STENCIL_DX;
    float acc[kStencil];
#pragma unroll
    for (int s = 0; s < kStencil; ++s) acc[s] = 0.f;
#pragma unroll
    for (int j = 0; j < LaneTaps<KS>::N; ++j) {
        if (j + 1 < LaneTaps<KS>::N || lane + 32 * j < KS * KS) {      // only the last round is ragged
            const float* base = org + taps.ty2[j] * stride + taps.tx2[j];
            const float wv = taps.w[j];
#pragma unroll
            for (int s = 0; s < kStencil; ++s) acc[s] = fmaf(wv, base[kStencilDy[s] * stride + kStencilDx[s]], acc[s]);
        }
    }
    const float mine = reduce_scatter13(acc, lane);          // blurred value of this lane's stencil slot
    const bool own = lane_has_slot(lane);
    const bool any_nan = __any_sync(SP_FULL, own && (mine != mine));
    const float lo = warp_min_f32(own ? mine : CUDART_INF_F);
    const float hi = warp_max_f32(own ? mine : -CUDART_INF_F);
    float bmax = 1.f;
    DirectView view{map};
    const int which = clamp_case(view, wts, H, W, KS, lane, lo, hi, any_nan, ori_max, bmax);
    if (which == 2) return false;
    const float mylog = (which == 0) ? logf(mine) : exact_log(mine, ori_max, bmax);   // one log per lane
    float L[kStencil];
#pragma unroll
    for (int s = 0; s < kStencil; ++s) L[s] = __shfl_sync(SP_FULL, mylog, lane_of_slot(s));
    return taylor_step(L, ox, oy);
}

// ---------------------------------------------------------------------------------------------
// everything after the argmax: coordinates, refinement, affine, stores
// ---------------------------------------------------------------------------------------------
// trans_inv row of the map's person, fetched before the scan so its latency is off the critical path
struct Affine {
    float a, b, c, d, e, f;
};
__device__ __forceinline__ Affine load_affine(const DecodeArgs& A, int m) {
    Affine T;
    T.a = 1.f; T.b = 0.f; T.c = 0.f; T.d = 0.f; T.e = 1.f; T.f = 0.f;
    if (A.mode != SP_DECODE_ARGMAX && A.trans_inv != nullptr && m < A.nmaps) {
        const float* p = A.trans_inv + 6 * (size_t)(m / A.K);
        T.a = __ldg(p + 0); T.b = __ldg(p + 1); T.c = __ldg(p + 2);
        T.d = __ldg(p + 3); T.e = __ldg(p + 4); T.f = __ldg(p + 5);
    }
    return T;
}

template <typename View, typename Refine>
__device__ __forceinline__ void finish_map(const DecodeArgs& A, const View& map, int m, Peak pk, int lane,
                                           const Affine T, Refine&& refine) {
    const int W = A.W, H = A.H;
    const bool positive = pk.value > 0.f;                 // false for NaN, like (max_val > 0.)
    const int iy = positive ? pk.index / W : 0;
    const int ix = positive ? pk.index - iy * W : 0;
    float x = (float)ix, y = (float)iy;

    if (A.mode == SP_DECODE_GAUSS_TAYLOR || A.mode == SP_DECODE_DARK_ORIGINAL) {
        const bool inner = (ix > 1) && (ix < W - 2) && (iy > 1) && (iy < H - 2);
        if (inner) {
            float ox = 0.f, oy = 0.f;
            if (refine(ix, iy, pk.value, ox, oy)) {
                const float nx = __fadd_rn(x, ox), ny = __fadd_rn(y, oy);
                if (A.mode == SP_DECODE_GAUSS_TAYLOR) {
                    x = (nx < 0.f) ? 0.f : nx;            // clamp(min=0) that keeps NaN
                    y = (ny < 0.f) ? 0.f : ny;
                } else {                                  // DarkPoseOriginalKeyPointDecoder.taylor: coord += offset
                    x = nx;
                    y = ny;
                }
            }
        }
    } else if (A.mode == SP_DECODE_BASIC) {
        const bool inner = (ix > 1) && (ix < W - 1) && (iy > 1) && (iy < H - 1);
        if (inner) {
            const float ddx = __fsub_rn(map.at(iy * W + ix + 1), map.at(iy * W + ix - 1));
            const float ddy = __fsub_rn(map.at((iy + 1) * W + ix), map.at((iy - 1) * W + ix));
            const float sx = (ddx > 0.f) ? 1.f : (ddx < 0.f) ? -1.f : ddx;   // torch.sign (NaN stays NaN)
            const float sy = (ddy > 0.f) ? 1.f : (ddy < 0.f) ? -1.f : ddy;
            x = __fadd_rn(x, __fmul_rn(sx, 0.25f));
            y = __fadd_rn(y, __fmul_rn(sy, 0.25f));
        }
    }
    if (lane == 0) {
        float outx = x, outy = y;
        if (A.mode != SP_DECODE_ARGMAX && A.trans_inv != nullptr) {
            outx = __fadd_rn(fmaf(y, T.b, __fmul_rn(x, T.a)), T.c);
            outy = __fadd_rn(fmaf(y, T.e, __fmul_rn(x, T.d)), T.f);
        }
        if (A.coords) reinterpret_cast<float2*>(A.coords)[m] = make_float2(outx, outy);
        if (A.maxval) A.maxval[m] = pk.value;
        if (A.argmax) A.argmax[m] = pk.index;
        if (A.rows) {
            const int person = m / A.K;
            float* r = A.rows + (size_t)person * A.row_stride + 3 * (m - person * A.K);
            r[0] = outx; r[1] = outy; r[2] = pk.value;
        }
    }
}


}  // namespace sp_dec
