// NumPy's float64 summation order on the device (np.sum / np.add.reduce / np.mean over a contiguous 1-D
// array), so that sums the reference computes with NumPy come out bit for bit: the OKS of the NMS (sp_oks.cu)
// and of COCOeval, the rescoring mean, and COCOeval's summary means (sp_coco_eval.cu).
#pragma once
#include <cuda_runtime.h>

namespace sp {

// NumPy's pairwise sum for n <= 128 fed one value at a time (numpy/core/src/umath/loops_utils:
// 8 running accumulators, tree-combined, then the n % 8 tail added in order; for n < 8 a plain
// running sum). The reduction starts from the identity: result = 0 + pairwise(values).
struct NumpySum {
    double r[8];
    double tail;
    int n_main, seen, n;
    __device__ void begin(int count) {
        n = count;
        n_main = (count < 8) ? 0 : count - (count % 8);
        seen = 0;
        tail = 0.0;
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = 0.0;
    }
    __device__ void push(double v) {
        if (seen < n_main) {
            const int j = seen & 7;
            // first round initialises the accumulator (r[j] = a[j]), later rounds add
            double cur = 0.0;
#pragma unroll
            for (int q = 0; q < 8; ++q) if (q == j) cur = r[q];
            cur = (seen < 8) ? v : __dadd_rn(cur, v);
#pragma unroll
            for (int q = 0; q < 8; ++q) if (q == j) r[q] = cur;
            if (seen + 1 == n_main)
                tail = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                                 __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
        } else {
            tail = __dadd_rn(tail, v);
        }
        ++seen;
    }
    __device__ double result() const { return __dadd_rn(0.0, tail); }
};

// The same sum over an array of any length: NumPy splits a block longer than 128 at n/2 rounded down to a
// multiple of 8 and adds the sums of the two halves; blocks of <= 128 are NumpySum's. `a` may be in any
// memory space. The split tree is walked with an explicit stack (depth <= 32 for any int n).
__device__ inline double numpy_sum_array(const double* a, int n) {
    int off[32], len[32];
    double part[32];
    unsigned char stage[32];
    int sp = 0;
    off[0] = 0;
    len[0] = n;
    stage[0] = 0;
    double ret = 0.0;
    while (sp >= 0) {
        const int o = off[sp], m = len[sp];
        if (m <= 128) {
            NumpySum acc;
            acc.begin(m);
            for (int i = 0; i < m; ++i) acc.push(a[o + i]);
            ret = acc.tail;                        // a block's own sum, without the reduction's identity
        } else if (stage[sp] == 0) {               // descend into the left half
            int h = m / 2;
            h -= h % 8;
            stage[sp] = 1;
            off[sp + 1] = o;
            len[sp + 1] = h;
            stage[sp + 1] = 0;
            ++sp;
            continue;
        } else if (stage[sp] == 1) {               // left half done: descend into the right half
            int h = m / 2;
            h -= h % 8;
            part[sp] = ret;
            stage[sp] = 2;
            off[sp + 1] = o + h;
            len[sp + 1] = m - h;
            stage[sp + 1] = 0;
            ++sp;
            continue;
        } else {
            ret = __dadd_rn(part[sp], ret);
        }
        --sp;
    }
    return __dadd_rn(0.0, ret);
}

}  // namespace sp
