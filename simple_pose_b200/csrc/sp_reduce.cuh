// Deterministic grid-wide sum of per-block float64 partials into one float32 loss value, in a
// single launch: every block parks its partial in the caller's workspace, takes a ticket, and
// the last block to arrive adds all partials in a fixed order. No floating-point atomics.
#pragma once
#include "sp_common.cuh"

namespace sp_reduce {

constexpr int kMaxPartials = 4096;

struct MseWorkspace {
    unsigned int ticket;          // blocks finished so far (returns to 0 at the end of a call)
    unsigned int next_work;       // grid-wide work counter of kernels that deal work dynamically (returns to 0 likewise)
    unsigned int pad[2];
    double partial[kMaxPartials];
};

// Called by ALL threads of every block (gridDim.x <= kMaxPartials, blockDim.x <= THREADS, a multiple
// of 32). loss = 0.5 * total * inv_count. Returns true in every thread of the last block, which has acquired the
// writes every block made before its call.
template <int THREADS>
__device__ __forceinline__ bool finish_loss(double block_sum, MseWorkspace* __restrict__ ws, float* __restrict__ loss,
                                            double inv_count) {
    __shared__ double warp_part[THREADS / 32];
    __shared__ bool am_last;
    block_sum = sp::warp_sum(block_sum);
    if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = block_sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += warp_part[w];
        ws->partial[blockIdx.x] = s;
        __threadfence();
        const unsigned int t = atomicAdd(&ws->ticket, 1u);
        am_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!am_last) return false;
    // last block: add the partials in index order (thread-strided, then a fixed tree)
    __threadfence();
    double s = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) s += __ldcg(&ws->partial[i]);
    s = sp::warp_sum(s);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += warp_part[w];
        *loss = (float)(0.5 * tot * inv_count);
        ws->ticket = 0u;      // restore the zero state for the next call on this stream
        ws->next_work = 0u;
    }
    return true;
}

}  // namespace sp_reduce
