// Deterministic per-column sums of the shared-mode backward kernels (nearest agents, range scan, time to collision).
//
// Determinism: these kernels add no float atomically, so two calls give the same bits.  One CTA sums one environment,
// its columns (agents) in passes of up to kColsPerPass.  Each of the CTA's W warps owns a [cols][C] float accumulator
// in shared memory, zeroed per pass; a warp adds its rows' terms to it in an order fixed by the code (by row, and
// within a row lane after lane where several of the row's lanes may add to one column: add_lane_serial).  The W
// accumulators are then added in warp order, from 0.0f (total), and stored.
#pragma once
#include <cuda_runtime.h>

namespace tds {

constexpr int kColsPerPass = 512;

// The per-warp accumulators [W][cols][C] at `all` (8-byte aligned); `acc` is the calling warp's [cols][C].
template <int W, int C>
struct ColSums {
    float* all;
    int cols;
    float* acc;

    __device__ __forceinline__ ColSums(float* all, int cols, int warp) : all(all), cols(cols), acc(all + warp * cols * C) {
        // with C even every column starts 8-byte aligned, so the compiler may pair a kernel's adds to one column
        if constexpr (C % 2 == 0) acc = static_cast<float*>(__builtin_assume_aligned(acc, 8));
    }

    // zeroes the first nc columns of the warp's accumulator; called by all 32 lanes
    __device__ __forceinline__ void zero(int nc, int lane) const {
        for (int q = lane; q < C * nc; q += 32) acc[q] = 0.0f;
        __syncwarp();
    }

    // the sum over warps 0..W-1, in order, of component comp of column n (after a __syncthreads)
    __device__ __forceinline__ float total(int n, int comp) const {
        float v = 0.0f;
#pragma unroll
        for (int w = 0; w < W; w++) v += all[w * cols * C + n * C + comp];
        return v;
    }
};

// Adds the terms of every lane with a column, lane after lane (lowest first): the terms v[K * C] of source lane src are
// dealt to lanes 0..K*C-1, and lane c adds term c to component c % C of column col[c / C] of the pass that starts at
// column n0 (skipped if col[c / C] is -1).  Called by all 32 lanes; the K columns of one lane must be distinct.
template <int C, int K>
__device__ __forceinline__ void add_lane_serial(float* acc, int n0, const int (&col)[K], const float (&v)[K * C], int lane) {
    bool any = false;
#pragma unroll
    for (int k = 0; k < K; k++) any |= col[k] >= 0;
    for (unsigned todo = __ballot_sync(0xffffffffu, any); todo; todo &= todo - 1) {
        const int src = __ffs(todo) - 1;
        int sc[K];
#pragma unroll
        for (int k = 0; k < K; k++) sc[k] = __shfl_sync(0xffffffffu, col[k], src);
        float mine = 0.0f;
#pragma unroll
        for (int c = 0; c < K * C; c++) {
            const float x = __shfl_sync(0xffffffffu, v[c], src);
            if (lane == c) mine = x;
        }
#pragma unroll
        for (int k = 0; k < K; k++)
            if ((unsigned)(lane - k * C) < (unsigned)C && sc[k] >= 0) acc[(sc[k] - n0) * C + lane - k * C] += mine;
        __syncwarp();
    }
}

}  // namespace tds
