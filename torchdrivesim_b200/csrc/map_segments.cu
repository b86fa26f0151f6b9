// Map observations: the k nearest lane-marking segments of every agent, in the agent's frame (tds_nearest_map_segments)
// and the gradient of that observation with respect to the agent's pose (tds_nearest_map_segments_bwd).  The segments
// and their grid are built once per map by tds_map_create (map.cu, tds::SegDev).
#include <cstdint>

#include "tds_map.cuh"
#include "tds_nearest.cuh"

namespace {

using tds::kNearEmpty;
using tds::SegDev;
using tds::SegSetDev;

constexpr int kSegWarps = 8;                  // warps per CTA of both kernels (one warp per agent)

// The squared distance from (x, y) to the segment q = (x0, y0, x1, y1), every operation rounded on its own (the library
// builds with -fmad=false; `/` is the IEEE division).  The clamp keeps a NaN, as torch.clamp does.
__device__ __forceinline__ float seg_key(float x, float y, float4 q) {
    const float ex = q.z - q.x, ey = q.w - q.y, wx = x - q.x, wy = y - q.y;
    const float l2 = ex * ex + ey * ey;
    float t = 0.0f;
    if (l2 > 0.0f) {
        const float u = (wx * ex + wy * ey) / l2;
        t = u < 0.0f ? 0.0f : (u > 1.0f ? 1.0f : u);
    }
    const float qx = wx - t * ex, qy = wy - t * ey;
    return qx * qx + qy * qy;
}

// One warp per agent (b, a), searching the segment grid around the agent by tds::seg_grid_walk.  Eligible candidates
// are words (key bits << 32 | s), kept by tds::near_insert.  The search stops when the bound dmin - slack on the
// unsearched segments, lowered by more than the rounding of the float32 keys, exceeds the k-th key (a later segment
// cannot enter the list, nor tie with its key) or the distance limit, or when no cell is left.
template <int R>
__global__ void __launch_bounds__(kSegWarps * 32) nearest_map_segments_kernel(SegSetDev maps, const int32_t* __restrict__ env_map,
                                                                              const float* __restrict__ state, int64_t rows,
                                                                              int A, int k, float r2, float4* __restrict__ out,
                                                                              int64_t* __restrict__ kind,
                                                                              int64_t* __restrict__ idx) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kSegWarps + warp;
    if (row >= rows) return;                                       // warp-uniform
    const SegDev& m = maps.m[env_map ? env_map[row / A] : 0];
    const float x = state[row * 4], y = state[row * 4 + 1];
    unsigned long long list[R];
#pragma unroll
    for (int r = 0; r < R; r++) list[r] = kNearEmpty;
    const int last_r = (k - 1) >> 5, last_lane = (k - 1) & 31;
    unsigned long long thr = kNearEmpty;                           // the word in slot k - 1
    if (isfinite(x) && isfinite(y) && m.n > 0) {
        tds::seg_grid_walk(
            m, x, y, lane,
            [&](int j) {
                unsigned long long cand = kNearEmpty;
                if (j >= 0) {
                    const float key = seg_key(x, y, m.seg[j]);
                    if (key <= r2) cand = ((unsigned long long)__float_as_uint(key) << 32) | (unsigned)j;
                }
                tds::near_insert<R>(list, cand, thr, last_r, last_lane, lane);
            },
            [&](double dmin) {
                // a float32 key errs by far less than 1e-5 of the distance plus 1e-3 m
                const double lb = (dmin - m.slack) * (1.0 - 1e-5) - 1e-3;
                return lb > 0.0 && ((double)__uint_as_float((unsigned)(thr >> 32)) < lb * lb || lb * lb > (double)r2);
            });
    }
    // indices and kinds first, the rows after the heading's sincos (an ABI call): the list is not live across it
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int sl = r * 32 + lane;
        if (sl >= k) break;
        const int64_t e = row * k + sl;
        int64_t j = -1, kd = -1;
        if (list[r] != kNearEmpty) {
            j = (int)(unsigned)list[r];
            kd = m.kind[j];
        }
        kind[e] = kd;
        idx[e] = j;
    }
    float s, c;
    tds::sincos_cr(-state[row * 4 + 2], s, c);
    for (int sl = lane; sl < k; sl += 32) {
        const int64_t e = row * k + sl;
        const int64_t j = idx[e];
        float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (j >= 0) {
            const float4 q = m.seg[j];
            const float dx0 = q.x - x, dy0 = q.y - y, dx1 = q.z - x, dy1 = q.w - y;
            v = make_float4(c * dx0 + (-s) * dy0, s * dx0 + c * dy0, c * dx1 + (-s) * dy1, s * dx1 + c * dy1);
        }
        out[e] = v;
    }
}

// One warp per agent.  Per filled slot and endpoint, with (s, c) = sincos_cr(-psi), d = endpoint - xy, (rx, ry) the
// forward's values and upstream (g0, g1): d x -= c g0 + s g1, d y -= -s g0 + c g1, d psi += g0 ry - g1 rx.  A lane sums
// its slots in order, then a fixed shuffle tree sums the lanes: no atomics, two calls give the same bits.  A slot whose
// index is not a segment of the map is skipped by a branch, so NaN upstream values there do not reach the gradient.
__global__ void __launch_bounds__(kSegWarps * 32) nearest_map_segments_bwd_kernel(SegSetDev maps, const int32_t* __restrict__ env_map,
                                                                                  const float* __restrict__ state,
                                                                                  const int64_t* __restrict__ idx,
                                                                                  const float* __restrict__ gout, int64_t rows,
                                                                                  int A, int k, float* __restrict__ gstate) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kSegWarps + warp;
    if (row >= rows) return;                                       // warp-uniform
    const SegDev& m = maps.m[env_map ? env_map[row / A] : 0];
    const float x = state[row * 4], y = state[row * 4 + 1];
    float s, c;
    tds::sincos_cr(-state[row * 4 + 2], s, c);
    float px = 0.0f, py = 0.0f, pp = 0.0f;
    for (int sl = lane; sl < k; sl += 32) {
        const int64_t e = row * k + sl;
        const int64_t j = idx[e];
        if (j < 0 || j >= m.n) continue;                           // an empty slot
        const float4 q = m.seg[j];
        const float* g = gout + e * 4;
#pragma unroll
        for (int p = 0; p < 2; p++) {
            const float dx = (p ? q.z : q.x) - x, dy = (p ? q.w : q.y) - y;
            const float g0 = g[2 * p], g1 = g[2 * p + 1];
            const float rx = c * dx + (-s) * dy, ry = s * dx + c * dy;
            px += c * g0 + s * g1;
            py += (-s) * g0 + c * g1;
            pp += g0 * ry - g1 * rx;
        }
    }
    px = tds::warp_sum(px);
    py = tds::warp_sum(py);
    pp = tds::warp_sum(pp);
    if (lane == 0) {
        float* w = gstate + row * 4;
        w[0] = -px;
        w[1] = -py;
        w[2] = pp;
        w[3] = 0.0f;
    }
}

}  // namespace

extern "C" int tds_nearest_map_segments(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                                        const float* d_state, int32_t B, int32_t A, int32_t k, float r2, float* d_out,
                                        int64_t* d_kind, int64_t* d_idx, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0, "nearest_map_segments: negative size");
    TDS_REQUIRE(k >= 1 && k <= 256, "nearest_map_segments: need 1 <= k <= 256, got %d", k);
    TDS_REQUIRE(r2 >= 0.0f, "nearest_map_segments: need r2 >= 0");
    SegSetDev set;
    if (int e = tds::gather_segments(maps, n_maps, set)) return e;
    const int64_t rows = (int64_t)B * A, blocks = (rows + kSegWarps - 1) / kSegWarps;
    if (rows == 0) return TDS_OK;
    TDS_REQUIRE(d_state && d_out && d_kind && d_idx, "nearest_map_segments: null pointer");
    TDS_REQUIRE(((uintptr_t)d_out & 15) == 0, "nearest_map_segments: d_out must be 16-byte aligned");
    TDS_REQUIRE(blocks <= 2147483647LL, "nearest_map_segments: too many agents");
    float4* out = reinterpret_cast<float4*>(d_out);
    const cudaStream_t st = (cudaStream_t)stream;
    if (k <= 32)
        nearest_map_segments_kernel<1><<<(unsigned)blocks, kSegWarps * 32, 0, st>>>(set, d_env_map, d_state, rows, A, k, r2, out, d_kind, d_idx);
    else if (k <= 64)
        nearest_map_segments_kernel<2><<<(unsigned)blocks, kSegWarps * 32, 0, st>>>(set, d_env_map, d_state, rows, A, k, r2, out, d_kind, d_idx);
    else if (k <= 128)
        nearest_map_segments_kernel<4><<<(unsigned)blocks, kSegWarps * 32, 0, st>>>(set, d_env_map, d_state, rows, A, k, r2, out, d_kind, d_idx);
    else
        nearest_map_segments_kernel<8><<<(unsigned)blocks, kSegWarps * 32, 0, st>>>(set, d_env_map, d_state, rows, A, k, r2, out, d_kind, d_idx);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_nearest_map_segments_bwd(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                                            const float* d_state, const int64_t* d_idx, const float* d_grad_out, int32_t B,
                                            int32_t A, int32_t k, float* d_grad_state, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0, "nearest_map_segments_bwd: negative size");
    TDS_REQUIRE(k >= 1 && k <= 256, "nearest_map_segments_bwd: need 1 <= k <= 256, got %d", k);
    SegSetDev set;
    if (int e = tds::gather_segments(maps, n_maps, set)) return e;
    const int64_t rows = (int64_t)B * A, blocks = (rows + kSegWarps - 1) / kSegWarps;
    if (rows == 0) return TDS_OK;
    TDS_REQUIRE(d_state && d_idx && d_grad_out && d_grad_state, "nearest_map_segments_bwd: null pointer");
    TDS_REQUIRE(blocks <= 2147483647LL, "nearest_map_segments_bwd: too many agents");
    nearest_map_segments_bwd_kernel<<<(unsigned)blocks, kSegWarps * 32, 0, (cudaStream_t)stream>>>(
        set, d_env_map, d_state, d_idx, d_grad_out, rows, A, k, d_grad_state);
    TDS_LAUNCH_OK();
    return TDS_OK;
}
