// Range-scan observations: the distance along R rays of every agent to the first agent box edge or lane-marking
// segment (tds_range_scan), and the gradient of the distances with respect to the agents' poses and sizes
// (tds_range_scan_bwd).  The markings and their grid are built once per map by tds_map_create (map.cu, tds::SegDev).
//
// Hit test of ray (o, d) and segment (p0, p1), float32, every operation rounded on its own (-fmad=false), IEEE division:
//   e = p1 - p0, w = p0 - o, den = dx*ey - dy*ex;  den == 0: no hit;
//   t = (wx*ey - wy*ex) / den, u = (wx*dy - wy*dx) / den;  hit iff 0 <= u <= 1 and 0 <= t <= max_range.
// The best hit of a ray is the smallest word (bits(t) << 32 | code): t >= 0 orders like its bits once -0 is made +0.
// Codes: 4 j + k for edge k of agent j, 4 N + s for marking s.
#include <math_constants.h>

#include <algorithm>
#include <cmath>
#include <cstdint>

#include "tds_colsum.cuh"
#include "tds_map.cuh"
#include "tds_nearest.cuh"

namespace {

using tds::kNearEmpty;
using tds::SegDev;
using tds::SegSetDev;

constexpr int kScanWarps = 8;            // warps per CTA of the forward (one warp per origin)
constexpr int kScanCacheAgents = 1024;   // the forward caches an environment's box corners (32 B per agent) up to this N
constexpr float kTwoPi = 6.28318530717958647692f;

// (float32 of cospi(2r/R), float32 of sinpi(2r/R)): ray r in the agent's frame, exact axis vectors at quarter turns.
__device__ __forceinline__ float2 ray_unit(int r, int R) {
    double s, c;
    sincospi((double)(2 * r) / (double)R, &s, &c);
    return make_float2((float)c, (float)s);
}

// d = (c ux - s uy, s ux + c uy): the ray in the world frame.
__device__ __forceinline__ float2 ray_world(float2 u, float s, float c) {
    return make_float2(c * u.x - s * u.y, s * u.x + c * u.y);
}

// The word of a hit of ray d on the segment with e = p1 - p0, w = p0 - o, or kNearEmpty.  NaN fails every comparison.
__device__ __forceinline__ unsigned long long hit_word(float dx, float dy, float ex, float ey, float wx, float wy,
                                                       float max_range, unsigned code) {
    const float den = dx * ey - dy * ex;
    if (den == 0.0f) return kNearEmpty;
    float t = (wx * ey - wy * ex) / den;
    const float u = (wx * dy - wy * dx) / den;
    if (!(u >= 0.0f && u <= 1.0f && t >= 0.0f && t <= max_range)) return kNearEmpty;
    if (t == 0.0f) t = 0.0f;                                       // -0 -> +0
    return ((unsigned long long)__float_as_uint(t) << 32) | code;
}

// Rounding margin of every distance bound below: a float32 t of a ray at a grazing angle to a far segment can be off
// by more than a float32 key of the map-segment kernel (the division by den amplifies the rounding of w and e), so the
// bounds here are lowered by 1e-3 of themselves and 5 cm.  A hit can only be missed if its t errs by more than that.
__device__ __forceinline__ double lower_bound(double d) { return d * (1.0 - 1e-3) - 0.05; }

// Tests one candidate segment (p0, p1) against the rays of one origin and keeps the best word of each ray in `best`.
// The rays tested are those inside the segment's angular interval as seen from o, widened by one ray spacing on each
// side (2 pi / R >= 0.0245 rad, far more than the float32 error of the angles and of the hit test near the interval's
// ends), or every ray when the segment is near the origin: an endpoint on it, endpoints at distances more than 64x
// apart, or an interval wider than 2.5 rad (where the sign of the cross product, hence the side of the interval, is
// beyond doubt).  A segment with a non-finite coordinate cannot hit (every case ends in a NaN or an infinite u or t),
// nor one further from o than max_range by the margin.
__device__ __forceinline__ void scan_segment(float ox, float oy, float4 p, unsigned code, float max_range, double range_lb2,
                                             float apsi, int R, const float2* __restrict__ dirs,
                                             unsigned long long* __restrict__ best) {
    if (!(isfinite(p.x) && isfinite(p.y) && isfinite(p.z) && isfinite(p.w))) return;
    const float ex = p.z - p.x, ey = p.w - p.y, wx = p.x - ox, wy = p.y - oy;
    const float w1x = p.z - ox, w1y = p.w - oy;
    {   // distance from o to the segment, in double: exact enough for any float inputs
        const double dex = (double)p.z - p.x, dey = (double)p.w - p.y, dwx = (double)ox - p.x, dwy = (double)oy - p.y;
        const double l2 = dex * dex + dey * dey;
        double tt = l2 > 0.0 ? (dwx * dex + dwy * dey) / l2 : 0.0;
        tt = fmin(fmax(tt, 0.0), 1.0);
        const double qx = dwx - tt * dex, qy = dwy - tt * dey;
        if (qx * qx + qy * qy > range_lb2) return;
    }
    int first = 0, count = R;
    const float n0 = wx * wx + wy * wy, n1 = w1x * w1x + w1y * w1y;
    const float cr = wx * w1y - wy * w1x, dt = wx * w1x + wy * w1y;
    if (isfinite(ex) && isfinite(ey) && isfinite(wx) && isfinite(wy) && isfinite(w1x) && isfinite(w1y) && isfinite(n0) &&
        isfinite(n1) && n0 > 0.0f && n1 > 0.0f && n0 <= 4096.0f * n1 && n1 <= 4096.0f * n0 && isfinite(cr) && isfinite(dt)) {
        const float arc = atan2f(fabsf(cr), dt);
        if (arc <= 2.5f) {
            const float a = (cr >= 0.0f ? atan2f(wy, wx) : atan2f(w1y, w1x)) - apsi;   // in (-2 pi, 2 pi)
            const float scale = (float)R / kTwoPi;
            const int lo = (int)floorf(a * scale) - 1;
            const int n = (int)ceilf(arc * scale) + 4;
            if (n < R) {
                first = ((lo % R) + R) % R;
                count = n;
            }
        }
    }
    for (int q = 0; q < count; q++) {
        int r = first + q;
        if (r >= R) r -= R;
        const float2 d = dirs[r];
        const unsigned long long wd = hit_word(d.x, d.y, ex, ey, wx, wy, max_range, code);
        if (wd < best[r]) atomicMin(best + r, wd);
    }
}

// Forward: one warp per origin row (b, i), kScanWarps per CTA.  Shared memory: the ray units u_r of the CTA, and per
// warp the world directions d_r and the best word of each ray (64-bit atomicMin: the minimum does not depend on the
// order of the candidates, so the result is deterministic).  When the CTA's rows belong to one environment and N <=
// kScanCacheAgents, the environment's box corners are computed once into shared memory (NaN for an absent agent, which
// then never hits).  The lanes take 32 candidates at a time: first the 4 N box edges, then the markings, walking the
// segment grid by tds::seg_grid_walk.  After a ring the search stops when the unsearched cells lie beyond max_range or
// beyond the t of every ray (by lower_bound), or when no cell is left.
__global__ void __launch_bounds__(kScanWarps * 32) range_scan_kernel(SegSetDev maps, int use_map,
                                                                     const int32_t* __restrict__ env_map,
                                                                     const float* __restrict__ absolute, int64_t rows,
                                                                     int A, int N, int R, float max_range,
                                                                     float* __restrict__ dist, int64_t* __restrict__ kind,
                                                                     int64_t* __restrict__ idx) {
    extern __shared__ unsigned long long s_scan[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned long long* best = s_scan + warp * R;                 // [kScanWarps][R]
    float2* units = reinterpret_cast<float2*>(s_scan + kScanWarps * R);       // [R]
    float2* dirs = units + R + warp * R;                           // [kScanWarps][R]
    float2* corners = units + R + kScanWarps * R;                  // [N][4] when cached
    const int64_t row0 = (int64_t)blockIdx.x * kScanWarps;
    const int64_t b0 = row0 / A;
    const bool cached = N <= kScanCacheAgents && b0 == (min(row0 + kScanWarps, rows) - 1) / A;  // CTA-uniform
    for (int r = threadIdx.x; r < R; r += blockDim.x) units[r] = ray_unit(r, R);
    if (cached) {
        const float* env = absolute + b0 * N * 6;
        for (int q = threadIdx.x; q < 4 * N; q += blockDim.x) {
            const float* a = env + (int64_t)(q >> 2) * 6;
            float2 v = make_float2(CUDART_NAN_F, CUDART_NAN_F);
            if (a[5] != 0.0f) {
                float s, c;
                tds::sincos_cr(a[2], s, c);
                tds::box_corner(a[0], a[1], a[3], a[4], s, c, q & 3, v.x, v.y);
            }
            corners[q] = v;
        }
    }
    __syncthreads();
    const int64_t row = row0 + warp;
    if (row >= rows) return;                                       // warp-uniform
    const int64_t b = row / A;
    const int i = (int)(row - b * A);
    const float* env = absolute + b * N * 6;
    const float ox = env[(int64_t)i * 6], oy = env[(int64_t)i * 6 + 1], psi = env[(int64_t)i * 6 + 2];
    for (int r = lane; r < R; r += 32) best[r] = kNearEmpty;
    if (isfinite(ox) && isfinite(oy) && isfinite(psi)) {
        float s, c;
        tds::sincos_cr(psi, s, c);
        const float apsi = atan2f(s, c);
        for (int r = lane; r < R; r += 32) dirs[r] = ray_world(units[r], s, c);
        const double lb = (double)max_range + 0.05;
        const double range_lb2 = (lb / (1.0 - 1e-3)) * (lb / (1.0 - 1e-3));   // lower_bound(dist) > max_range beyond it
        __syncwarp();
        for (int q0 = 0; q0 < 4 * N; q0 += 32) {                   // the box edges
            const int q = q0 + lane;
            const int j = q >> 2;
            if (q < 4 * N && j != i) {
                const int k = q & 3, k1 = (k + 1) & 3;
                float4 p;
                if (cached) {
                    const float2 c0 = corners[q], c1 = corners[(q & ~3) + k1];
                    p = make_float4(c0.x, c0.y, c1.x, c1.y);
                } else {
                    const float* a = env + (int64_t)j * 6;
                    p = make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F);
                    if (a[5] != 0.0f) {
                        float sj, cj;
                        tds::sincos_cr(a[2], sj, cj);
                        tds::box_corner(a[0], a[1], a[3], a[4], sj, cj, k, p.x, p.y);
                        tds::box_corner(a[0], a[1], a[3], a[4], sj, cj, k1, p.z, p.w);
                    }
                }
                scan_segment(ox, oy, p, (unsigned)q, max_range, range_lb2, apsi, R, dirs, best);
            }
        }
        const SegDev& m = maps.m[env_map ? env_map[b] : 0];
        if (use_map && m.n > 0) {
            const unsigned base = 4u * (unsigned)N;
            tds::seg_grid_walk(
                m, ox, oy, lane,
                [&](int sg) {
                    if (sg >= 0)
                        scan_segment(ox, oy, m.seg[sg], base + (unsigned)sg, max_range, range_lb2, apsi, R, dirs, best);
                },
                [&](double dmin) {
                    const double lbd = lower_bound(dmin - m.slack);
                    if (lbd > (double)max_range) return true;
                    if (lbd > 0.0) {
                        __syncwarp();
                        unsigned top = 0;                          // the largest t bits of the rays (no hit: NaN bits)
                        for (int r = lane; r < R; r += 32) top = max(top, (unsigned)(best[r] >> 32));
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) top = max(top, __shfl_xor_sync(0xffffffffu, top, o));
                        if (lbd > (double)__uint_as_float(top)) return true;  // false for NaN
                    }
                    return false;
                });
        }
    }
    __syncwarp();
    for (int r = lane; r < R; r += 32) {
        const unsigned long long wd = best[r];
        const int64_t e = row * R + r;
        if (wd == kNearEmpty) {
            dist[e] = max_range;
            kind[e] = -1;
            idx[e] = -1;
        } else {
            const unsigned code = (unsigned)wd;
            dist[e] = __uint_as_float((unsigned)(wd >> 32));
            const bool agent = code < 4u * (unsigned)N;
            kind[e] = agent ? 0 : 1;
            idx[e] = agent ? (int64_t)(code >> 2) : (int64_t)(code - 4u * (unsigned)N);
        }
    }
}

// Backward: one CTA per environment, a tds::ColSums column sum (tds_colsum.cuh) over (x, y, psi, length, width).  Each
// warp takes origin rows i = warp, warp + 8, ...; its lanes take the row's rays.  A ray's winner is recomputed from
// kind and idx; with q = g / den:
//   origin:        d x += -ey q,  d y += ex q,  d psi += t (d . e) q;
//   edge (p0, p1): d p0 += (1 - u) (ey q, -ex q),  d p1 += u (ey q, -ex q),
// and a corner's gradient (gx, gy) reaches its agent as d x += gx, d y += gy, d psi += -gx ry + gy rx ((rx, ry) the
// rotated half-extents), d length += sx (gx c + gy s), d width += sy (-gx s + gy c).  The agent terms of the rays are
// added to the accumulator by tds::add_lane_serial (several rays may hit one agent); the origin terms are summed per
// lane over its rays and then by a shuffle tree, and added to column i after the row.  The output's present column
// gets 0.  A ray whose kind / idx is not a hit of this row (no hit, an agent index out of range or i itself, a
// marking index out of range) is skipped by a branch, so a NaN upstream value there does not reach the gradient.
__global__ void __launch_bounds__(kScanWarps * 32) range_scan_bwd_kernel(SegSetDev maps, int use_map,
                                                                         const int32_t* __restrict__ env_map,
                                                                         const float* __restrict__ absolute,
                                                                         const int64_t* __restrict__ kind,
                                                                         const int64_t* __restrict__ idx,
                                                                         const float* __restrict__ gout, int A, int N,
                                                                         int R, int cols, float* __restrict__ gabs) {
    extern __shared__ float s_bwd[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t b = blockIdx.x;
    float2* units = reinterpret_cast<float2*>(s_bwd);              // [R]
    const tds::ColSums<kScanWarps, 5> sums(s_bwd + 2 * R, cols, warp);
    for (int r = threadIdx.x; r < R; r += blockDim.x) units[r] = ray_unit(r, R);
    const float* ab = absolute + b * N * 6;
    float* gw = gabs + b * N * 6;
    const SegDev& m = maps.m[env_map ? env_map[b] : 0];
    const int n_seg = use_map ? m.n : 0;
    __syncthreads();
    for (int n0 = 0; n0 < N; n0 += cols) {
        const int nc = min(cols, N - n0);
        sums.zero(nc, lane);
        for (int i = warp; i < A; i += kScanWarps) {
            const bool own = i >= n0 && i < n0 + nc;               // warp-uniform: the origin's column is in this pass
            const float* o = ab + (int64_t)i * 6;
            const float ox = o[0], oy = o[1];
            float s, c;
            tds::sincos_cr(o[2], s, c);
            float px = 0.0f, py = 0.0f, pp = 0.0f;
            for (int r0 = 0; r0 < R; r0 += 32) {
                const int r = r0 + lane;
                const int64_t e = ((int64_t)b * A + i) * R + r;
                int j[1] = {-1};                                   // the hit agent, when its column is in this pass
                float v[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
                if (r < R) {
                    const int64_t kd = kind[e], id = idx[e];
                    const bool agent = kd == 0 && id >= 0 && id < N && id != i;
                    const bool mark = kd == 1 && id >= 0 && id < n_seg;
                    const bool col = agent && id >= n0 && id < n0 + nc;
                    if (col || ((agent || mark) && own)) {
                        const float2 d = ray_world(units[r], s, c);
                        float4 p;
                        float sj = 0.0f, cj = 0.0f;
                        int k = 0;
                        const float* a = ab + id * 6;
                        if (agent) {
                            // the winning edge: recompute the 4 edges' words, as the forward compares them
                            tds::sincos_cr(a[2], sj, cj);
                            unsigned long long bw = kNearEmpty;
                            float cxs[4], cys[4];
#pragma unroll
                            for (int kk = 0; kk < 4; kk++) tds::box_corner(a[0], a[1], a[3], a[4], sj, cj, kk, cxs[kk], cys[kk]);
#pragma unroll
                            for (int kk = 0; kk < 4; kk++) {
                                const int k1 = (kk + 1) & 3;
                                const unsigned long long wd = hit_word(d.x, d.y, cxs[k1] - cxs[kk], cys[k1] - cys[kk],
                                                                       cxs[kk] - ox, cys[kk] - oy, CUDART_INF_F, kk);
                                if (wd < bw) {
                                    bw = wd;
                                    k = kk;
                                }
                            }
                            p = make_float4(cxs[k], cys[k], cxs[(k + 1) & 3], cys[(k + 1) & 3]);
                        } else {
                            p = m.seg[id];
                        }
                        const float ex = p.z - p.x, ey = p.w - p.y, wx = p.x - ox, wy = p.y - oy;
                        const float den = d.x * ey - d.y * ex;
                        const float t = (wx * ey - wy * ex) / den;
                        const float u = (wx * d.y - wy * d.x) / den;
                        const float q = gout[e] / den;
                        if (own) {
                            px += -(ey * q);
                            py += ex * q;
                            pp += (t * (d.x * ex + d.y * ey)) * q;
                        }
                        if (col) {
                            j[0] = (int)id;
                            const float gx = ey * q, gy = -(ex * q);
                            const float sx0 = (k == 0 || k == 3) ? 0.5f : -0.5f, sy0 = k < 2 ? 0.5f : -0.5f;
                            const int k1 = (k + 1) & 3;
                            const float sx1 = (k1 == 0 || k1 == 3) ? 0.5f : -0.5f, sy1 = k1 < 2 ? 0.5f : -0.5f;
                            const float w0 = 1.0f - u;
                            const float g0x = w0 * gx, g0y = w0 * gy, g1x = u * gx, g1y = u * gy;
                            // the rotated half-extents of the two corners, as box_corner forms them
                            const float ux0 = sx0 * a[3], uy0 = sy0 * a[4], ux1 = sx1 * a[3], uy1 = sy1 * a[4];
                            const float rx0 = ux0 * cj + uy0 * (-sj), ry0 = ux0 * sj + uy0 * cj;
                            const float rx1 = ux1 * cj + uy1 * (-sj), ry1 = ux1 * sj + uy1 * cj;
                            v[0] = g0x + g1x;
                            v[1] = g0y + g1y;
                            v[2] = (g0y * rx0 - g0x * ry0) + (g1y * rx1 - g1x * ry1);
                            v[3] = sx0 * (g0x * cj + g0y * sj) + sx1 * (g1x * cj + g1y * sj);
                            v[4] = sy0 * (g0y * cj - g0x * sj) + sy1 * (g1y * cj - g1x * sj);
                        }
                    }
                }
                tds::add_lane_serial<5, 1>(sums.acc, n0, j, v, lane);
            }
            if (own) {
                px = tds::warp_sum(px);
                py = tds::warp_sum(py);
                pp = tds::warp_sum(pp);
                if (lane == 0) {
                    float* a = sums.acc + (i - n0) * 5;
                    a[0] += px;
                    a[1] += py;
                    a[2] += pp;
                }
            }
            __syncwarp();
        }
        __syncthreads();
        for (int q = threadIdx.x; q < 6 * nc; q += blockDim.x) {   // coalesced: the pass's columns x 6 values
            const int n = q / 6, comp = q - n * 6;
            gw[(int64_t)n0 * 6 + q] = comp < 5 ? sums.total(n, comp) : 0.0f;
        }
        __syncthreads();
    }
}

}  // namespace

extern "C" int tds_range_scan(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                              const float* d_absolute, int32_t B, int32_t A, int32_t N, int32_t R, float max_range,
                              float* d_dist, int64_t* d_kind, int64_t* d_idx, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "range_scan: need 0 <= A <= N");
    TDS_REQUIRE(N <= (1 << 28), "range_scan: at most 2^28 agents per environment");
    TDS_REQUIRE(R >= 1 && R <= 256, "range_scan: need 1 <= R <= 256, got %d", R);
    TDS_REQUIRE(std::isfinite(max_range) && max_range > 0.0f, "range_scan: max_range must be finite and > 0");
    SegSetDev set = {};
    if (n_maps > 0) {
        if (int e = tds::gather_segments(maps, n_maps, set)) return e;
    }
    const int64_t rows = (int64_t)B * A, blocks = (rows + kScanWarps - 1) / kScanWarps;
    if (rows == 0) return TDS_OK;
    TDS_REQUIRE(d_absolute && d_dist && d_kind && d_idx, "range_scan: null pointer");
    TDS_REQUIRE(blocks <= 2147483647LL, "range_scan: too many agents");
    const size_t smem = (size_t)kScanWarps * R * 8 + (size_t)R * 8 + (size_t)kScanWarps * R * 8 +
                        (N <= kScanCacheAgents ? (size_t)N * 32 : 0);
    if (int e = tds::allow_dynamic_smem(range_scan_kernel, smem)) return e;
    range_scan_kernel<<<(unsigned)blocks, kScanWarps * 32, smem, (cudaStream_t)stream>>>(
        set, n_maps > 0 ? 1 : 0, n_maps > 0 ? d_env_map : nullptr, d_absolute, rows, A, N, R, max_range, d_dist, d_kind,
        d_idx);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_range_scan_bwd(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                                  const float* d_absolute, const int64_t* d_kind, const int64_t* d_idx,
                                  const float* d_grad_dist, int32_t B, int32_t A, int32_t N, int32_t R,
                                  float* d_grad_absolute, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "range_scan_bwd: need 0 <= A <= N");
    TDS_REQUIRE(R >= 1 && R <= 256, "range_scan_bwd: need 1 <= R <= 256, got %d", R);
    SegSetDev set = {};
    if (n_maps > 0) {
        if (int e = tds::gather_segments(maps, n_maps, set)) return e;
    }
    if ((int64_t)B * N == 0) return TDS_OK;
    TDS_REQUIRE(d_absolute && d_grad_absolute && (A == 0 || (d_kind && d_idx && d_grad_dist)), "range_scan_bwd: null pointer");
    const int cols = std::min(N, tds::kColsPerPass);
    const size_t smem = (size_t)R * 8 + (size_t)kScanWarps * cols * 5 * sizeof(float);
    if (int e = tds::allow_dynamic_smem(range_scan_bwd_kernel, smem)) return e;
    range_scan_bwd_kernel<<<(unsigned)B, kScanWarps * 32, smem, (cudaStream_t)stream>>>(
        set, n_maps > 0 ? 1 : 0, n_maps > 0 ? d_env_map : nullptr, d_absolute, d_kind, d_idx, d_grad_dist, A, N, R, cols,
        d_grad_absolute);
    TDS_LAUNCH_OK();
    return TDS_OK;
}
