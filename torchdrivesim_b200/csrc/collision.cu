// Pairwise oriented-box collision metrics.
//
// discs : TrafficSim disc approximation, collision_detection_with_discs + bbox2discs
//         (torchdrivesim/infractions.py:503-545, 378-409), forward and backward.
// iou   : rotated-box IoU, iou_differentiable_fast (torchdrivesim/_iou_utils.py:344-367), forward.
//         The reference finds the intersection polygon by sorting 24 candidate vertices by angle
//         in world coordinates; in fp32 that is chaotic on the diagonal (SURVEY.md App. C-8).
//         Here box 2 is moved into the frame of box 1 and clipped against an axis-aligned
//         rectangle (Sutherland-Hodgman), which computes the same area and agrees with the
//         reference evaluated in float64 to ~1e-7.
// all-pairs: Simulator.compute_collision (torchdrivesim/simulator.py:1161-1194, 1064-1109):
//         out[b,i] = sum_j o_ij m_j - max_j o_ij m_j, one warp per row i, lanes over columns j,
//         warp-shuffle reductions; per-environment box data staged in shared memory.
// This work is FP32-pipe bound (no HBM traffic to speak of: 20 B per box in, 4 B per row out).
#include <cooperative_groups.h>
#include <math_constants.h>

#include "tds_colsum.cuh"
#include "tds_common.cuh"
#include "tds_nearest.cuh"

namespace {

constexpr int kDiscs = 5;

struct Discs {
    float cx[kDiscs], cy[kDiscs];
    float r;        // disc radius = min(l, w) / 2
    float half;     // max(l, w) / 2   (bounding radius along the major axis)
    float x, y;     // box centre
};

// bbox2discs, infractions.py:378-409 (nan_to_num of the box as in simulator.py:1095-1096)
__device__ __forceinline__ Discs make_discs(float x, float y, float l, float w, float psi) {
    Discs d;
    if (x != x) x = 0.f;
    if (y != y) y = 0.f;
    if (l != l) l = 0.f;
    if (w != w) w = 0.f;
    if (psi != psi) psi = 0.f;
    d.x = x; d.y = y;
    d.r = fminf(l, w) / 2.0f;
    d.half = fmaxf(l, w) / 2.0f;
    const float span = d.half - d.r;
    const float yaw = psi + 1.5707963705062866f * (w > l ? 1.0f : 0.0f);   // float32(pi/2)
    float s, c;
    tds::sincos_cr(yaw, s, c);
#pragma unroll
    for (int i = 0; i < kDiscs; i++) {
        const float off = ((float)(i - 2) * span) / 2.0f;
        d.cx[i] = off * c + x;
        d.cy[i] = off * s + y;
    }
    return d;
}

// overlap in [0,1]; amin/bmin receive the argmin disc pair (first in row-major order), dmin the distance
__device__ __forceinline__ float discs_overlap(const Discs& p, const Discs& q, int* amin, int* bmin, float* dmin) {
    float best = CUDART_INF_F;
    int ba = 0, bb = 0;
#pragma unroll
    for (int a = 0; a < kDiscs; a++) {
#pragma unroll
        for (int b = 0; b < kDiscs; b++) {
            const float dx = p.cx[a] - q.cx[b], dy = p.cy[a] - q.cy[b];
            const float d2 = dx * dx + dy * dy;
            if (d2 < best) { best = d2; ba = a; bb = b; }
        }
    }
    const float d = sqrtf(best);
    if (amin) { *amin = ba; *bmin = bb; *dmin = d; }
    float o = 1.0f - d / (p.r + q.r);
    o = o > 0.0f ? o : 0.0f;         // relu; NaN (0/0 for zero-size boxes) compares false -> 0, as nan_to_num
    return o;
}

// ---------------------------------------------------------------- IoU
struct Box {
    float x, y, l, w, s, c;   // s, c = sin/cos(psi)
};

__device__ __forceinline__ Box make_box(float x, float y, float l, float w, float psi) {
    Box b;
    if (x != x) x = 0.f;
    if (y != y) y = 0.f;
    if (l != l) l = 0.f;
    if (w != w) w = 0.f;
    if (psi != psi) psi = 0.f;
    b.x = x; b.y = y; b.l = l; b.w = w;
    tds::sincos_cr(psi, b.s, b.c);
    return b;
}

// clip polygon (px,py,n) against  sign*coord <= bound  (coord = x if axis==0 else y)
__device__ __forceinline__ int clip_axis(const float* px, const float* py, int n, float* qx, float* qy, int axis,
                                         float sign, float bound) {
    int m = 0;
    for (int i = 0; i < n; i++) {
        const int j = (i + 1 == n) ? 0 : i + 1;
        const float ax = px[i], ay = py[i], bx = px[j], by = py[j];
        const float da = sign * (axis ? ay : ax) - bound;
        const float db = sign * (axis ? by : bx) - bound;
        const bool ina = da <= 0.0f, inb = db <= 0.0f;
        if (ina) { qx[m] = ax; qy[m] = ay; m++; }
        if (ina != inb) {
            const float t = da / (da - db);
            qx[m] = ax + t * (bx - ax);
            qy[m] = ay + t * (by - ay);
            m++;
        }
    }
    return m;
}

// intersection area of two oriented boxes: q is clipped against p in p's frame (Sutherland-Hodgman)
__device__ float inter_area(const Box& p, const Box& q) {
    // bounding-circle early out: exact 0 in the reference for disjoint boxes
    const float dx = q.x - p.x, dy = q.y - p.y;
    const float rp = 0.5f * sqrtf(p.l * p.l + p.w * p.w), rq = 0.5f * sqrtf(q.l * q.l + q.w * q.w);
    const float reach = rp + rq;
    if (dx * dx + dy * dy > reach * reach * 1.0001f + 1e-6f) return 0.0f;
    // box q in the frame of box p: rotate by -psi_p
    const float cr = p.c * q.c + p.s * q.s;       // cos(psi_q - psi_p)
    const float sr = p.c * q.s - p.s * q.c;       // sin(psi_q - psi_p)
    const float tx = p.c * dx + p.s * dy;
    const float ty = p.c * dy - p.s * dx;
    const float hx = 0.5f * q.l, hy = 0.5f * q.w;
    float px[10], py[10], qx[10], qy[10];
    const float sx[4] = {1.f, -1.f, -1.f, 1.f}, sy[4] = {1.f, 1.f, -1.f, -1.f};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float ux = sx[k] * hx, uy = sy[k] * hy;
        px[k] = tx + (ux * cr - uy * sr);
        py[k] = ty + (ux * sr + uy * cr);
    }
    const float bx = 0.5f * p.l, by = 0.5f * p.w;
    int n = 4;
    n = clip_axis(px, py, n, qx, qy, 0, 1.f, bx);
    n = clip_axis(qx, qy, n, px, py, 0, -1.f, bx);
    n = clip_axis(px, py, n, qx, qy, 1, 1.f, by);
    n = clip_axis(qx, qy, n, px, py, 1, -1.f, by);
    if (n < 3) return 0.0f;
    float tot = 0.0f;
    for (int i = 0; i < n; i++) {
        const int j = (i + 1 == n) ? 0 : i + 1;
        tot += px[i] * py[j] - py[i] * px[j];
    }
    return 0.5f * fabsf(tot);
}

__device__ float iou_pair(const Box& p, const Box& q) {
    const float a1 = p.l * p.w, a2 = q.l * q.w;
    const float inter = inter_area(p, q);
    if (inter == 0.0f) return 0.0f;
    const float iou = inter / (a1 + a2 - inter);
    return iou == iou ? iou : 0.0f;               // nan_to_num, simulator.py:1103
}

// ---- traffic-light violations (TrafficLightControl.compute_violation, traffic_controls.py:152-178): an agent
// violates iff some RED light's stop-line rectangle overlaps, with positive area, the rear `rear_factor` part of
// the agent's box (box2corners_with_rear_factor, _iou_utils.py:302-341).  One thread per agent, L lights each.
__global__ void __launch_bounds__(128) tl_violation_kernel(const float* __restrict__ agent_box, const float* __restrict__ tl_corners,
                                                           const int32_t* __restrict__ tl_state, const uint8_t* __restrict__ present,
                                                           int B, int A, int L, int red, float rear, uint8_t* __restrict__ out) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (int64_t)B * A) return;
    const int b = (int)(g / A);
    const float* ab = agent_box + g * 5;
    Box p = make_box(ab[0], ab[1], ab[2], ab[3], ab[4]);
    const float shift = (p.l * (1.0f - rear)) / 2.0f;          // centre of the rear part, along the heading
    p.x = p.x - shift * p.c;
    p.y = p.y - shift * p.s;
    p.l = p.l * rear;
    bool hit = false;
    if (!present || present[g]) {
        for (int l = 0; l < L && !hit; l++) {
            if (tl_state[(int64_t)b * L + l] != red) continue;
            // stop-line rectangle from its corners (+,+), (-,+), (-,-), (+,-)  (box2corners_th)
            const float* c = tl_corners + ((int64_t)b * L + l) * 8;
            const float ex = c[0] - c[2], ey = c[1] - c[3];        // corner0 - corner1 = length * (cos, sin)
            const float fx = c[0] - c[6], fy = c[1] - c[7];        // corner0 - corner3 = width * (-sin, cos)
            Box q;
            q.l = sqrtf(ex * ex + ey * ey);
            q.w = sqrtf(fx * fx + fy * fy);
            if (!(q.l > 0.0f) || !(q.w > 0.0f)) continue;          // masked / degenerate control: no area
            q.x = 0.5f * (c[0] + c[4]);
            q.y = 0.5f * (c[1] + c[5]);
            q.c = ex / q.l;
            q.s = ey / q.l;
            hit = inter_area(p, q) > 0.0f;
        }
    }
    out[g] = hit ? 1 : 0;
}

// ---- non-visual observations (Simulator.get_all_agents_relative, simulator.py:748-781; utils.relative /
// rotate / normalize_angle, utils.py:31-79): the pose of every agent j in the frame of every origin agent i.
// rel_pair writes one output row: agent t in the frame of origin o.  agents_relative and nearest_agents_relative both
// use it, so a nearest-agent slot holds the bits of the matching agents_relative entry.
__device__ __forceinline__ void rel_pair(const float* __restrict__ o, const float* __restrict__ t, float2* w) {
    const float ang = -o[2];
    float s, c;
    tds::sincos_cr(ang, s, c);
    const float dx = t[0] - o[0], dy = t[1] - o[1];
    // remainder with the sign of the divisor (torch.remainder), then shift back: normalize_angle
    const float two_pi = 6.283185307179586f, pi = 3.141592653589793f;
    float r = fmodf((t[2] - o[2]) + pi, two_pi);
    if (r != 0.0f && r < 0.0f) r += two_pi;
    w[0] = make_float2(c * dx + (-s) * dy, s * dx + c * dy);
    w[1] = make_float2(r - pi, t[3]);
    w[2] = make_float2(t[4], t[5]);
}

// One thread per output row (b, i, k); with exclude_self row k of origin i is agent j = k + (k >= i), which is the
// reference's boolean-mask removal of the diagonal without its host synchronisation.
__global__ void __launch_bounds__(256) agents_relative_kernel(const float* __restrict__ absolute, int B, int A, int N,
                                                              int exclude_self, int per_origin, float* __restrict__ out) {
    const int M = exclude_self ? N - 1 : N;
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (int64_t)B * A * M) return;
    const int k = (int)(g % M);
    const int64_t bi = g / M;
    const int i = (int)(bi % A);
    const int64_t b = bi / A;
    const int j = exclude_self ? k + (k >= i) : k;
    // per_origin: absolute is [B,A,N,6], what each origin agent perceives (simulator.py:784-821)
    const float* base = per_origin ? absolute + (b * A + i) * (int64_t)N * 6 : absolute + b * (int64_t)N * 6;
    rel_pair(base + (int64_t)i * 6, base + (int64_t)j * 6, reinterpret_cast<float2*>(out + g * 6));
}

// ---- backward of agents_relative (autograd through utils.relative / rotate / normalize_angle).  For a pair (origin
// i, observed j) with s, c = sincos_cr(-psi_i), (rx, ry) recomputed as in the forward and upstream row g = (g0..g5):
//   observed j: d x_j = c g0 + s g1,  d y_j = -s g0 + c g1,  d psi_j = g2 (torch.remainder's backward is 1),
//               d (length, width, present)_j = (g3, g4, g5)
//   origin i:   d x_i = -d x_j,  d y_i = -d y_j,  d psi_i = g0 ry - g1 rx - g2
// No float atomics: every gradient element sums its terms in an order fixed by the code, whatever the grid, so two
// calls return the same bits.  An invalid pair (the self entry with exclude_self, a column past N) is skipped by a
// branch, not multiplied by 0, so a NaN pose of one agent does not reach the gradients of the others.
constexpr int kRelWarps = 8;         // warps per CTA of both backward kernels
constexpr int kRelChunk = 1024;      // origins per pass of the shared-mode kernel (shared memory: 28 B per origin)

struct RelPairGrad {
    float tx, ty, tpsi;              // observed terms d x_j, d y_j; origin term d psi_i
};

__device__ __forceinline__ RelPairGrad rel_pair_grad(float s, float c, float dx, float dy, float2 g01, float g2) {
    const float rx = c * dx + (-s) * dy, ry = s * dx + c * dy;
    return {c * g01.x + s * g01.y, (-s) * g01.x + c * g01.y, (g01.x * ry - g01.y * rx) - g2};
}

// Shared mode (absolute [B,N,6], the first A agents are the origins): one CTA per environment.  The columns are
// taken 32 at a time, one per lane; the warps deal out the origin rows (row i to warp i mod 8, two rows in flight per
// warp), so a warp reads 768 contiguous bytes of a row per step and the whole gradient is read once.  Per tile:
//   - a lane sums the observed terms of its column over its warp's rows; the 8 warp partials meet in shared memory
//     and are added in warp order, then written (or, past the first chunk of origins, added) to d absolute;
//   - the origin terms of a row are summed over the tile's lanes by shuffles and added, tile by tile, to the row's
//     sum in shared memory (only the row's warp touches it), which is added to d absolute at the end of the chunk.
__global__ void __launch_bounds__(kRelWarps * 32) agents_relative_bwd_kernel(const float* __restrict__ absolute,
                                                                              const float* __restrict__ gout, int A, int N,
                                                                              int exclude_self, float* __restrict__ gabs) {
    extern __shared__ float4 s_org[];                              // [chunk] x, y, s, c of the origins
    const int chunk = min(A, kRelChunk);
    float* s_row = reinterpret_cast<float*>(s_org + chunk);        // [chunk][3] sums of the origin terms
    float* s_col = s_row + 3 * chunk;                              // [kRelWarps][32][6] column partials of a tile
    const int M = exclude_self ? N - 1 : N;
    const int64_t b = blockIdx.x;
    const float* ab = absolute + b * N * 6;
    const float* gb = gout + b * A * (int64_t)M * 6;
    float* gw = gabs + b * N * 6;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int a0 = 0; a0 == 0 || a0 < A; a0 += kRelChunk) {        // once with A = 0: the zero gradient is written
        const int a1 = min(A, a0 + kRelChunk);
        for (int t = threadIdx.x; t < a1 - a0; t += blockDim.x) {
            const float* o = ab + (int64_t)(a0 + t) * 6;
            float s, c;
            tds::sincos_cr(-o[2], s, c);
            s_org[t] = make_float4(o[0], o[1], s, c);
            s_row[3 * t] = s_row[3 * t + 1] = s_row[3 * t + 2] = 0.0f;
        }
        __syncthreads();
        for (int n0 = 0; n0 < N; n0 += 32) {
            const int n = n0 + lane;
            const bool col = n < N;
            const float xn = col ? ab[(int64_t)n * 6] : 0.0f, yn = col ? ab[(int64_t)n * 6 + 1] : 0.0f;
            float acc[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
            for (int i0 = a0 + warp; i0 < a1; i0 += 2 * kRelWarps) {
                float2 g[2][3];
                bool valid[2];
#pragma unroll
                for (int r = 0; r < 2; r++) {                      // both rows' loads first: 1.5 KB in flight per warp
                    const int i = i0 + r * kRelWarps;
                    valid[r] = col && i < a1 && !(exclude_self && n == i);
                    const int k = exclude_self ? n - (n > i) : n;
                    const float2* p = reinterpret_cast<const float2*>(gb + ((int64_t)i * M + k) * 6);
#pragma unroll
                    for (int q = 0; q < 3; q++) g[r][q] = valid[r] ? __ldcs(p + q) : make_float2(0.0f, 0.0f);
                }
#pragma unroll
                for (int r = 0; r < 2; r++) {
                    const int i = i0 + r * kRelWarps;
                    if (i >= a1) break;                            // warp-uniform
                    const float4 o = s_org[i - a0];
                    RelPairGrad t = {0.0f, 0.0f, 0.0f};
                    if (valid[r]) {
                        t = rel_pair_grad(o.z, o.w, xn - o.x, yn - o.y, g[r][0], g[r][1].x);
                        acc[0] += t.tx;
                        acc[1] += t.ty;
                        acc[2] += g[r][1].x;
                        acc[3] += g[r][1].y;
                        acc[4] += g[r][2].x;
                        acc[5] += g[r][2].y;
                    }
                    const float sx = tds::warp_sum(t.tx), sy = tds::warp_sum(t.ty), sp = tds::warp_sum(t.tpsi);
                    if (lane == 0) {
                        float* rs = s_row + 3 * (i - a0);
                        rs[0] += sx;
                        rs[1] += sy;
                        rs[2] += sp;
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 6; q++) s_col[(warp * 32 + lane) * 6 + q] = acc[q];
            __syncthreads();
            if (threadIdx.x < 32 * 6 && n0 + (int)threadIdx.x / 6 < N) {     // coalesced: 32 columns x 6 values
                float v = 0.0f;
#pragma unroll
                for (int w = 0; w < kRelWarps; w++) v += s_col[w * 32 * 6 + threadIdx.x];
                float* dst = gw + (int64_t)n0 * 6 + threadIdx.x;
                *dst = a0 == 0 ? v : *dst + v;
            }
            __syncthreads();
        }
        // the origins' own terms: d xy_i = -(sum of the observed xy terms of row i), d psi_i = sum of its psi terms
        for (int t = threadIdx.x; t < 3 * (a1 - a0); t += blockDim.x) {
            float* dst = gw + (int64_t)(a0 + t / 3) * 6 + t % 3;
            *dst = t % 3 == 2 ? *dst + s_row[t] : *dst - s_row[t];
        }
        __syncthreads();
    }
}

// Per-origin mode (absolute [B,A,N,6], row (b,i) relative to its own entry [b,i,i]): every entry but the origin's is
// read by exactly one output row, so one warp per row (b,i) writes the observed terms of entries j != i as it reads the
// row, lane by lane, and sums the origin terms into entry i: per lane over its columns, then a shuffle tree; without
// exclude_self the self row's observed terms are added to that last.
__global__ void __launch_bounds__(kRelWarps * 32) agents_relative_bwd_per_origin_kernel(const float* __restrict__ absolute,
                                                                                         const float* __restrict__ gout,
                                                                                         int64_t rows, int A, int N,
                                                                                         int exclude_self,
                                                                                         float* __restrict__ gabs) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kRelWarps + warp;
    if (row >= rows) return;                                       // warp-uniform
    const int M = exclude_self ? N - 1 : N;
    const int i = (int)(row % A);
    const float* ab = absolute + row * N * 6;
    const float* gr = gout + row * M * 6;
    float* out = gabs + row * N * 6;
    const float xo = ab[(int64_t)i * 6], yo = ab[(int64_t)i * 6 + 1];
    float s, c;
    tds::sincos_cr(-ab[(int64_t)i * 6 + 2], s, c);
    float px = 0.0f, py = 0.0f, pp = 0.0f;
    float2 self[3] = {};
#pragma unroll 4
    for (int j = lane; j < N; j += 32) {
        if (exclude_self && j == i) continue;
        const int k = exclude_self ? j - (j > i) : j;
        const float2* p = reinterpret_cast<const float2*>(gr + (int64_t)k * 6);
        const float2 g01 = __ldcs(p), g23 = __ldcs(p + 1), g45 = __ldcs(p + 2);
        const float2 xy = __ldcs(reinterpret_cast<const float2*>(ab + (int64_t)j * 6));
        const RelPairGrad t = rel_pair_grad(s, c, xy.x - xo, xy.y - yo, g01, g23.x);
        px += t.tx;
        py += t.ty;
        pp += t.tpsi;
        const float2 d[3] = {make_float2(t.tx, t.ty), g23, g45};
        if (j == i) {
            self[0] = d[0]; self[1] = d[1]; self[2] = d[2];
        } else {
            float2* w = reinterpret_cast<float2*>(out + (int64_t)j * 6);
#pragma unroll
            for (int q = 0; q < 3; q++) __stcs(w + q, d[q]);
        }
    }
    px = tds::warp_sum(px);
    py = tds::warp_sum(py);
    pp = tds::warp_sum(pp);
    if (lane == (i & 31)) {                                        // the lane that holds the self row
        float2* w = reinterpret_cast<float2*>(out + (int64_t)i * 6);
        w[0] = make_float2(self[0].x - px, self[0].y - py);
        w[1] = make_float2(self[1].x + pp, self[1].y);
        w[2] = self[2];
    }
}

// ---- nearest-agent observations: the k nearest eligible agents of every origin, as rows of agents_relative (without
// exclusion).  Candidate j != i of origin i is eligible iff present_j != 0 and key = dx*dx + dy*dy <= r2 (float32,
// every operation rounded on its own; a NaN key fails the test).  Eligible candidates are ordered by (key, j): both
// are packed into one 64-bit word, key bits above j, and a non-negative float orders like its bit pattern, so the
// words are distinct and order like the pairs.  Slots past the eligible candidates are zero with index -1.
constexpr int kNearWarps = 8;                 // warps per CTA of the nearest-agent kernels
using tds::kNearEmpty;

// One warp per origin row (b, i).  The warp keeps the k smallest words seen so far as a sorted list in registers
// (tds::near_insert); the lanes take 32 candidates at a time.  The k winners' rows are written by rel_pair.
template <int R>
__global__ void __launch_bounds__(kNearWarps * 32) nearest_agents_relative_kernel(const float* __restrict__ absolute,
                                                                                  int64_t rows, int A, int N, int k,
                                                                                  int per_origin, float r2,
                                                                                  float* __restrict__ out,
                                                                                  int64_t* __restrict__ idx) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kNearWarps + warp;
    if (row >= rows) return;                                       // warp-uniform
    const int i = (int)(row % A);
    const float* base = absolute + (per_origin ? row : row / A) * (int64_t)N * 6;
    const float* o = base + (int64_t)i * 6;
    const float xo = o[0], yo = o[1];
    unsigned long long list[R];
#pragma unroll
    for (int r = 0; r < R; r++) list[r] = kNearEmpty;
    const int last_r = (k - 1) >> 5, last_lane = (k - 1) & 31;
    unsigned long long thr = kNearEmpty;                           // the word in slot k - 1
    for (int j0 = 0; j0 < N; j0 += 32) {
        const int j = j0 + lane;
        unsigned long long cand = kNearEmpty;
        if (j < N && j != i) {
            const float* t = base + (int64_t)j * 6;
            const float2 xy = *reinterpret_cast<const float2*>(t);
            const float dx = xy.x - xo, dy = xy.y - yo;
            const float key = dx * dx + dy * dy;
            if (t[5] != 0.0f && key <= r2) cand = ((unsigned long long)__float_as_uint(key) << 32) | (unsigned)j;
        }
        tds::near_insert<R>(list, cand, thr, last_r, last_lane, lane);
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int s = r * 32 + lane;
        if (s >= k) break;
        const int64_t e = row * k + s;
        float2* w = reinterpret_cast<float2*>(out + e * 6);
        if (list[r] != kNearEmpty) {
            const int j = (int)(unsigned)list[r];
            rel_pair(o, base + (int64_t)j * 6, w);
            idx[e] = j;
        } else {
            w[0] = w[1] = w[2] = make_float2(0.0f, 0.0f);
            idx[e] = -1;
        }
    }
}

// Backward, per-origin mode (absolute [B,A,N,6]): one warp per row (b, i).  The row's gradient is zeroed, then the
// lanes take the slots: slot s with agent j writes the observed terms of the pair (i, j) into entry j (the agents of a
// row are distinct, so no two slots write one entry), and the origin terms, summed per lane over its slots and then by
// a shuffle tree, go into entry i.  A slot whose index is not an agent of the row other than i is skipped by a branch.
__global__ void __launch_bounds__(kNearWarps * 32) nearest_agents_relative_bwd_per_origin_kernel(
    const float* __restrict__ absolute, const int64_t* __restrict__ idx, const float* __restrict__ gout, int64_t rows,
    int A, int N, int k, float* __restrict__ gabs) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kNearWarps + warp;
    if (row >= rows) return;                                       // warp-uniform
    const int i = (int)(row % A);
    const float* ab = absolute + row * N * 6;
    float* out = gabs + row * N * 6;
    float2* z = reinterpret_cast<float2*>(out);
    for (int q = lane; q < 3 * N; q += 32) z[q] = make_float2(0.0f, 0.0f);
    __syncwarp();
    const float xo = ab[(int64_t)i * 6], yo = ab[(int64_t)i * 6 + 1];
    float s, c;
    tds::sincos_cr(-ab[(int64_t)i * 6 + 2], s, c);
    float px = 0.0f, py = 0.0f, pp = 0.0f;
    for (int sl = lane; sl < k; sl += 32) {
        const int64_t e = row * k + sl;
        const int64_t j = idx[e];
        if (j < 0 || j >= N || j == i) continue;                   // an empty slot
        const float2* p = reinterpret_cast<const float2*>(gout + e * 6);
        const float2 g01 = p[0], g23 = p[1], g45 = p[2];
        const float2 xy = *reinterpret_cast<const float2*>(ab + j * 6);
        const RelPairGrad t = rel_pair_grad(s, c, xy.x - xo, xy.y - yo, g01, g23.x);
        px += t.tx;
        py += t.ty;
        pp += t.tpsi;
        float2* w = reinterpret_cast<float2*>(out + j * 6);
        w[0] = make_float2(t.tx, t.ty);
        w[1] = g23;
        w[2] = g45;
    }
    px = tds::warp_sum(px);
    py = tds::warp_sum(py);
    pp = tds::warp_sum(pp);
    if (lane == 0) {                                               // entry i is never a slot: only the origin terms
        out[(int64_t)i * 6] = -px;
        out[(int64_t)i * 6 + 1] = -py;
        out[(int64_t)i * 6 + 2] = pp;
    }
}

// Backward, shared mode (absolute [B,N,6]): one CTA per environment, a tds::ColSums column sum (tds_colsum.cuh).  Each
// warp takes origin rows i = warp, warp + 8, ...; its lanes take the row's slots and add the observed terms of slot
// (i, s) to the accumulator of column j directly (distinct within a row; a __syncwarp separates the rows).  In the pass
// that holds column i, the row's origin terms are summed by a shuffle tree and added to column i too.  Memory is
// O(B A k + B N); no dense [B,A,N,6] is formed.
__global__ void __launch_bounds__(kNearWarps * 32) nearest_agents_relative_bwd_kernel(
    const float* __restrict__ absolute, const int64_t* __restrict__ idx, const float* __restrict__ gout, int A, int N,
    int k, int cols, float* __restrict__ gabs) {
    extern __shared__ float s_acc[];                               // [kNearWarps][cols][6]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t b = blockIdx.x;
    const float* ab = absolute + b * N * 6;
    const int64_t* ib = idx + b * A * (int64_t)k;
    const float* gb = gout + b * A * (int64_t)k * 6;
    float* gw = gabs + b * N * 6;
    const tds::ColSums<kNearWarps, 6> sums(s_acc, cols, warp);
    for (int n0 = 0; n0 < N; n0 += cols) {
        const int nc = min(cols, N - n0);
        sums.zero(nc, lane);
        for (int i = warp; i < A; i += kNearWarps) {
            const bool own = i >= n0 && i < n0 + nc;               // warp-uniform: the origin's column is in this pass
            const float* o = ab + (int64_t)i * 6;
            const float xo = o[0], yo = o[1];
            float s, c;
            tds::sincos_cr(-o[2], s, c);
            float px = 0.0f, py = 0.0f, pp = 0.0f;
            for (int sl = lane; sl < k; sl += 32) {
                const int64_t e = (int64_t)i * k + sl;
                const int64_t j = ib[e];
                const bool valid = j >= 0 && j < N && j != i;      // else an empty slot
                const bool col = valid && j >= n0 && j < n0 + nc;
                if (!col && !(valid && own)) continue;
                const float2* p = reinterpret_cast<const float2*>(gb + e * 6);
                const float2 g01 = p[0], g23 = p[1], g45 = p[2];
                const float2 xy = *reinterpret_cast<const float2*>(ab + j * 6);
                const RelPairGrad t = rel_pair_grad(s, c, xy.x - xo, xy.y - yo, g01, g23.x);
                px += t.tx;
                py += t.ty;
                pp += t.tpsi;
                if (col) {
                    float* a = sums.acc + (j - n0) * 6;
                    a[0] += t.tx;
                    a[1] += t.ty;
                    a[2] += g23.x;
                    a[3] += g23.y;
                    a[4] += g45.x;
                    a[5] += g45.y;
                }
            }
            if (own) {
                px = tds::warp_sum(px);
                py = tds::warp_sum(py);
                pp = tds::warp_sum(pp);
                __syncwarp();
                if (lane == 0) {
                    float* a = sums.acc + (i - n0) * 6;
                    a[0] -= px;
                    a[1] -= py;
                    a[2] += pp;
                }
            }
            __syncwarp();
        }
        __syncthreads();
        for (int q = threadIdx.x; q < 6 * nc; q += blockDim.x)     // coalesced: the pass's columns x 6 values
            gw[(int64_t)n0 * 6 + q] = sums.total(q / 6, q % 6);
        __syncthreads();
    }
}

// ---- noisy observations (StandardSensingObservationNoise, observation_noise.py:69-132).
// get_noisy_state: what origin agent a perceives of agent e = its state + eps * deviation(distance), the deviation
// growing in steps at 0.5, 25, 50 and 100 m.  The normal deviates eps are an input (torch.randn on the device).
__global__ void __launch_bounds__(256) sensing_noise_kernel(const float4* __restrict__ all_state, const float4* __restrict__ eps,
                                                            int64_t n, int A, int N, float4* __restrict__ out) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    const int e = (int)(g % N);
    const int a = (int)((g / N) % A);
    const int64_t b = g / ((int64_t)N * A);
    const float4 ego = all_state[b * N + a], t = all_state[b * N + e], z = eps[g];
    const float dx = ego.x - t.x, dy = ego.y - t.y;
    const float dist = sqrtf(dx * dx + dy * dy);
    const float dev = dist > 100.0f ? 3.83f : (dist > 50.0f ? 3.2f : (dist > 25.0f ? 1.6f : (dist > 0.5f ? 0.19f : 0.0f)));
    out[g] = make_float4(t.x + z.x * dev, t.y + z.y * dev, t.z + z.z * dev, t.w + z.w * dev);
}

// get_noisy_present_mask: agent e is hidden from origin a if the segment a -> e crosses the circle (radius = half the
// width) of any third agent o, o != e, o != a (utils.line_circle_intersection, utils.py:139-187; absent agents occlude
// too, as in the reference).  One CTA per (environment, origin), the agents' circles staged in shared memory.
__global__ void __launch_bounds__(128) sensing_occlusion_kernel(const float4* __restrict__ all_state, const float2* __restrict__ all_size,
                                                                const uint8_t* __restrict__ base_mask, int A, int N,
                                                                uint8_t* __restrict__ out) {
    extern __shared__ float s_circ[];            // [N][3] x, y, radius
    const int a = blockIdx.x;
    const int64_t b = blockIdx.y;
    for (int o = threadIdx.x; o < N; o += blockDim.x) {
        const float4 st = all_state[b * N + o];
        s_circ[3 * o] = st.x; s_circ[3 * o + 1] = st.y; s_circ[3 * o + 2] = all_size[b * N + o].y / 2.0f;
    }
    __syncthreads();
    const float ex = s_circ[3 * a], ey = s_circ[3 * a + 1];
    for (int e = threadIdx.x; e < N; e += blockDim.x) {
        const float dx = s_circ[3 * e] - ex, dy = s_circ[3 * e + 1] - ey;
        const float qa = dx * dx + dy * dy;
        const float a_safe = fabsf(qa) < 1e-8f ? 1e-8f : qa;
        bool hidden = false;
        for (int o = 0; o < N && !hidden; o++) {
            if (o == e || o == a) continue;
            const float fx = ex - s_circ[3 * o], fy = ey - s_circ[3 * o + 1], r = s_circ[3 * o + 2];
            const float qb = 2.0f * (fx * dx + fy * dy);
            const float qc = (fx * fx + fy * fy) - r * r;
            const float disc = qb * qb - (4.0f * qa) * qc;
            if (disc >= 0.0f) {
                const float sq = sqrtf(fmaxf(disc, 0.0f));
                const float t1 = ((-qb) - sq) / (2.0f * a_safe), t2 = ((-qb) + sq) / (2.0f * a_safe);
                hidden = fminf(t1, t2) <= 1.0f && fmaxf(t1, t2) >= 0.0f;
            }
        }
        out[(b * A + a) * N + e] = (base_mask[b * N + e] != 0 && !hidden) ? 1 : 0;
    }
}

// ---- aggregate infraction metrics of a step (the vector that is all-reduced over the GPUs, SURVEY.md §8e):
// acc[0..5] += sum of collision over present agents, sum of offroad, agents with collision > 0, agents with
// offroad > 0, present agents, agent slots.  One cluster of kMetricCtas CTAs with a fixed reduction order: thread t of
// the cluster sums elements t, t + 8192, ... in order, then warps (shuffle tree), the 32 warps of a CTA and the CTAs of
// the cluster (in CTA 0's shared memory) are summed in index order.  The sums are reproducible run to run; the counts
// are exact.  Versions that reduced in one CTA summed in another order: their float64 sums differ from these in the last
// bits, the counts are the same.
constexpr int kMetricCtas = 8;
__global__ void __cluster_dims__(kMetricCtas, 1, 1) __launch_bounds__(1024)
infraction_metrics_kernel(const float* __restrict__ collision, const float* __restrict__ offroad,
                          const uint8_t* __restrict__ present, int64_t n, double* __restrict__ acc) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ double s_part[32][5];
    __shared__ double s_cta[kMetricCtas][5];          // used in CTA 0: one row per CTA of the cluster
    const int rank = (int)cluster.block_rank();
    double v[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    const int64_t stride = (int64_t)kMetricCtas * blockDim.x;
    for (int64_t i = (int64_t)rank * blockDim.x + threadIdx.x; i < n; i += stride) {
        const bool here = present ? present[i] != 0 : true;
        const float c = collision[i], o = offroad[i];
        if (here) { v[0] += (double)c; v[1] += (double)o; v[2] += c > 0.0f; v[3] += o > 0.0f; v[4] += 1.0; }
    }
#pragma unroll
    for (int k = 0; k < 5; k++)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0)
        for (int k = 0; k < 5; k++) s_part[warp][k] = v[k];
    __syncthreads();
    if (threadIdx.x < 5) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += s_part[w][threadIdx.x];
        cluster.map_shared_rank(&s_cta[0][0], 0)[rank * 5 + threadIdx.x] = t;
    }
    cluster.sync();
    if (rank == 0 && threadIdx.x < 5) {
        double t = 0.0;
        for (int r = 0; r < kMetricCtas; r++) t += s_cta[r][threadIdx.x];
        acc[threadIdx.x] += t;
    }
    if (rank == 0 && threadIdx.x == 5) acc[5] += (double)n;
}

// ---- IoU backward.  d(intersection area) is the boundary integral of the normal velocity: every edge of
// the clipped polygon lies either on a face of box q (it moves with q's pose and size) or on a face of box p
// (it moves with p's size).  Each polygon vertex carries the tag of the edge that leaves it:
//   0..3 = q's edge k (corner k -> k+1: faces +y_q, -x_q, -y_q, +x_q), 4..7 = p's faces +x, -x, +y, -y.
struct TaggedPoly {
    float x[10], y[10];
    int tag[10];
    int n;
};

__device__ __forceinline__ void clip_axis_tagged(const TaggedPoly& in, TaggedPoly& out, int axis, float sign, float bound,
                                                 int plane_tag) {
    int m = 0;
    for (int i = 0; i < in.n; i++) {
        const int j = (i + 1 == in.n) ? 0 : i + 1;
        const float ax = in.x[i], ay = in.y[i], bx = in.x[j], by = in.y[j];
        const float da = sign * (axis ? ay : ax) - bound;
        const float db = sign * (axis ? by : bx) - bound;
        const bool ina = da <= 0.0f, inb = db <= 0.0f;
        if (ina) { out.x[m] = ax; out.y[m] = ay; out.tag[m] = in.tag[i]; m++; }
        if (ina != inb) {
            const float t = da / (da - db);
            out.x[m] = ax + t * (bx - ax);
            out.y[m] = ay + t * (by - ay);
            // leaving the half-plane: the next edge runs along the clip line; entering: it continues on edge i
            out.tag[m] = ina ? plane_tag : in.tag[i];
            m++;
        }
    }
    out.n = m;
}

// accumulates wgt * d IoU / d(box p), d(box q) into gp, gq (x, y, l, w, psi).  Returns false for no overlap.
__device__ bool iou_pair_grad(const float* praw, const float* qraw, float wgt, float* gp, float* gq) {
    const Box p = make_box(praw[0], praw[1], praw[2], praw[3], praw[4]);
    const Box q = make_box(qraw[0], qraw[1], qraw[2], qraw[3], qraw[4]);
    const float dx = q.x - p.x, dy = q.y - p.y;
    const float rp = 0.5f * sqrtf(p.l * p.l + p.w * p.w), rq = 0.5f * sqrtf(q.l * q.l + q.w * q.w);
    const float reach = rp + rq;
    if (dx * dx + dy * dy > reach * reach * 1.0001f + 1e-6f) return false;
    const float cr = p.c * q.c + p.s * q.s, sr = p.c * q.s - p.s * q.c;     // rotation of q in p's frame
    const float tx = p.c * dx + p.s * dy, ty = p.c * dy - p.s * dx;         // centre of q in p's frame
    const float hx = 0.5f * q.l, hy = 0.5f * q.w;
    TaggedPoly a, b;
    const float sx[4] = {1.f, -1.f, -1.f, 1.f}, sy[4] = {1.f, 1.f, -1.f, -1.f};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float ux = sx[k] * hx, uy = sy[k] * hy;
        a.x[k] = tx + (ux * cr - uy * sr);
        a.y[k] = ty + (ux * sr + uy * cr);
        a.tag[k] = k;
    }
    a.n = 4;
    const float bx = 0.5f * p.l, by = 0.5f * p.w;
    clip_axis_tagged(a, b, 0, 1.f, bx, 4);
    clip_axis_tagged(b, a, 0, -1.f, bx, 5);
    clip_axis_tagged(a, b, 1, 1.f, by, 6);
    clip_axis_tagged(b, a, 1, -1.f, by, 7);
    if (a.n < 3) return false;
    float tot = 0.0f;
    // gradients of the intersection area in p's frame
    float g_tx = 0.f, g_ty = 0.f, g_rot = 0.f, g_lq = 0.f, g_wq = 0.f, g_lp = 0.f, g_wp = 0.f;
    // outward normals of q's faces in p's frame: +y_q, -x_q, -y_q, +x_q
    const float nqx[4] = {-sr, -cr, sr, cr}, nqy[4] = {cr, -sr, -cr, sr};
    for (int i = 0; i < a.n; i++) {
        const int j = (i + 1 == a.n) ? 0 : i + 1;
        tot += a.x[i] * a.y[j] - a.y[i] * a.x[j];
        const float ex = a.x[j] - a.x[i], ey = a.y[j] - a.y[i];
        const float len = sqrtf(ex * ex + ey * ey);
        const int tg = a.tag[i];
        if (tg < 4) {
            const float nx = nqx[tg], ny = nqy[tg];
            g_tx += nx * len;
            g_ty += ny * len;
            const float mx = 0.5f * (a.x[i] + a.x[j]) - tx, my = 0.5f * (a.y[i] + a.y[j]) - ty;
            g_rot += (nx * (-my) + ny * mx) * len;          // n . (z x (m - t))
            if (tg == 0 || tg == 2) g_wq += 0.5f * len; else g_lq += 0.5f * len;
        } else if (tg < 6) {
            g_lp += 0.5f * len;
        } else {
            g_wp += 0.5f * len;
        }
    }
    const float inter = 0.5f * fabsf(tot);
    const float a1 = p.l * p.w, a2 = q.l * q.w;
    const float U = a1 + a2 - inter;
    if (!(U > 0.0f) || !(inter > 0.0f)) return false;
    // IoU = A / U, U = a1 + a2 - A:  dIoU = kA dA - kU d(a1 + a2)
    const float kA = wgt * (1.0f / U + inter / (U * U));
    const float kU = wgt * inter / (U * U);
    // chain to world parameters: t = R(-psi_p) (c_q - c_p), rot = psi_q - psi_p
    const float wx = p.c * g_tx - p.s * g_ty, wy = p.s * g_tx + p.c * g_ty;   // R(psi_p) g_t
    gq[0] += kA * wx; gq[1] += kA * wy;
    gp[0] -= kA * wx; gp[1] -= kA * wy;
    gq[4] += kA * g_rot;
    gp[4] += kA * (-g_rot + g_tx * ty - g_ty * tx);
    gq[2] += kA * g_lq - kU * q.w; gq[3] += kA * g_wq - kU * q.l;
    gp[2] += kA * g_lp - kU * p.w; gp[3] += kA * g_wp - kU * p.l;
    return true;
}

// ---------------------------------------------------------------- element-wise API
__global__ void __launch_bounds__(256) pairwise_fwd_kernel(const float* __restrict__ b1, const float* __restrict__ b2,
                                                           int64_t n, int metric, float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = b1 + 5 * i;
    const float* q = b2 + 5 * i;
    if (metric == TDS_METRIC_DISCS) {
        const Discs dp = make_discs(p[0], p[1], p[2], p[3], p[4]);
        const Discs dq = make_discs(q[0], q[1], q[2], q[3], q[4]);
        out[i] = discs_overlap(dp, dq, nullptr, nullptr, nullptr);
    } else {
        out[i] = iou_pair(make_box(p[0], p[1], p[2], p[3], p[4]), make_box(q[0], q[1], q[2], q[3], q[4]));
    }
}

// gradient of one disc pair w.r.t. both boxes, scaled by wgt; returns false if the pair has zero gradient
struct BoxGrad {
    float g[5];
};
__device__ __forceinline__ void disc_center_grad(float l, float w, float psi, int k, float gcx, float gcy, float gr,
                                                 BoxGrad& out) {
    // centre_k = (x,y) + off_k (cos yaw, sin yaw), off_k = (k-2) (half - r) / 2, yaw = psi + pi/2 [w > l]
    const float yaw = psi + 1.5707963705062866f * (w > l ? 1.0f : 0.0f);
    float s, c;
    tds::sincos_cr(yaw, s, c);
    const float half = fmaxf(l, w) / 2.0f, r = fminf(l, w) / 2.0f;
    const float kk = (float)(k - 2) * 0.5f;
    const float off = kk * (half - r);
    const float goff = gcx * c + gcy * s;
    out.g[0] += gcx;
    out.g[1] += gcy;
    out.g[4] += off * (gcy * c - gcx * s);
    // d half / d(l,w), d r / d(l,w): torch.maximum / minimum split the gradient evenly on ties
    float hl, hw, rl, rw;
    if (l > w) { hl = 0.5f; hw = 0.f; rl = 0.f; rw = 0.5f; }
    else if (l < w) { hl = 0.f; hw = 0.5f; rl = 0.5f; rw = 0.f; }
    else { hl = hw = rl = rw = 0.25f; }
    out.g[2] += goff * kk * (hl - rl) + gr * rl;
    out.g[3] += goff * kk * (hw - rw) + gr * rw;
}

__device__ __forceinline__ bool discs_pair_grad(const float* p, const float* q, float wgt, BoxGrad& gp, BoxGrad& gq) {
    const Discs dp = make_discs(p[0], p[1], p[2], p[3], p[4]);
    const Discs dq = make_discs(q[0], q[1], q[2], q[3], q[4]);
    int a, b;
    float d;
    const float o = discs_overlap(dp, dq, &a, &b, &d);
    if (!(o > 0.0f) || wgt == 0.0f) return false;
    const float R = dp.r + dq.r;
    const float go_d = -wgt / R;                 // d o / d dist
    const float go_R = wgt * d / (R * R);        // d o / d (r1 + r2)
    float ux = 0.f, uy = 0.f;                    // cdist backward: 0 at zero distance
    if (d > 0.0f) { ux = (dp.cx[a] - dq.cx[b]) / d; uy = (dp.cy[a] - dq.cy[b]) / d; }
    disc_center_grad(p[2], p[3], p[4], a, go_d * ux, go_d * uy, go_R, gp);
    disc_center_grad(q[2], q[3], q[4], b, -go_d * ux, -go_d * uy, go_R, gq);
    return true;
}

__global__ void __launch_bounds__(256) pairwise_bwd_kernel(const float* __restrict__ b1, const float* __restrict__ b2,
                                                           int64_t n, int metric, const float* __restrict__ gout,
                                                           float* __restrict__ g1, float* __restrict__ g2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    BoxGrad gp = {}, gq = {};
    if (metric == TDS_METRIC_DISCS) discs_pair_grad(b1 + 5 * i, b2 + 5 * i, gout[i], gp, gq);
    else iou_pair_grad(b1 + 5 * i, b2 + 5 * i, gout[i], gp.g, gq.g);
#pragma unroll
    for (int k = 0; k < 5; k++) {
        if (g1) g1[5 * i + k] = gp.g[k];
        if (g2) g2[5 * i + k] = gq.g[k];
    }
}

// ---------------------------------------------------------------- all-pairs
constexpr int kRowsPerCta = 64;
constexpr int kWarps = 8;

// shared memory: all N column boxes of the environment, as discs (12 floats + mask) or Box (6 floats + mask); the
// discs of the CTA's own rows follow the columns, so that every box goes through make_discs (and its double-precision
// sincos) once per CTA, all of them at the same time, and the row loop reads nothing but shared memory
template <int METRIC>
__global__ void __launch_bounds__(kWarps * 32) allpairs_fwd_kernel(const float* __restrict__ ego, const float* __restrict__ all,
                                                                  const uint8_t* __restrict__ mask, int A, int N,
                                                                  int ego_is_prefix, float* __restrict__ out,
                                                                  int32_t* __restrict__ argmax) {
    extern __shared__ float smem[];
    __shared__ int s_queue[METRIC == TDS_METRIC_IOU ? kWarps : 1][64];      // columns waiting for the clipping (IoU)
    constexpr int STRIDE = METRIC == TDS_METRIC_DISCS ? 13 : 7;   // odd strides: conflict-free column reads
    const int b = blockIdx.y;
    const int row0 = blockIdx.x * kRowsPerCta;
    const float* allb = all + (size_t)b * N * 5;
    const uint8_t* mb = mask + (size_t)b * N;
    const int staged = METRIC == TDS_METRIC_DISCS ? N + min(kRowsPerCta, A - row0) : N;
    for (int j = threadIdx.x; j < staged; j += blockDim.x) {
        const float* q = j < N ? allb + 5 * j : ego + ((size_t)b * A + row0 + (j - N)) * 5;
        float* s = smem + j * STRIDE;
        if (METRIC == TDS_METRIC_DISCS) {
            const Discs d = make_discs(q[0], q[1], q[2], q[3], q[4]);
#pragma unroll
            for (int k = 0; k < kDiscs; k++) { s[2 * k] = d.cx[k]; s[2 * k + 1] = d.cy[k]; }
            s[10] = d.r; s[11] = d.half; s[12] = j >= N || mb[j] ? 1.0f : 0.0f;
        } else {
            const Box d = make_box(q[0], q[1], q[2], q[3], q[4]);
            s[0] = d.x; s[1] = d.y; s[2] = d.l; s[3] = d.w; s[4] = d.s; s[5] = d.c; s[6] = mb[j] ? 1.0f : 0.0f;
        }
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int r = warp; r < kRowsPerCta; r += kWarps) {
        const int i = row0 + r;
        if (i >= A) break;
        const float* p = ego + ((size_t)b * A + i) * 5;
        float sum = 0.0f, best = -CUDART_INF_F;
        int besti = 0;
        if (METRIC == TDS_METRIC_DISCS) {
            Discs dp;
            {
                const float* s = smem + (N + r) * STRIDE;
#pragma unroll
                for (int k = 0; k < kDiscs; k++) { dp.cx[k] = s[2 * k]; dp.cy[k] = s[2 * k + 1]; }
                dp.r = s[10]; dp.half = s[11];
            }
            for (int j = lane; j < N; j += 32) {
                const float* s = smem + j * STRIDE;
                Discs dq;
#pragma unroll
                for (int k = 0; k < kDiscs; k++) { dq.cx[k] = s[2 * k]; dq.cy[k] = s[2 * k + 1]; }
                dq.r = s[10]; dq.half = s[11];
                float o = 0.0f;
                // centres further apart than the two half-lengths cannot have touching discs
                const float ddx = dp.cx[2] - dq.cx[2], ddy = dp.cy[2] - dq.cy[2];
                const float reach = dp.half + dq.half;
                if (ddx * ddx + ddy * ddy <= reach * reach * 1.0001f + 1e-6f)
                    o = discs_overlap(dp, dq, nullptr, nullptr, nullptr);
                o *= s[12];
                sum += o;
                if (o > best) { best = o; besti = j; }
            }
        } else {
            // Most pairs of a crowded scene end at the bounding-circle test and the few that need the clipping would
            // each hold up their warp: the columns that pass the test are queued per warp and clipped 32 at a time,
            // one per lane.  (best, besti) = the largest overlap and the lowest column that attains it, whatever
            // the order the columns are visited in.
            const Box bp = make_box(p[0], p[1], p[2], p[3], p[4]);
            const float rp = 0.5f * sqrtf(bp.l * bp.l + bp.w * bp.w);
            int* queue = s_queue[warp];
            int nq = 0;                                   // uniform over the warp
            auto take = [&](int j, float o) {
                sum += o;
                if (o > best || (o == best && j < besti)) { best = o; besti = j; }
            };
            auto clip = [&](int j) {
                const float* s = smem + j * STRIDE;
                Box bq;
                bq.x = s[0]; bq.y = s[1]; bq.l = s[2]; bq.w = s[3]; bq.s = s[4]; bq.c = s[5];
                take(j, iou_pair(bp, bq) * s[6]);
            };
            for (int j0 = 0; j0 < N; j0 += 32) {
                const int j = j0 + lane;
                bool cand = false;
                if (j < N) {
                    const float* s = smem + j * STRIDE;
                    if (ego_is_prefix && j == i) {
                        take(j, 1.0f * s[6]);
                    } else {
                        const float dx = s[0] - bp.x, dy = s[1] - bp.y;
                        const float reach = rp + 0.5f * sqrtf(s[2] * s[2] + s[3] * s[3]);
                        cand = s[6] != 0.0f && !(dx * dx + dy * dy > reach * reach * 1.0001f + 1e-6f);   // inter_area's own test
                        if (!cand) take(j, 0.0f);
                    }
                }
                const unsigned m = __ballot_sync(0xffffffffu, cand);
                if (cand) queue[nq + __popc(m & ((1u << lane) - 1u))] = j;
                nq += __popc(m);
                __syncwarp();
                if (nq >= 32) {
                    nq -= 32;
                    clip(queue[nq + lane]);
                    __syncwarp();
                }
            }
            if (lane < nq) clip(queue[lane]);
            __syncwarp();
        }
        sum = tds::warp_sum(sum);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
            if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
        }
        if (lane == 0) {
            const bool any = N > 0;
            out[(size_t)b * A + i] = any ? sum - best : 0.0f;
            if (argmax) argmax[(size_t)b * A + i] = besti;
        }
    }
}

template <int METRIC>
__global__ void __launch_bounds__(kWarps * 32) allpairs_bwd_kernel(const float* __restrict__ ego, const float* __restrict__ all,
                                                                  const uint8_t* __restrict__ mask, int A, int N,
                                                                  int ego_is_prefix, const float* __restrict__ gout,
                                                                        const int32_t* __restrict__ argmax,
                                                                        float* __restrict__ g_ego, float* __restrict__ g_all) {
    extern __shared__ float gcol[];              // [N][5] column gradients of this CTA
    const int b = blockIdx.y;
    const int row0 = blockIdx.x * kRowsPerCta;
    const float* allb = all + (size_t)b * N * 5;
    const uint8_t* mb = mask + (size_t)b * N;
    for (int k = threadIdx.x; k < N * 5; k += blockDim.x) gcol[k] = 0.0f;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int r = warp; r < kRowsPerCta; r += kWarps) {
        const int i = row0 + r;
        if (i >= A) break;
        const float* p = ego + ((size_t)b * A + i) * 5;
        const float g = gout[(size_t)b * A + i];
        const int am = argmax[(size_t)b * A + i];
        BoxGrad gp = {};
        for (int j = lane; j < N; j += 32) {
            // d out_i / d o_ij = m_j (1 - [j == argmax_i])
            const float wgt = (mb[j] && j != am) ? g : 0.0f;
            if (wgt == 0.0f) continue;
            if (METRIC == TDS_METRIC_IOU && ego_is_prefix && j == i) continue;   // o(i,i) := 1, a constant
            BoxGrad gq = {};
            const bool hit = METRIC == TDS_METRIC_DISCS ? discs_pair_grad(p, allb + 5 * j, wgt, gp, gq)
                                                        : iou_pair_grad(p, allb + 5 * j, wgt, gp.g, gq.g);
            if (hit) {
#pragma unroll
                for (int k = 0; k < 5; k++) atomicAdd(&gcol[5 * j + k], gq.g[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < 5; k++) {
            const float v = tds::warp_sum(gp.g[k]);
            if (lane == 0) g_ego[((size_t)b * A + i) * 5 + k] = v;
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < N * 5; k += blockDim.x) {
        const float v = gcol[k];
        if (v != 0.0f) atomicAdd(&g_all[(size_t)b * N * 5 + k], v);
    }
}

}  // namespace

extern "C" int tds_traffic_light_violation(const float* d_agent_box, const float* d_tl_corners, const int32_t* d_tl_state,
                                           const uint8_t* d_present, int32_t B, int32_t A, int32_t L, int32_t red_state,
                                           float rear_factor, uint8_t* d_out, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && L >= 0, "traffic_light_violation: negative size");
    if (B == 0 || A == 0) return TDS_OK;
    TDS_REQUIRE(d_agent_box && d_out, "traffic_light_violation: null pointer");
    TDS_REQUIRE(L == 0 || (d_tl_corners && d_tl_state), "traffic_light_violation: null traffic light tensors");
    TDS_REQUIRE(rear_factor > 0.0f && rear_factor <= 1.0f, "traffic_light_violation: rear_factor must be in (0, 1]");
    const int64_t n = (int64_t)B * A;
    tl_violation_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(d_agent_box, d_tl_corners, d_tl_state,
                                                                                   d_present, B, A, L, red_state,
                                                                                   rear_factor, d_out);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_infraction_metrics(const float* d_collision, const float* d_offroad, const uint8_t* d_present,
                                      int64_t n, double* d_acc, void* stream) {
    TDS_REQUIRE(n >= 0, "infraction_metrics: negative size");
    TDS_REQUIRE(d_acc && (n == 0 || (d_collision && d_offroad)), "infraction_metrics: null pointer");
    infraction_metrics_kernel<<<kMetricCtas, 1024, 0, (cudaStream_t)stream>>>(d_collision, d_offroad, d_present, n, d_acc);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_sensing_noise(const float* d_all_state, const float* d_eps, int32_t B, int32_t A, int32_t N,
                                 float* d_out, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "sensing_noise: need 0 <= A <= N");
    const int64_t n = (int64_t)B * A * N;
    if (n == 0) return TDS_OK;
    TDS_REQUIRE(d_all_state && d_eps && d_out, "sensing_noise: null pointer");
    sensing_noise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const float4*)d_all_state, (const float4*)d_eps,
                                                                                    n, A, N, (float4*)d_out);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_sensing_occlusion(const float* d_all_state, const float* d_all_size, const uint8_t* d_base_mask,
                                     int32_t B, int32_t A, int32_t N, uint8_t* d_out, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "sensing_occlusion: need 0 <= A <= N");
    if (B == 0 || A == 0 || N == 0) return TDS_OK;
    TDS_REQUIRE(d_all_state && d_all_size && d_base_mask && d_out, "sensing_occlusion: null pointer");
    TDS_REQUIRE(B <= 65535, "sensing_occlusion: B=%d exceeds 65535 (shard the batch)", B);
    const size_t smem = (size_t)N * 3 * sizeof(float);
    TDS_REQUIRE(smem <= 200 * 1024, "sensing_occlusion: N=%d does not fit shared memory", N);
    if (int e = tds::allow_dynamic_smem(sensing_occlusion_kernel, smem)) return e;
    sensing_occlusion_kernel<<<dim3(A, B), 128, smem, (cudaStream_t)stream>>>((const float4*)d_all_state, (const float2*)d_all_size,
                                                                             d_base_mask, A, N, d_out);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_agents_relative(const float* d_absolute, int32_t B, int32_t A, int32_t N, int32_t exclude_self,
                                   int32_t per_origin, float* d_out, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "agents_relative: need 0 <= A <= N");
    const int64_t M = exclude_self ? N - 1 : N;
    const int64_t n = (int64_t)B * A * M;
    if (n <= 0) return TDS_OK;
    TDS_REQUIRE(d_absolute && d_out, "agents_relative: null pointer");
    TDS_REQUIRE((n + 255) / 256 <= 2147483647LL, "agents_relative: too many pairs");
    agents_relative_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_absolute, B, A, N, exclude_self, per_origin, d_out);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_agents_relative_bwd(const float* d_absolute, const float* d_grad_out, int32_t B, int32_t A, int32_t N,
                                       int32_t exclude_self, int32_t per_origin, float* d_grad_absolute, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "agents_relative_bwd: need 0 <= A <= N");
    const int64_t M = exclude_self ? N - 1 : N;
    const int64_t agents = per_origin ? (int64_t)B * A * N : (int64_t)B * N;     // rows of d_absolute
    if (agents == 0) return TDS_OK;
    TDS_REQUIRE(d_absolute && d_grad_absolute && (A * M == 0 || d_grad_out), "agents_relative_bwd: null pointer");
    if (per_origin) {
        const int64_t rows = (int64_t)B * A, blocks = (rows + kRelWarps - 1) / kRelWarps;
        TDS_REQUIRE(blocks <= 2147483647LL, "agents_relative_bwd: too many rows");
        agents_relative_bwd_per_origin_kernel<<<(unsigned)blocks, kRelWarps * 32, 0, (cudaStream_t)stream>>>(
            d_absolute, d_grad_out, rows, A, N, exclude_self, d_grad_absolute);
    } else {
        const size_t smem = (size_t)std::min(A, kRelChunk) * 28 + kRelWarps * 32 * 6 * sizeof(float);
        agents_relative_bwd_kernel<<<(unsigned)B, kRelWarps * 32, smem, (cudaStream_t)stream>>>(
            d_absolute, d_grad_out, A, N, exclude_self, d_grad_absolute);
    }
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_nearest_agents_relative(const float* d_absolute, int32_t B, int32_t A, int32_t N, int32_t k,
                                           int32_t per_origin, float r2, float* d_out, int64_t* d_idx, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "nearest_agents_relative: need 0 <= A <= N");
    TDS_REQUIRE(k >= 1 && k <= 64, "nearest_agents_relative: need 1 <= k <= 64, got %d", k);
    TDS_REQUIRE(r2 >= 0.0f, "nearest_agents_relative: need r2 >= 0");
    const int64_t rows = (int64_t)B * A, blocks = (rows + kNearWarps - 1) / kNearWarps;
    if (rows == 0) return TDS_OK;
    TDS_REQUIRE(d_absolute && d_out && d_idx, "nearest_agents_relative: null pointer");
    TDS_REQUIRE(blocks <= 2147483647LL, "nearest_agents_relative: too many rows");
    if (k <= 32)
        nearest_agents_relative_kernel<1><<<(unsigned)blocks, kNearWarps * 32, 0, (cudaStream_t)stream>>>(
            d_absolute, rows, A, N, k, per_origin, r2, d_out, d_idx);
    else
        nearest_agents_relative_kernel<2><<<(unsigned)blocks, kNearWarps * 32, 0, (cudaStream_t)stream>>>(
            d_absolute, rows, A, N, k, per_origin, r2, d_out, d_idx);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_nearest_agents_relative_bwd(const float* d_absolute, const int64_t* d_idx, const float* d_grad_out,
                                               int32_t B, int32_t A, int32_t N, int32_t k, int32_t per_origin,
                                               float* d_grad_absolute, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "nearest_agents_relative_bwd: need 0 <= A <= N");
    TDS_REQUIRE(k >= 1 && k <= 64, "nearest_agents_relative_bwd: need 1 <= k <= 64, got %d", k);
    const int64_t agents = per_origin ? (int64_t)B * A * N : (int64_t)B * N;     // rows of d_absolute
    if (agents == 0) return TDS_OK;
    TDS_REQUIRE(d_absolute && d_grad_absolute && (A == 0 || (d_idx && d_grad_out)),
                "nearest_agents_relative_bwd: null pointer");
    if (per_origin) {
        const int64_t rows = (int64_t)B * A, blocks = (rows + kNearWarps - 1) / kNearWarps;
        TDS_REQUIRE(blocks <= 2147483647LL, "nearest_agents_relative_bwd: too many rows");
        nearest_agents_relative_bwd_per_origin_kernel<<<(unsigned)blocks, kNearWarps * 32, 0, (cudaStream_t)stream>>>(
            d_absolute, d_idx, d_grad_out, rows, A, N, k, d_grad_absolute);
    } else {
        const int cols = std::min(N, tds::kColsPerPass);
        const size_t smem = (size_t)kNearWarps * cols * 6 * sizeof(float);
        if (int e = tds::allow_dynamic_smem(nearest_agents_relative_bwd_kernel, smem)) return e;
        nearest_agents_relative_bwd_kernel<<<(unsigned)B, kNearWarps * 32, smem, (cudaStream_t)stream>>>(
            d_absolute, d_idx, d_grad_out, A, N, k, cols, d_grad_absolute);
    }
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_collision_pairwise_fwd(const float* d_box1, const float* d_box2, int64_t p, int32_t metric,
                                          float* d_out, void* stream) {
    TDS_REQUIRE(d_box1 && d_box2 && d_out, "collision_pairwise: null pointer");
    TDS_REQUIRE(metric == TDS_METRIC_DISCS || metric == TDS_METRIC_IOU, "collision_pairwise: unknown metric %d", metric);
    TDS_REQUIRE(p >= 0, "collision_pairwise: negative size");
    if (p == 0) return TDS_OK;
    pairwise_fwd_kernel<<<(unsigned)((p + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_box1, d_box2, p, metric, d_out);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_collision_pairwise_bwd(const float* d_box1, const float* d_box2, int64_t p, int32_t metric,
                                          const float* d_grad_out, float* d_grad_box1, float* d_grad_box2,
                                          void* stream) {
    TDS_REQUIRE(p >= 0, "collision_pairwise_bwd: negative size");
    if (p == 0) return TDS_OK;
    TDS_REQUIRE(d_box1 && d_box2 && d_grad_out, "collision_pairwise_bwd: null pointer");
    TDS_REQUIRE(metric == TDS_METRIC_DISCS || metric == TDS_METRIC_IOU, "collision_pairwise_bwd: unknown metric %d", metric);
    pairwise_bwd_kernel<<<(unsigned)((p + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_box1, d_box2, p, metric, d_grad_out,
                                                                                       d_grad_box1, d_grad_box2);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_collision_allpairs_fwd(const float* d_ego_box, const float* d_all_box, const uint8_t* d_mask,
                                          int32_t B, int32_t A, int32_t N, int32_t metric, int32_t ego_is_prefix,
                                          float* d_out, int32_t* d_argmax, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0, "collision_allpairs: negative size");
    if (B == 0 || A == 0) return TDS_OK;
    TDS_REQUIRE(d_ego_box && d_out, "collision_allpairs: null pointer");
    TDS_REQUIRE(N == 0 || (d_all_box && d_mask), "collision_allpairs: null pointer");
    TDS_REQUIRE(metric == TDS_METRIC_DISCS || metric == TDS_METRIC_IOU, "collision_allpairs: unknown metric %d", metric);
    TDS_REQUIRE(B <= 65535, "collision_allpairs: B=%d exceeds 65535 (shard the batch)", B);
    const dim3 grid((A + kRowsPerCta - 1) / kRowsPerCta, B);
    const size_t cols = (size_t)N * (metric == TDS_METRIC_DISCS ? 13 : 7) * sizeof(float);
    TDS_REQUIRE(cols <= 200 * 1024, "collision_allpairs: N=%d does not fit shared memory", N);
    // discs: the CTA's rows (at most 3.3 KB) come on top of the columns, within the 227 KB a CTA may have
    const size_t smem = metric == TDS_METRIC_DISCS ? cols + (size_t)std::min(A, kRowsPerCta) * 13 * sizeof(float) : cols;
    const auto kernel = metric == TDS_METRIC_DISCS ? allpairs_fwd_kernel<TDS_METRIC_DISCS> : allpairs_fwd_kernel<TDS_METRIC_IOU>;
    if (int e = tds::allow_dynamic_smem(kernel, smem)) return e;
    kernel<<<grid, kWarps * 32, smem, (cudaStream_t)stream>>>(d_ego_box, d_all_box, d_mask, A, N, ego_is_prefix, d_out, d_argmax);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_collision_allpairs_bwd(const float* d_ego_box, const float* d_all_box, const uint8_t* d_mask,
                                          int32_t B, int32_t A, int32_t N, int32_t metric, int32_t ego_is_prefix,
                                          const float* d_grad_out, const int32_t* d_argmax, float* d_grad_ego,
                                          float* d_grad_all, void* stream) {
    TDS_REQUIRE(metric == TDS_METRIC_DISCS || metric == TDS_METRIC_IOU, "collision_allpairs_bwd: unknown metric %d", metric);
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0, "collision_allpairs_bwd: negative size");
    if (B == 0 || A == 0 || N == 0) return TDS_OK;
    TDS_REQUIRE(d_ego_box && d_all_box && d_mask && d_grad_out && d_argmax && d_grad_ego && d_grad_all,
                "collision_allpairs_bwd: null pointer");
    TDS_REQUIRE(B <= 65535, "collision_allpairs_bwd: B=%d exceeds 65535 (shard the batch)", B);
    const dim3 grid((A + kRowsPerCta - 1) / kRowsPerCta, B);
    const size_t smem = (size_t)N * 5 * sizeof(float);
    TDS_REQUIRE(smem <= 200 * 1024, "collision_allpairs_bwd: N=%d does not fit shared memory", N);
    const auto kernel = metric == TDS_METRIC_DISCS ? allpairs_bwd_kernel<TDS_METRIC_DISCS> : allpairs_bwd_kernel<TDS_METRIC_IOU>;
    if (int e = tds::allow_dynamic_smem(kernel, smem)) return e;
    kernel<<<grid, kWarps * 32, smem, (cudaStream_t)stream>>>(d_ego_box, d_all_box, d_mask, A, N, ego_is_prefix,
                                                              d_grad_out, d_argmax, d_grad_ego, d_grad_all);
    TDS_LAUNCH_OK();
    return TDS_OK;
}
