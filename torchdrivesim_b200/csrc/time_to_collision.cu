// Time to collision: the first contact of every origin agent with any other present agent when every agent keeps its
// heading and speed (tds_time_to_collision), and the gradient of that time with respect to the states and sizes of
// the two agents of each contact (tds_time_to_collision_bwd).
//
// Pair (i, j), float32, every operation rounded on its own (-fmad=false), IEEE division.  Agent k: (s_k, c_k) =
// sincos_cr(psi_k), velocity (v_k c_k, v_k s_k), half-extents hl_k = 0.5 length_k, hw_k = 0.5 width_k.  Axes in this
// order: u_i = (c_i, s_i), u_i⊥ = (-s_i, c_i), u_j, u_j⊥.  On axis n: d0 = n·(xy_j - xy_i), s = n·(v_j - v_i), and
// R = h_i + h_j, where a box's half-extent is hl (hw) on its own u (u⊥) and |n·u| hl + |n·u⊥| hw on the other's axes.
// s != 0: entry / exit = min / max of (-R - d0) / s and (R - d0) / s;  s == 0: (-inf, inf) if |d0| <= R, else no
// contact.  T_in = max of the entries, T_out = min of the exits (a NaN entry or exit: no contact); contact within H iff
// max(T_in, 0) <= min(T_out, H), at time T_in > 0 ? T_in : +0.  The winner of a row is the smallest
// (bits(t) << 32 | j): t >= 0 orders like its bits.
#include <math_constants.h>

#include <algorithm>
#include <cmath>
#include <cstdint>

#include "tds_colsum.cuh"
#include "tds_common.cuh"
#include "tds_nearest.cuh"

namespace {

using tds::kNearEmpty;

constexpr int kTtcWarps = 8;        // warps per CTA of both kernels
constexpr int kTtcRows = 64;        // origin rows per CTA of the forward, 8 per warp
constexpr int kTtcTile = 1024;      // columns staged in shared memory at a time by the forward
constexpr int kTtcStride = 11;      // floats per staged agent (odd: conflict-free column reads)

// What both kernels need of an agent, in the staged order.
struct TtcAgent {
    float x, y, c, s, vx, vy, hl, hw, r, sp, present;
};

__device__ __forceinline__ void ttc_stage(const float* __restrict__ state, const float* __restrict__ size,
                                          const uint8_t* __restrict__ present, int64_t e, float* __restrict__ d) {
    const float4 st = *reinterpret_cast<const float4*>(state + e * 4);
    const float2 sz = *reinterpret_cast<const float2*>(size + e * 2);
    float s, c;
    tds::sincos_cr(st.z, s, c);
    d[0] = st.x;
    d[1] = st.y;
    d[2] = c;
    d[3] = s;
    d[4] = st.w * c;
    d[5] = st.w * s;
    d[6] = 0.5f * sz.x;
    d[7] = 0.5f * sz.y;
    d[8] = 0.5f * sqrtf(sz.x * sz.x + sz.y * sz.y);     // circumradius (broad phase only)
    d[9] = fabsf(st.w);                                 // speed (broad phase only)
    d[10] = present[e] ? 1.0f : 0.0f;
}

__device__ __forceinline__ TtcAgent ttc_agent(const float* d) {
    return TtcAgent{d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7], d[8], d[9], d[10]};
}

__device__ __forceinline__ TtcAgent ttc_agent(const float* __restrict__ state, const float* __restrict__ size,
                                              const uint8_t* __restrict__ present, int64_t e) {
    float d[kTtcStride];
    ttc_stage(state, size, present, e, d);
    return ttc_agent(d);
}

// Axis k of the pair (0: u_i, 1: u_i⊥, 2: u_j, 3: u_j⊥) and what the contact time on it depends on.
struct TtcAxis {
    float nx, ny;    // the axis
    float p, q;      // n·u and n·u⊥ of the agent that does not own the axis
    float d0, sv, R;
};

__device__ __forceinline__ TtcAxis ttc_axis(const TtcAgent& I, const TtcAgent& J, int k) {
    const TtcAgent& own = k < 2 ? I : J;
    const TtcAgent& oth = k < 2 ? J : I;
    TtcAxis a;
    a.nx = (k & 1) ? -own.s : own.c;
    a.ny = (k & 1) ? own.c : own.s;
    a.p = a.nx * oth.c + a.ny * oth.s;
    a.q = a.nx * (-oth.s) + a.ny * oth.c;
    const float h_own = (k & 1) ? own.hw : own.hl;
    const float h_oth = fabsf(a.p) * oth.hl + fabsf(a.q) * oth.hw;
    a.R = k < 2 ? h_own + h_oth : h_oth + h_own;                    // h_i + h_j
    a.d0 = a.nx * (J.x - I.x) + a.ny * (J.y - I.y);
    a.sv = a.nx * (J.vx - I.vx) + a.ny * (J.vy - I.vy);
    return a;
}

// The contact time of the pair within [0, H], or -1 for no contact; `axis` gets the first axis whose entry is T_in.
__device__ __forceinline__ float ttc_pair(const TtcAgent& I, const TtcAgent& J, float H, int& axis) {
    float tin = -CUDART_INF_F, tout = CUDART_INF_F;
    bool nan = false;
    axis = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const TtcAxis a = ttc_axis(I, J, k);
        float en, ex;
        if (a.sv != 0.0f) {                                          // true for a NaN s
            const float ta = (-a.R - a.d0) / a.sv, tb = (a.R - a.d0) / a.sv;
            nan |= ta != ta || tb != tb;
            en = fminf(ta, tb);
            ex = fmaxf(ta, tb);
        } else {
            if (!(fabsf(a.d0) <= a.R)) return -1.0f;
            en = -CUDART_INF_F;
            ex = CUDART_INF_F;
        }
        if (en > tin) {
            tin = en;
            axis = k;
        }
        tout = fminf(tout, ex);
    }
    if (nan || !(fmaxf(tin, 0.0f) <= fminf(tout, H))) return -1.0f;
    return tin > 0.0f ? tin : 0.0f;
}

// Broad phase: true when the pair cannot touch within [0, H], so the SAT test above would find no contact.
// In real arithmetic, boxes that touch at time t have centres at most r_i + r_j apart (r the circumradius), so a pair
// whose centre offset D(t) = Δc + t Δv stays farther than that over [0, H] never touches.  The float SAT can accept a
// time t* a little outside the real contact: d0, s and R carry a few ulps relative to |Δc|, |v_i| + |v_j| and R, and
// the divisions and the bound t* <= H turn that into |n·D(t*)| <= R + e on every axis with
// e <= ~20 u (r_i + r_j + |Δc| + H (|v_i| + |v_j|)), u = 2^-24.  Boxes whose half-extents are widened by e overlap then
// (their projections grow by >= e on every unit axis), so |D(t*)| <= r_i + r_j + 1.5 e.  The closest point of the
// segment, evaluated at a rounded time in float32, errs by a few u of the same terms.  The bound below is wider than
// all of it by two orders of magnitude: 1e-4 (~1700 u) of those terms, and on top the IoU test's 1.0001 x + 1e-6 on
// the square.  Any non-finite input gives no rejection (a NaN comparison is false, an infinite offset meets an
// infinite bound), and negative sizes only shrink the SAT extents, which the absolute values in r cover.
__device__ __forceinline__ bool ttc_far(const TtcAgent& I, const TtcAgent& J, float H) {
    const float dx = J.x - I.x, dy = J.y - I.y, dvx = J.vx - I.vx, dvy = J.vy - I.vy;
    const float vv = dvx * dvx + dvy * dvy;
    float tc = 0.0f;
    if (vv > 0.0f) {
        tc = -(dx * dvx + dy * dvy) / vv;
        if (!isfinite(tc)) return false;
        tc = fminf(fmaxf(tc, 0.0f), H);
    }
    const float ex = dx + tc * dvx, ey = dy + tc * dvy;
    const float d2 = ex * ex + ey * ey;
    const float reach = (I.r + J.r) * 1.0001f + 1e-4f * (fabsf(dx) + fabsf(dy) + H * (I.sp + J.sp));
    return d2 > reach * reach * 1.0001f + 1e-6f;
}

// Forward: a CTA per (environment, 64 origin rows), 8 warps, rows r = warp, warp + 8, ... of the tile to each warp,
// the lanes over the columns.  The CTA's origins and then the environment's columns, kTtcTile at a time, are staged in
// shared memory (stride 11).  Each lane keeps the smallest word of its columns per row in registers; the row minimum
// is taken by shuffles after the last tile.
__global__ void __launch_bounds__(kTtcWarps * 32) ttc_fwd_kernel(const float* __restrict__ state,
                                                                 const float* __restrict__ size,
                                                                 const uint8_t* __restrict__ present, int A, int N,
                                                                 float H, float* __restrict__ ttc,
                                                                 int64_t* __restrict__ idx) {
    extern __shared__ float s_col[];                                 // [tile][kTtcStride]
    __shared__ float s_org[kTtcRows * kTtcStride];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t b = blockIdx.y;
    const int row0 = blockIdx.x * kTtcRows;
    const int64_t base = b * N;
    for (int q = threadIdx.x; q < kTtcRows; q += blockDim.x)
        if (row0 + q < A) ttc_stage(state, size, present, base + row0 + q, s_org + q * kTtcStride);
    unsigned long long best[kTtcRows / kTtcWarps];
#pragma unroll
    for (int rr = 0; rr < kTtcRows / kTtcWarps; rr++) best[rr] = kNearEmpty;
    for (int t0 = 0; t0 < N; t0 += kTtcTile) {
        const int nt = min(kTtcTile, N - t0);
        __syncthreads();                                             // the previous tile is consumed
        for (int q = threadIdx.x; q < nt; q += blockDim.x) ttc_stage(state, size, present, base + t0 + q, s_col + q * kTtcStride);
        __syncthreads();
#pragma unroll
        for (int rr = 0; rr < kTtcRows / kTtcWarps; rr++) {
            const int r = warp + rr * kTtcWarps;
            const int i = row0 + r;
            if (i >= A || s_org[r * kTtcStride + 10] == 0.0f) continue;   // warp-uniform
            const TtcAgent I = ttc_agent(s_org + r * kTtcStride);
            for (int q = lane; q < nt; q += 32) {
                const int j = t0 + q;
                const float* cj = s_col + q * kTtcStride;
                if (j == i || cj[10] == 0.0f) continue;
                const TtcAgent J = ttc_agent(cj);
                if (ttc_far(I, J, H)) continue;
                int axis;
                const float t = ttc_pair(I, J, H, axis);
                if (t >= 0.0f) {
                    const unsigned long long w = ((unsigned long long)__float_as_uint(t) << 32) | (unsigned)j;
                    best[rr] = w < best[rr] ? w : best[rr];
                }
            }
        }
    }
#pragma unroll
    for (int rr = 0; rr < kTtcRows / kTtcWarps; rr++) {
        const int i = row0 + warp + rr * kTtcWarps;
        unsigned long long w = best[rr];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long v = __shfl_xor_sync(0xffffffffu, w, o);
            w = v < w ? v : w;
        }
        if (lane == 0 && i < A) {
            const int64_t e = b * A + i;
            ttc[e] = w == kNearEmpty ? CUDART_INF_F : __uint_as_float((unsigned)(w >> 32));
            idx[e] = w == kNearEmpty ? -1 : (int64_t)(unsigned)w;
        }
    }
}

// The 12 gradient terms of one contact at time t > 0 on axis k, for upstream gradient g: go[6] of the origin i and
// gj[6] of agent j, each (x, y, psi, v, length, width).  With t = -(d0 + sgn(s) R) / s:
//   dt/dd0 = -1/s, dt/dR = -1/|s|, dt/ds = -t/s,
// chained through d0 = n·(xy_j - xy_i), s = n·(v_j - v_i) with v = (v c, v s), R = h_own + |p| hl_oth + |q| hw_oth
// (p = n·u_oth, q = n·u_oth⊥, d|x|/dx = sgn(x), 0 at 0), and n, which turns with psi of the axis' owner (dn/dpsi =
// (-ny, nx)).
__device__ __forceinline__ void ttc_pair_grad(const TtcAgent& I, const TtcAgent& J, int k, float t, float g,
                                              float* __restrict__ go, float* __restrict__ gj) {
    const TtcAxis a = ttc_axis(I, J, k);
    const float gd0 = -g / a.sv, gR = -g / fabsf(a.sv), gs = -(g * t) / a.sv;
    const float gx = gd0 * a.nx, gy = gd0 * a.ny;                   // d xy_j; d xy_i is its negative
    const float gvx = gs * a.nx, gvy = gs * a.ny;                   // d v_j (vector); d v_i is its negative
    float gnx = gd0 * (J.x - I.x) + gs * (J.vx - I.vx);
    float gny = gd0 * (J.y - I.y) + gs * (J.vy - I.vy);
    const TtcAgent& oth = k < 2 ? J : I;
    const float sp = a.p > 0.0f ? 1.0f : (a.p < 0.0f ? -1.0f : 0.0f);
    const float sq = a.q > 0.0f ? 1.0f : (a.q < 0.0f ? -1.0f : 0.0f);
    const float gp = gR * oth.hl * sp, gq = gR * oth.hw * sq;
    gnx += gp * oth.c + gq * (-oth.s);
    gny += gp * oth.s + gq * oth.c;
    go[0] = -gx;
    go[1] = -gy;
    go[2] = gvx * I.vy - gvy * I.vx;                                 // -(gvx (-vy) + gvy vx): the velocity turns with psi
    go[3] = -(gvx * I.c + gvy * I.s);
    go[4] = go[5] = 0.0f;
    gj[0] = gx;
    gj[1] = gy;
    gj[2] = gvy * J.vx - gvx * J.vy;
    gj[3] = gvx * J.c + gvy * J.s;
    gj[4] = gj[5] = 0.0f;
    float* gown = k < 2 ? go : gj;
    float* goth = k < 2 ? gj : go;
    gown[2] += gny * a.nx - gnx * a.ny;                              // the axis turns with its owner
    gown[(k & 1) ? 5 : 4] += 0.5f * gR;                              // h_own = hl or hw
    goth[2] += gp * a.q - gq * a.p;                                  // dp/dpsi = q, dq/dpsi = -p
    goth[4] += 0.5f * (gR * fabsf(a.p));
    goth[5] += 0.5f * (gR * fabsf(a.q));
}

// Backward: one CTA per environment, a tds::ColSums column sum (tds_colsum.cuh) over (x, y, psi, v, length, width).
// Each warp takes origin rows 32 at a time (rows 32 (8 m + warp) + lane).  A lane recomputes its row's contact with
// agent idx (and so its axis) from the inputs; a row whose contact is not at a time in (0, H] (ttc == 0, idx == -1, an
// index that is not another present agent) is skipped by a branch, so an inf or NaN upstream value there reaches
// nothing.  The rows' 12 terms are added to the accumulator by tds::add_lane_serial, one row after the other (origin
// terms by lanes 0-5, hit-agent terms by lanes 6-11; i != j, so they never meet in one step).
__global__ void __launch_bounds__(kTtcWarps * 32) ttc_bwd_kernel(const float* __restrict__ state,
                                                                 const float* __restrict__ size,
                                                                 const uint8_t* __restrict__ present,
                                                                 const float* __restrict__ gout,
                                                                 const int64_t* __restrict__ idx, int A, int N,
                                                                 float H, int cols, float* __restrict__ gstate,
                                                                 float* __restrict__ gsize) {
    extern __shared__ float s_acc[];                                 // [kTtcWarps][cols][6]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t b = blockIdx.x;
    const int64_t base = b * N;
    const tds::ColSums<kTtcWarps, 6> sums(s_acc, cols, warp);
    for (int n0 = 0; n0 < N; n0 += cols) {
        const int nc = min(cols, N - n0);
        sums.zero(nc, lane);
        for (int i0 = warp * 32; i0 < A; i0 += kTtcWarps * 32) {
            const int i = i0 + lane;
            int cl[2] = {-1, -1};                                    // the columns of the origin and hit-agent terms
            float v[12];
#pragma unroll
            for (int c = 0; c < 12; c++) v[c] = 0.0f;
            if (i < A) {
                const int64_t e = b * A + i;
                const int64_t j = idx[e];
                const bool own = i >= n0 && i < n0 + nc;
                const bool col = j >= n0 && j < n0 + nc;
                if (j >= 0 && j < N && j != i && (own || col) && present[base + i] && present[base + j]) {
                    const TtcAgent I = ttc_agent(state, size, present, base + i);
                    const TtcAgent J = ttc_agent(state, size, present, base + j);
                    int axis;
                    const float t = ttc_pair(I, J, H, axis);
                    if (t > 0.0f) {
                        ttc_pair_grad(I, J, axis, t, gout[e], v, v + 6);
                        cl[0] = own ? i : -1;
                        cl[1] = col ? (int)j : -1;
                    }
                }
            }
            tds::add_lane_serial<6, 2>(sums.acc, n0, cl, v, lane);
        }
        __syncthreads();
        for (int q = threadIdx.x; q < 6 * nc; q += blockDim.x) {
            const int n = q / 6, comp = q - n * 6;
            const float s = sums.total(n, comp);
            const int64_t e = base + n0 + n;
            if (comp < 4) gstate[e * 4 + comp] = s;
            else gsize[e * 2 + comp - 4] = s;
        }
        __syncthreads();
    }
}

}  // namespace

extern "C" int tds_time_to_collision(const float* d_state, const float* d_size, const uint8_t* d_present, int32_t B,
                                     int32_t A, int32_t N, float horizon, float* d_ttc, int64_t* d_idx, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "time_to_collision: need 0 <= A <= N");
    TDS_REQUIRE(std::isfinite(horizon) && horizon > 0.0f, "time_to_collision: the horizon must be finite and > 0");
    if ((int64_t)B * A == 0) return TDS_OK;
    TDS_REQUIRE(d_state && d_size && d_present && d_ttc && d_idx, "time_to_collision: null pointer");
    TDS_REQUIRE(B <= 65535, "time_to_collision: at most 65535 environments");
    const dim3 grid((unsigned)((A + kTtcRows - 1) / kTtcRows), (unsigned)B);
    const size_t smem = (size_t)std::min(N, kTtcTile) * kTtcStride * sizeof(float);
    ttc_fwd_kernel<<<grid, kTtcWarps * 32, smem, (cudaStream_t)stream>>>(d_state, d_size, d_present, A, N, horizon,
                                                                        d_ttc, d_idx);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_time_to_collision_bwd(const float* d_state, const float* d_size, const uint8_t* d_present, int32_t B,
                                         int32_t A, int32_t N, float horizon, const float* d_grad_ttc,
                                         const int64_t* d_idx, float* d_grad_state, float* d_grad_size, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0 && N >= 0 && A <= N, "time_to_collision_bwd: need 0 <= A <= N");
    TDS_REQUIRE(std::isfinite(horizon) && horizon > 0.0f, "time_to_collision_bwd: the horizon must be finite and > 0");
    if ((int64_t)B * N == 0) return TDS_OK;
    TDS_REQUIRE(d_state && d_size && d_present && d_grad_state && d_grad_size && (A == 0 || (d_grad_ttc && d_idx)),
                "time_to_collision_bwd: null pointer");
    const int cols = std::min(N, tds::kColsPerPass);
    const size_t smem = (size_t)kTtcWarps * cols * 6 * sizeof(float);
    if (int e = tds::allow_dynamic_smem(ttc_bwd_kernel, smem)) return e;
    ttc_bwd_kernel<<<(unsigned)B, kTtcWarps * 32, smem, (cudaStream_t)stream>>>(d_state, d_size, d_present, d_grad_ttc,
                                                                               d_idx, A, N, horizon, cols, d_grad_state,
                                                                               d_grad_size);
    TDS_LAUNCH_OK();
    return TDS_OK;
}
