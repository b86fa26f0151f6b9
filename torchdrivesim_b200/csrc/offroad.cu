// Offroad infraction: squared distance from the four box corners to the nearest map face.
//
// Reference: offroad_infraction_loss (torchdrivesim/infractions.py:176-229, pure-torch branch) and
// point_to_mesh_distance_pt (infractions.py:86-173), which expand the mesh to a
// [B*A*4, F, 3, 3] tensor (290 TB at 1024 x 64 agents on Town01).  Here a corner that the per-map
// distance bound places within the threshold is settled at once; the others are searched by a warp that
// walks the per-map uniform grid in expanding rings; the per-face arithmetic is the
// reference's, operation for operation (fp32, no FMA), so the minimum over the visited faces is
// the reference's minimum over all faces.  The grid (~1 MB per map) is L2 resident; HBM traffic is
// the 28 B per agent of state/size in and 4 B out.
#include <algorithm>
#include <cstdlib>
#include <math_constants.h>

#include "tds_map.cuh"

namespace {

using tds::MapDev;
using tds::MapSetDev;

struct EdgeHit {
    float d2, qx, qy;   // squared distance and closest point
};

__device__ __forceinline__ EdgeHit edge_dist2(float px, float py, float ax, float ay, float bx, float by) {
    const float abx = bx - ax, aby = by - ay;
    const float l2 = abx * abx + aby * aby;
    const float t = (abx * (px - ax) + aby * (py - ay)) / (l2 + 1e-8f);
    const float tt = fminf(fmaxf(t, 0.f), 1.f);
    EdgeHit h;
    h.qx = ax + tt * abx;
    h.qy = ay + tt * aby;
    if (l2 <= 1e-8f) { h.qx = bx; h.qy = by; }     // degenerate edge: distance to v1 (infractions.py:156-158)
    const float dx = px - h.qx, dy = py - h.qy;
    h.d2 = dx * dx + dy * dy;
    return h;
}

// infractions.py:100-169 for z = 0: 0 inside a non-degenerate triangle, else min edge distance
__device__ __forceinline__ float point_tri_dist2(float px, float py, float x0, float y0, float x1, float y1, float x2,
                                                 float y2) {
    const float ax = x2 - x0, ay = y2 - y0, bx = x1 - x0, by = y1 - y0;
    const float cz = ax * by - ay * bx;
    const float p2x = px - x0, p2y = py - y0;
    const float d00 = bx * bx + by * by;
    const float d01 = bx * ax + by * ay;
    const float d11 = ax * ax + ay * ay;
    const float d20 = p2x * bx + p2y * by;
    const float d21 = p2x * ax + p2y * ay;
    const float denom = d00 * d11 - d01 * d01 + 1e-8f;
    const float w1 = (d11 * d20 - d01 * d21) / denom;
    const float w2 = (d00 * d21 - d01 * d20) / denom;
    const float w0 = 1.0f - w1 - w2;
    const bool inside = (0.f <= w0) & (w0 <= 1.f) & (0.f <= w1) & (w1 <= 1.f) & (0.f <= w2) & (w2 <= 1.f);
    const float area = fabsf(bx * ay - by * ax) / 2.0f;
    const bool cond = inside & !(area < 5e-3f) & (fabsf(cz) > 1e-8f);
    if (cond) return 0.0f;
    const float e01 = edge_dist2(px, py, x0, y0, x1, y1).d2;
    const float e02 = edge_dist2(px, py, x0, y0, x2, y2).d2;
    const float e12 = edge_dist2(px, py, x1, y1, x2, y2).d2;
    return fminf(fminf(e01, e02), e12);
}

// squared distance from p to an axis-aligned box (0 inside)
__device__ __forceinline__ float box_dist2(float px, float py, float x0, float y0, float x1, float y1) {
    const float dx = fmaxf(fmaxf(x0 - px, px - x1), 0.0f), dy = fmaxf(fmaxf(y0 - py, py - y1), 0.0f);
    return dx * dx + dy * dy;
}

// A face (or cell) whose bounding box is further than the current best cannot lower the minimum; the
// 1e-5 relative slack covers the rounding of the reference's own distance formula.
__device__ __forceinline__ bool cannot_improve(float lower_bound2, float best) {
    return lower_bound2 > best * 1.00001f + 1e-9f;
}

// ---- nearest face of ONE point by ONE warp.  The faces of the visited cells are spread over the 32 lanes (cells are
// pruned by their box first, then a prefix sum of the cells' face counts maps a flat face index back to its cell), the
// lanes share their minimum after every round of 32 faces, so the bounding-box pruning of the next round uses it.
__device__ __forceinline__ void warp_min(float& best, int& bf) {
    // squared distances are >= 0 (or +inf) and never NaN here, so they order like their bit patterns: two warp
    // reductions (redux.sync) give the minimum and the lowest face index that attains it (-1 = none, the largest)
    const unsigned mn = __reduce_min_sync(0xffffffffu, __float_as_uint(best));
    const unsigned f = __reduce_min_sync(0xffffffffu, __float_as_uint(best) == mn ? (unsigned)bf : 0xffffffffu);
    best = __uint_as_float(mn);
    bf = (int)f;
}

// lane l proposes cell (cx, cy) (valid or not); all their faces are evaluated, 32 per round.  SINGLE: every lane
// proposes the same cell (the point's own), so a flat face index is an offset into that cell.
template <bool SINGLE>
__device__ __forceinline__ void visit_cells(const MapDev& m, bool valid, int cx, int cy, float px, float py, float stop,
                                            float& best, int& bf, int lane) {
    int e0 = 0, cnt = 0;
    if (valid) {
        // cell bounds (faces are binned with 1 mm of slack, see map.cu)
        const float x0 = m.ox0 + (float)cx * m.ocs, y0 = m.oy0 + (float)cy * m.ocs;
        if (!cannot_improve(box_dist2(px, py, x0 - 2e-3f, y0 - 2e-3f, x0 + m.ocs + 2e-3f, y0 + m.ocs + 2e-3f), best)) {
            const int c = cy * m.ogx + cx;
            e0 = __ldg(m.ocell + c);
            cnt = __ldg(m.ocell + c + 1) - e0;
        }
    }
    int incl = cnt;
    if (!SINGLE) {
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
    }
    const int excl = incl - cnt;
    const int total = SINGLE ? cnt : __shfl_sync(0xffffffffu, incl, 31);
    for (int f0 = 0; f0 < total; f0 += 32) {              // uniform over the warp
        const int f = f0 + lane;
        int e = e0 + f;
        if (!SINGLE) {
            // owner of flat face f = the last lane whose exclusive prefix is <= f
            int lo = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
                const int v = __shfl_sync(0xffffffffu, excl, lo + step);     // lo + step <= 31
                if (v <= f) lo += step;
            }
            e = __shfl_sync(0xffffffffu, e0, lo) + (f - __shfl_sync(0xffffffffu, excl, lo));
        }
        if (f < total) {
            const float4 a = __ldg(m.orec + 2 * (int64_t)e), b = __ldg(m.orec + 2 * (int64_t)e + 1);
            const float bx0 = fminf(fminf(a.x, a.z), b.x), bx1 = fmaxf(fmaxf(a.x, a.z), b.x);
            const float by0 = fminf(fminf(a.y, a.w), b.y), by1 = fmaxf(fmaxf(a.y, a.w), b.y);
            if (!cannot_improve(box_dist2(px, py, bx0, by0, bx1, by1), best)) {
                const float d = point_tri_dist2(px, py, a.x, a.y, a.z, a.w, b.x, b.y);
                const int fi = __float_as_int(b.z);
                if (d < best || (d == best && fi < bf)) { best = d; bf = fi; }
            }
        }
        warp_min(best, bf);
        if (best <= stop) return;
    }
}

// min over all faces of the map; returns the squared distance, *face = argmin (lowest face index among equal
// distances).  The search ends as soon as a face within `stop` (the threshold of the loss, >= 0) is found: the loss
// of this corner and its gradient are then 0 whatever the true minimum is (F.threshold, infractions.py:172), and the
// returned value / face are those of that face.  All 32 lanes of the warp search for the same point and return the
// same result.
__device__ float nearest_face(const MapDev& m, float px, float py, float stop, int* face, int lane) {
    float best = CUDART_INF_F;
    int bf = -1;
    if (m.nf == 0) { *face = -1; return 0.0f; }
    const float fx = floorf((px - m.ox0) * m.oinv), fy = floorf((py - m.oy0) * m.oinv);
    const int cx = (int)fminf(fmaxf(fx, -1.0e6f), 1.0e6f), cy = (int)fminf(fmaxf(fy, -1.0e6f), 1.0e6f);
    const int kmax = max(max(cx, m.ogx - 1 - cx), max(cy, m.ogy - 1 - cy));
    // first ring that touches the grid at all
    int k0 = max(max(-cx, cx - (m.ogx - 1)), max(-cy, cy - (m.ogy - 1)));
    k0 = max(k0, 0);
    // faces are binned by bounding box, so after ring k every unvisited face lies outside the square of visited
    // cells: further away than k cells plus the distance from p to the border of its own cell
    const float ux = px - (m.ox0 + (float)cx * m.ocs), uy = py - (m.oy0 + (float)cy * m.ocs);
    const float inner = fminf(fmaxf(fminf(fminf(ux, m.ocs - ux), fminf(uy, m.ocs - uy)), 0.0f), m.ocs);
    for (int k = k0; k <= kmax; k++) {
        if (k == 0) {
            visit_cells<true>(m, true, cx, cy, px, py, stop, best, bf, lane);
        } else {
            // the in-grid cells of ring k: top row, bottom row, left column, right column
            const int xa = max(cx - k, 0), xb = min(cx + k, m.ogx - 1);
            const int ya = max(cy - k + 1, 0), yb = min(cy + k - 1, m.ogy - 1);
            const int nx = max(xb - xa + 1, 0), ny = max(yb - ya + 1, 0);
            const int nt = cy - k >= 0 ? nx : 0, nb = cy + k < m.ogy ? nx : 0;
            const int nl = cx - k >= 0 ? ny : 0, nr = cx + k < m.ogx ? ny : 0;
            const int n = nt + nb + nl + nr;
            for (int i0 = 0; i0 < n; i0 += 32) {
                const int i = i0 + lane;
                int x, y;
                if (i < nt) { x = xa + i; y = cy - k; }
                else if (i < nt + nb) { x = xa + (i - nt); y = cy + k; }
                else if (i < nt + nb + nl) { x = cx - k; y = ya + (i - nt - nb); }
                else { x = cx + k; y = ya + (i - nt - nb - nl); }
                visit_cells<false>(m, i < n, x, y, px, py, stop, best, bf, lane);
                if (best <= stop) break;
            }
        }
        // (1 mm slack for the cell assignment of p itself)
        if (best <= stop) break;
        const float reach = fmaxf((float)k * m.ocs + inner - 1e-3f, 0.0f);
        if (best <= reach * reach) break;
    }
    if (!(best < CUDART_INF_F)) best = 0.0f;   // NaN position / distance: nan_to_num, infractions.py:171
    *face = bf;
    return best;
}

__device__ __forceinline__ void corner_of(const float* st, const float* lw, int k, float& px, float& py, float& s, float& c) {
    tds::sincos_cr(st[2], s, c);
    tds::box_corner(st[0], st[1], lw[0], lw[1], s, c, k, px, py);
}

// ---- distance bound of the map (MapDev::obound), built once by tds_map_create.
//
// The forward settles a corner without a search when the bound of its subcell says d2 <= thr: the loss of that corner
// is then 0 (F.threshold) whatever its exact distance.  For that, the bound must hold for the distance the search would
// compute, i.e. the reference's fp32 formula d_ref(p) = min over faces of g_f(p), g_f = 0 if the fp32 barycentric test
// says "inside", else the fp32 edge distance.  d_ref itself cannot serve at the subcell centre c: for an ill-conditioned
// face the fp32 barycentric test can say "inside" for a point metres away, so d_ref(c) = 0 would say nothing about
// the other points of the subcell.  The centre is measured instead in double precision with a distance D' that counts
// a face as a solid triangle only where the reference's inside test is reliable (below), and as its three edges
// elsewhere.  D' is a minimum of distances to closed sets, so it is 1-Lipschitz, and for p in the subcell
//   d_ref(p) <= D'(p) + kFp32Err + kInsideBand <= D'(c) + |p - c| + kFp32Err + kInsideBand,
// |p - c| <= half diagonal + kLookupErr.  The stored code is that sum rounded up to 1/64 m:
//   kLookupErr  1e-4 m: the corner is placed in its subcell from (px - x0) rounded to fp32, 3e-5 m at 400 m.
//   kFp32Err    2e-3 m: the reference's fp32 edge distance (projection, clamp, closest point, squared norm) is off the
//               exact one by a few eps times (|coordinates| + edge length), 3e-4 m for 400 m coordinates and 100 m edges.
//   kInsideBand 1e-2 m: a face is solid for D' only if its area is >= 5.05e-3 (the reference skips faces under 5e-3) and
//               the fp32 barycentric weights are accurate to dw with dw * L <= kInsideBand (L = longest edge): a point
//               inside such a face is either found inside by the reference (g = 0) or lies within dw * L of an edge.
//               The weights are ratios of products of four edge-length factors over (2 area)^2, so
//               dw <= 40 eps L^4 / (2 area)^2 + 1e-8 / (2 area)^2 (the second term is the reference's +1e-8).
// The slack, kSlack = 0.02 m, is larger than their sum; the margin it costs is small next to sqrt(thr) - half diagonal.
// Only faces binned into the offroad cells within kReach of the centre are visited: a minimum over fewer faces is
// still an upper bound, and any face nearer than the largest code that can be stored is among them.
constexpr double kSlack = 0.02, kInsideBand = 1e-2, kReach = 4.0;

__device__ double seg_dist2_d(double px, double py, double ax, double ay, double bx, double by) {
    const double abx = bx - ax, aby = by - ay, l2 = abx * abx + aby * aby;
    double t = l2 > 0.0 ? (abx * (px - ax) + aby * (py - ay)) / l2 : 0.0;
    t = fmin(fmax(t, 0.0), 1.0);
    const double dx = px - (ax + t * abx), dy = py - (ay + t * aby);
    return dx * dx + dy * dy;
}

__device__ double bound_face_dist2(double px, double py, float4 a, float4 b) {
    const double x0 = a.x, y0 = a.y, x1 = a.z, y1 = a.w, x2 = b.x, y2 = b.y;
    const double e = fmin(fmin(seg_dist2_d(px, py, x0, y0, x1, y1), seg_dist2_d(px, py, x0, y0, x2, y2)),
                          seg_dist2_d(px, py, x1, y1, x2, y2));
    const double cz = (x1 - x0) * (y2 - y0) - (y1 - y0) * (x2 - x0);      // 2 * signed area
    const double l2 = fmax(fmax((x1 - x0) * (x1 - x0) + (y1 - y0) * (y1 - y0), (x2 - x0) * (x2 - x0) + (y2 - y0) * (y2 - y0)),
                           (x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1));
    const double L = sqrt(l2), a4 = cz * cz;
    const double dw = (40.0 * 5.960464477539063e-08 * l2 * l2 + 1e-8) / a4;
    if (fabs(cz) >= 2.0 * 5.05e-3 && dw * L <= kInsideBand) {
        const double o0 = (x1 - px) * (y2 - py) - (y1 - py) * (x2 - px);
        const double o1 = (x2 - px) * (y0 - py) - (y2 - py) * (x0 - px);
        const double o2 = (x0 - px) * (y1 - py) - (y0 - py) * (x1 - px);
        const bool inside = cz > 0.0 ? (o0 >= 0.0 && o1 >= 0.0 && o2 >= 0.0) : (o0 <= 0.0 && o1 <= 0.0 && o2 <= 0.0);
        if (inside) return 0.0;
    }
    return e;                                     // NaN for a face with a non-finite vertex: ignored by the caller
}

// one thread per subcell
__global__ void __launch_bounds__(256) offroad_bound_kernel(MapDev m, uint8_t* __restrict__ obound) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)m.bgx * m.bgy) return;
    const int sx = (int)(i % m.bgx), sy = (int)(i / m.bgx);
    const double cx = (double)m.bx0 + ((double)sx + 0.5) * m.bcs, cy = (double)m.by0 + ((double)sy + 0.5) * m.bcs;
    const int ix0 = max((int)floor((cx - kReach - m.ox0) / m.ocs), 0), ix1 = min((int)floor((cx + kReach - m.ox0) / m.ocs), m.ogx - 1);
    const int iy0 = max((int)floor((cy - kReach - m.oy0) / m.ocs), 0), iy1 = min((int)floor((cy + kReach - m.oy0) / m.ocs), m.ogy - 1);
    double best = CUDART_INF;
    for (int y = iy0; y <= iy1; y++)
        for (int x = ix0; x <= ix1; x++) {
            const int c = y * m.ogx + x;
            for (int e = m.ocell[c]; e < m.ocell[c + 1]; e++) {
                const double d = bound_face_dist2(cx, cy, m.orec[2 * (int64_t)e], m.orec[2 * (int64_t)e + 1]);
                if (d < best) best = d;
            }
        }
    const double ub = sqrt(best) + 0.7071067811865476 * m.bcs + kSlack;          // +inf when no face was near
    const double q = ceil(ub * tds::kBoundPerMetre);
    obound[i] = q < (double)tds::kBoundUnknown ? (uint8_t)q : (uint8_t)tds::kBoundUnknown;
}

// the corner's squared distance is known to be <= thr from its subcell's bound (false for NaN, outside the grid, thr <= 0)
__device__ __forceinline__ bool settled_by_bound(const MapDev& m, float px, float py, float thr) {
    const float fx = (px - m.bx0) * m.binv, fy = (py - m.by0) * m.binv;
    if (!(fx >= 0.0f && fy >= 0.0f && fx < (float)m.bgx && fy < (float)m.bgy)) return false;
    const int q = __ldg(m.obound + (int64_t)(int)fy * m.bgx + (int)fx);
    return q < tds::kBoundUnknown && (float)(q * q) <= thr * (float)(tds::kBoundPerMetre * tds::kBoundPerMetre);
}

// A warp holds 8 agents, lane l = corner l & 3 of agent 8 * group + l / 4.  Each lane places its corner and looks up the
// map's distance bound: a corner whose bound is within the threshold is settled (value 0, face -1, the search would
// have stopped at a face with d2 <= thr and returned 0 too).  The warp then searches the undecided corners one after
// another with nearest_face, all 32 lanes on one corner.  Face -1 for a settled corner is what the backward needs: it
// skips f < 0, and with the face of the search it would have skipped the corner as well (d2 <= thr); FusedRollout goes
// through the same backward, and nothing else reads the face.  triage = false (TDS_OFFROAD_TRIAGE=0) searches every
// corner: the values are the same, the faces of on-road corners are those of the search.
#ifndef TDS_OFFROAD_MINB
#define TDS_OFFROAD_MINB 4
#endif
__global__ void __launch_bounds__(256, TDS_OFFROAD_MINB) offroad_fwd_kernel(MapSetDev maps, const int32_t* __restrict__ env_map,
                                                          const float* __restrict__ state, const float* __restrict__ lenwid,
                                                          const uint8_t* __restrict__ present, int B, int A, float thr, bool triage,
                                                          float* __restrict__ out, int32_t* __restrict__ face) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, k = lane & 3;
    const unsigned n_agents = (unsigned)B * (unsigned)A;          // < 2^31, checked by the host
    const unsigned n_groups = (n_agents + 7) / 8;
    const unsigned n_warps = gridDim.x * (blockDim.x >> 5);
    for (unsigned g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); g < n_groups; g += n_warps) {
        const unsigned agent = 8 * g + (lane >> 2);
        const bool valid = agent < n_agents;
        const bool here = valid && (present ? present[agent] != 0 : true);
        float v = 0.0f, px = 0.0f, py = 0.0f;
        int bf = -1, mi = 0;
        bool search = false;
        if (here) {
            float s, c;
            corner_of(state + 4 * (size_t)agent, lenwid + 2 * (size_t)agent, k, px, py, s, c);
            mi = env_map ? env_map[agent / (unsigned)A] : 0;
            search = !(triage && settled_by_bound(maps.m[mi], px, py, thr));
        }
        for (unsigned todo = __ballot_sync(full, search); todo; todo &= todo - 1) {
            const int src = __ffs(todo) - 1;
            const int smi = __shfl_sync(full, mi, src);
            const float sx = __shfl_sync(full, px, src), sy = __shfl_sync(full, py, src);
            int sf;
            const float d2 = nearest_face(maps.m[smi], sx, sy, fmaxf(thr, 0.0f), &sf, lane);
            if (lane == src) {
                v = d2 > thr ? d2 : 0.0f;           // F.threshold(d2, thr, 0), infractions.py:172
                bf = sf;
            }
        }
        if (valid && face) face[4 * (size_t)agent + k] = bf;
        // sum of the 4 corners, in corner order
        const int c0 = lane & ~3;
        const float v0 = __shfl_sync(full, v, c0), v1 = __shfl_sync(full, v, c0 + 1);
        const float v2 = __shfl_sync(full, v, c0 + 2), v3 = __shfl_sync(full, v, c0 + 3);
        if (valid && k == 0) out[agent] = ((v0 + v1) + v2) + v3;
    }
}

__global__ void __launch_bounds__(128) offroad_bwd_kernel(MapSetDev maps, const int32_t* __restrict__ env_map,
                                                          const float* __restrict__ state, const float* __restrict__ lenwid,
                                                          const uint8_t* __restrict__ present, int B, int A, float thr,
                                                          const int32_t* __restrict__ face, const float* __restrict__ gout,
                                                          float* __restrict__ g_state, float* __restrict__ g_lenwid) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t agent = t >> 2;
    const int k = (int)(t & 3);
    const bool valid = agent < (int64_t)B * A;
    float gx = 0.f, gy = 0.f, gpsi = 0.f, gl = 0.f, gw = 0.f;
    if (valid) {
        const int b = (int)(agent / A);
        const bool here = present ? present[agent] != 0 : true;
        const int f = face[t];
        if (here && f >= 0) {
            const MapDev& m = maps.m[env_map ? env_map[b] : 0];
            const float* st = state + 4 * agent;
            const float* lw = lenwid + 2 * agent;
            float px, py, s, c;
            corner_of(st, lw, k, px, py, s, c);
            const float2* tr = reinterpret_cast<const float2*>(m.tri + 6 * (size_t)f);
            const float2 v0 = tr[0], v1 = tr[1], v2 = tr[2];
            const float d2 = point_tri_dist2(px, py, v0.x, v0.y, v1.x, v1.y, v2.x, v2.y);
            if (d2 > thr) {
                // d2 is the smallest of the three edge distances; d d2 / d p = 2 (p - q)
                EdgeHit h = edge_dist2(px, py, v0.x, v0.y, v1.x, v1.y);
                const EdgeHit h2 = edge_dist2(px, py, v0.x, v0.y, v2.x, v2.y);
                const EdgeHit h3 = edge_dist2(px, py, v1.x, v1.y, v2.x, v2.y);
                if (h2.d2 < h.d2) h = h2;
                if (h3.d2 < h.d2) h = h3;
                const float g = gout[agent];
                const float dpx = 2.0f * (px - h.qx) * g, dpy = 2.0f * (py - h.qy) * g;
                const float sx = (k == 0 || k == 3) ? 0.5f : -0.5f;
                const float sy = (k < 2) ? 0.5f : -0.5f;
                const float ux = sx * lw[0], uy = sy * lw[1];
                gx = dpx;
                gy = dpy;
                gpsi = dpx * (-ux * s - uy * c) + dpy * (ux * c - uy * s);
                gl = sx * (dpx * c + dpy * s);
                gw = sy * (dpy * c - dpx * s);
            }
        }
    }
    const unsigned full = 0xffffffffu;
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
        gx += __shfl_xor_sync(full, gx, o);
        gy += __shfl_xor_sync(full, gy, o);
        gpsi += __shfl_xor_sync(full, gpsi, o);
        gl += __shfl_xor_sync(full, gl, o);
        gw += __shfl_xor_sync(full, gw, o);
    }
    if (valid && k == 0) {
        if (g_state) reinterpret_cast<float4*>(g_state)[agent] = make_float4(gx, gy, gpsi, 0.0f);
        if (g_lenwid) reinterpret_cast<float2*>(g_lenwid)[agent] = make_float2(gl, gw);
    }
}

}  // namespace

extern "C" int tds_offroad_fwd(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                               const float* d_state, const float* d_lenwid, const uint8_t* d_present,
                               int32_t B, int32_t A, float threshold, float* d_out, int32_t* d_face, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0, "offroad: negative size");
    if (B == 0 || A == 0) return TDS_OK;
    TDS_REQUIRE(d_state && d_lenwid && d_out, "offroad: null pointer");
    MapSetDev set;
    if (int e = tds::gather_maps(maps, n_maps, set)) return e;
    // groups of 8 agents are dealt round-robin to the warps of a grid that holds them all at once for the benchmark's
    // 65 536 agents (a warp whose corners are all settled is done after a few hundred cycles)
    TDS_REQUIRE((int64_t)B * A <= 2147483647LL, "offroad: too many agents");
    const int64_t groups = ((int64_t)B * A + 7) / 8;
    const int64_t grid = std::min<int64_t>((groups + 7) / 8, (int64_t)tds::sm_count() * 16);
    bool triage = true;
    if (const char* e = getenv("TDS_OFFROAD_TRIAGE")) triage = atoi(e) != 0;      // test hook: search every corner
    offroad_fwd_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(
        set, d_env_map, d_state, d_lenwid, d_present, B, A, threshold, triage, d_out, d_face);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

extern "C" int tds_offroad_bwd(const tds_map_t* const* maps, int32_t n_maps, const int32_t* d_env_map,
                               const float* d_state, const float* d_lenwid, const uint8_t* d_present,
                               int32_t B, int32_t A, float threshold, const int32_t* d_face, const float* d_grad_out,
                               float* d_grad_state, float* d_grad_lenwid, void* stream) {
    TDS_REQUIRE(B >= 0 && A >= 0, "offroad_bwd: negative size");
    if (B == 0 || A == 0) return TDS_OK;
    TDS_REQUIRE(d_state && d_lenwid && d_face && d_grad_out, "offroad_bwd: null pointer");
    MapSetDev set;
    if (int e = tds::gather_maps(maps, n_maps, set)) return e;
    const int64_t threads = (int64_t)B * A * 4;
    offroad_bwd_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        set, d_env_map, d_state, d_lenwid, d_present, B, A, threshold, d_face, d_grad_out, d_grad_state, d_grad_lenwid);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

int tds::offroad_bound_build(const MapDev& d, uint8_t* obound) {
    const int64_t n = (int64_t)d.bgx * d.bgy;
    if (d.nf == 0) {                             // nothing to bound: every corner takes the search, which returns at once
        TDS_CUDA_OK(cudaMemset(obound, kBoundUnknown, (size_t)n));
        return TDS_OK;
    }
    offroad_bound_kernel<<<(unsigned)((n + 255) / 256), 256>>>(d, obound);
    TDS_LAUNCH_OK();
    TDS_CUDA_OK(cudaStreamSynchronize(0));
    return TDS_OK;
}
