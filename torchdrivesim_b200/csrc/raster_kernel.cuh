// Birdview rasteriser, pixel-identical to the reference's cv2 backend.
//
// Reference pipeline replaced here (per camera):
//   BirdviewRGBMeshGenerator.generate      torchdrivesim/mesh.py:1053-1157  (scene assembly; 1.86 MB per camera)
//   BirdviewRenderer.render_frame          torchdrivesim/rendering/base.py:167-204
//   CV2Renderer.render_rgb_mesh            torchdrivesim/rendering/cv2.py:27-70
//     translate -> trim to the 1.05x view quad (mesh.py:308-348, utils.py:99-122) -> painter's order by z
//     -> project + truncate to int32 -> cv2.fillConvexPoly per triangle -> transpose
//
// Design (DESIGN.md section 4 has the measurements behind every choice)
//   * persistent grid; a warp (tiles <= 96x96) or a CTA of independent warps (larger tiles) pulls cameras from a
//     global counter;
//   * the static mesh is never expanded per camera: the candidates of a camera are the records of the grid cells
//     its view quad's bounding box touches - one contiguous range per grid row;
//   * ONE pass over the candidates; painter's order is kept in per-class BITPLANES (one bit per pixel and draw
//     rank, shared memory, red.shared.or), resolved once at the end and expanded through a colour LUT;
//   * stage 1S - STRIPS (4 faces over 6 vertices, one record, one thread: lane markings and road surfaces): six
//     projections instead of twelve; every in-image vertex of a kept face is a covered pixel (the outline contains its
//     end points), so the six vertices are plotted at once and only faces whose bounding box exceeds 2x2 pixels go on;
//     64x64 tiles: the two quads of a strip whose shape is in the coverage-pattern table (tds_quad_table.h) are queued
//     as ONE item each, drawn by OR-ing the rows of the pattern;
//   * stage 1F - single faces (dynamic primitives, faces outside strips): cull + project + truncate, plotted (<= 2x2
//     pixels) or queued by kind (inside the image, crossing the border);
//   * stage 2 - whenever a queue holds 32 items: one face per thread, the cv2 rule per image row in closed form
//     (tds_raster_rows.h), one 64-bit row mask = at most two atomic ORs per row; faces that cross the border: four
//     lanes per face;
//   * the planes are stored x-major, which IS the reference's final transpose (cv2.py:61); the image leaves as
//     streaming 128-bit stores (float32, the reference's dtype) or as uint8 RGB / uint8 draw rank;
//   * 64x64 tiles run as TWO kernels (PHASE 1 of raster_kernel = draw, raster_finish_kernel = border-crossing faces +
//     resolve) that hand the bitplanes over in memory: each program fits the 32 KB instruction cache of an SM, the
//     one-pass program does not and loses a third of its issue slots to instruction fetch.
// HBM traffic per camera: 12 * res^2 bytes of float32 image out (49 KB at 64x64); the map records are L2 hits.
#pragma once
#include <algorithm>
#include <cstdlib>

#include "tds_map.cuh"
#include "tds_raster_tri.h"
#include "tds_raster_rows.h"
#include "tds_quad_table.h"

namespace tds_raster {

using tds::kMaxRasterRows;
using tds::MapDev;
using tds::MapSetDev;



struct PaletteDev {
    int32_t n_classes;
    int32_t order[TDS_MAX_CLASSES];               // classes in draw order
    float rgb[TDS_MAX_CLASSES + 1][3];            // [0] = background
    int32_t agent_type_class[TDS_MAX_AGENT_TYPES];
    int32_t direction_class;
    int32_t tl_state_class[TDS_MAX_TL_STATES];
    uint32_t dyn_mask;                            // classes that dynamic primitives may carry
    int8_t plane_of_class[TDS_MAX_CLASSES];       // draw rank (plane) of every class, -1: inactive (filled by the host)
};

// ceil(2^32 / (2 dy)) for dy <= 1024 (tds::row_rcp), evaluated by the compiler: the kernels copy the entries they need
// into shared memory instead of carrying division code in their prologue
struct RcpTable { uint32_t v[1025]; };
constexpr RcpTable make_rcp_table() {
    RcpTable t{};
    for (int i = 1; i <= 1024; i++) t.v[i] = 0xffffffffu / (uint32_t)(2 * i) + 1u;
    return t;
}
static __device__ const RcpTable g_rcp = make_rcp_table();


// workspace layout per environment: float tri[T][6] followed by uint8 cls[Tpad]
__host__ __device__ inline int64_t ws_env_bytes(int T) { return (int64_t)T * 24 + ((T + 15) / 16) * 16; }

// ------------------------------------------------------------------ camera
struct Camera {
    float ncx, ncy;            // -camera position
    float S, C, scale, fmin, half;
    float kscale;              // -(scale * res / 2), exact for power-of-two res
    float r_in, r_out;         // max-norm radii (pixels) deciding "inside / outside the 1.05x quad" away from its boundary
    int res;
};

__device__ __forceinline__ void make_camera(Camera& cam, float cx, float cy, float S, float C, float scale, int res) {
    cam.ncx = -cx; cam.ncy = -cy; cam.S = S; cam.C = C; cam.scale = scale; cam.res = res;
    cam.fmin = (float)res;
    cam.half = (float)res / 2.0f;
    cam.kscale = -(scale * cam.half);
    // fp32 disagreement between the pixel-space and the edge-function test is < 1e-4 m; band = 0.01 px + 2e-3 m
    const float band = 0.01f + 0.002f * (scale * cam.half);
    cam.r_in = 0.525f * cam.fmin - band;
    cam.r_out = 0.525f * cam.fmin + band;
}

// The reference's own test of a camera-relative point against the 1.05x view quad: rendering/cv2.py:34-40 with
// base.py:117-130 (cameras.xy is zero after the translate) for the quad, utils.py:99-122 for the edge functions, all
// in its fp32 operation order.  Only vertices within the thin band around the quad's boundary get here (a handful
// per camera), so the quad is rebuilt on every call instead of living in registers or shared memory: the routine
// stays out of the instruction-cache footprint of the main loop.
static __device__ __noinline__ bool inside_quad(float S, float C, float scale, int res, float x, float y) {
    const float half = (float)res / 2.0f;
    const float cxs[4] = {0.f, 0.f, (float)res, (float)res};
    const float cys[4] = {0.f, (float)res, (float)res, 0.f};
    float qx[4], qy[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        float px = cxs[i] - half, py = cys[i] - half;
        px = px / half; py = py / half;
        px = (-px) / scale; py = (-py) / scale;
        qx[i] = (C * px + (-S) * py) + 0.0f;
        qy[i] = (S * px + C * py) + 0.0f;
    }
    const float mx = (((qx[0] + qx[1]) + qx[2]) + qx[3]) / 4.0f;
    const float my = (((qy[0] + qy[1]) + qy[2]) + qy[3]) / 4.0f;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        qx[i] = mx + (qx[i] - mx) * 1.05f;
        qy[i] = my + (qy[i] - my) * 1.05f;
    }
    int nr = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int j = (i + 1) & 3;
        const float ea = qy[j] - qy[i], eb = qx[i] - qx[j];
        const float ec = (-ea) * qx[i] - eb * qy[i];
        nr += ((ea * x + eb * y) + ec) >= 0.0f;
    }
    return nr == 4 || nr == 0;
}
__device__ __forceinline__ bool inside_quad(const Camera& cam, float x, float y) {
    return inside_quad(cam.S, cam.C, cam.scale, cam.res, x, y);
}

// ---- stage 1: cull (mesh.py:311-313) + project one world-space triangle --------------------------
// Pixel-space shortcut for the cull: the 1.05x view quad is the image square scaled by 1.05 about its
// centre, i.e. the max-norm ball of radius 0.525 res around the image centre in pixel coordinates.  A
// projected vertex further than ~0.01 px from that boundary is decided from its pixel coordinates; the
// thin band around the boundary falls back to the reference's fp32 edge functions, so the decision is
// always the reference's.
template <bool POW2>
__device__ __forceinline__ void project_f(const Camera& cam, float x, float y, float& u0, float& u1) {
    u0 = cam.C * x + cam.S * y;
    u1 = (-cam.S) * x + cam.C * y;
    if (POW2) {
        // res is a power of two: the multiplications by res and by 1/2 are exact, so they commute with the
        // rounding of (-u) * scale and fold into one constant (bit-identical to the chain below)
        u0 = u0 * cam.kscale + cam.half;
        u1 = u1 * cam.kscale + cam.half;
    } else {
        u0 = (-u0) * cam.scale; u1 = (-u1) * cam.scale;     // rendering/base.py:102-115, operation by operation
        u0 = u0 * cam.fmin;     u1 = u1 * cam.fmin;
        u0 = u0 / 2.0f;         u1 = u1 / 2.0f;
        u0 = u0 + cam.half;     u1 = u1 + cam.half;
    }
}

// kind of a candidate after cull + projection + truncation (rendering/cv2.py:52-56)
enum { kCulled = 0, kVerts = 1, kHuge = 2, kShort = 3, kTall = 4, kClipped = 5 };
#ifndef TDS_SHORT_ROWS
#define TDS_SHORT_ROWS 5
#endif
constexpr int kShortRows = TDS_SHORT_ROWS;      // inside triangles spanning at most this many row steps go to the "short" queue

template <bool POW2>
__device__ __forceinline__ int setup_triangle(const Camera& cam, float x0, float y0, float x1, float y1, float x2,
                                              float y2, int own, int xy[6]) {
    const float px0 = x0 + cam.ncx, py0 = y0 + cam.ncy;
    const float px1 = x1 + cam.ncx, py1 = y1 + cam.ncy;
    const float px2 = x2 + cam.ncx, py2 = y2 + cam.ncy;
    float u0, v0, u1, v1, u2, v2;
    project_f<POW2>(cam, px0, py0, u0, v0);
    project_f<POW2>(cam, px1, py1, u1, v1);
    project_f<POW2>(cam, px2, py2, u2, v2);
    const float d0 = fmaxf(fabsf(u0 - cam.half), fabsf(v0 - cam.half));
    const float d1 = fmaxf(fabsf(u1 - cam.half), fabsf(v1 - cam.half));
    const float d2 = fmaxf(fabsf(u2 - cam.half), fabsf(v2 - cam.half));
    if (fminf(fminf(d0, d1), d2) > cam.r_out) return kCulled;       // all vertices clearly outside (NaN: falls through)
    bool c0 = d0 < cam.r_in, c1 = d1 < cam.r_in, c2 = d2 < cam.r_in;
    const bool und0 = !c0 && !(d0 > cam.r_out), und1 = !c1 && !(d1 > cam.r_out), und2 = !c2 && !(d2 > cam.r_out);
    if (und0 | und1 | und2) {       // some vertex is within the band around the quad boundary (or NaN): exact test
        // one rolled loop over the three vertices keeps this rare path small; the edge functions live in smem
        float ex = px0, ey = py0;
#pragma unroll 1
        for (int k = 0; k < 3; k++) {
            const bool r = inside_quad(cam, ex, ey);
            if (k == 0) { if (und0) c0 = r; ex = px1; ey = py1; }
            else if (k == 1) { if (und1) c1 = r; ex = px2; ey = py2; }
            else { if (und2) c2 = r; }
        }
        if (!(c0 | c1 | c2)) return kCulled;
    }
    const int first = c0 ? 0 : (c1 ? 1 : 2);
    if (!((own >> first) & 1)) return kCulled;    // another cell's copy of this face draws it
    xy[0] = __float2int_rz(u0); xy[1] = __float2int_rz(v0);
    xy[2] = __float2int_rz(u1); xy[3] = __float2int_rz(v1);
    xy[4] = __float2int_rz(u2); xy[5] = __float2int_rz(v2);
    // |coordinates| >= 8000 (or NaN): 64-bit rule
    if (!(fmaxf(fmaxf(d0, d1), d2) < 8000.0f - cam.half)) return kHuge;
    // integer bounding box entirely off the image: clipLine rejects all three edges and the fill returns early
    const int res = cam.res;
    const int xmin = min(min(xy[0], xy[2]), xy[4]), xmax = max(max(xy[0], xy[2]), xy[4]);
    const int ymin = min(min(xy[1], xy[3]), xy[5]), ymax = max(max(xy[1], xy[3]), xy[5]);
    if (((xmax | ymax) < 0) | (xmin >= res) | (ymin >= res)) return kCulled;
    // bounding box within 2x2 pixels: the coverage is the set of in-image vertices (tds_raster_tri.h)
    if (((xmax - xmin) | (ymax - ymin)) <= 1) return kVerts;
    const bool inside = ((xmin | ymin) >= 0) & (xmax < res) & (ymax < res);
    return !inside ? kClipped : (ymax - ymin <= kShortRows ? kShort : kTall);
}

// ---- shared memory is addressed through 32-bit shared-window addresses and explicit ld/st/red.shared: with
// generic pointers the compiler re-derives the window base (S2R SR_CgaCtaId, LEA, IMAD ...) at every access site.
__device__ __forceinline__ uint32_t smem_addr(const void* p) {
    // the volatile move makes the address a plain register value: it is computed once instead of being
    // rematerialised from the special registers wherever it is used
    uint32_t a = (uint32_t)__cvta_generic_to_shared(p), r;
    asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(a));
    return r;
}
__device__ __forceinline__ void sred_or(uint32_t a, uint32_t v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t slds(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t slds_const(uint32_t a) {      // tables that never change after the prologue
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void ssts(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint4 slds4(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void ssts4(uint32_t a, uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---- bitplanes: one bit per pixel and draw rank; plane p, word column w, row y at word  p * res * W32 + w * res + y.
// `plane` below is the shared-window BYTE address of a plane.
__device__ __forceinline__ void or_bit(uint32_t plane, int res, int x, int y) {
    sred_or(plane + 4u * (uint32_t)((x >> 5) * res + y), 1u << (x & 31));
}

__device__ __forceinline__ void or_span(uint32_t plane, int res, int y, int lo, int hi) {
    for (int w = lo >> 5; w <= (hi >> 5); w++) {
        const int l = max(lo - 32 * w, 0), h = min(hi - 32 * w, 31);
        sred_or(plane + 4u * (uint32_t)(w * res + y), (0xffffffffu >> (31 - (h - l))) << l);
    }
}

// 64-pixel rows: the two 32-bit halves of a row mask.  Both are OR-ed unconditionally: ptxas turns a predicated
// red.shared into a branch around it (ISETP, BSSY, BRA, BSYNC), which costs more issue slots than the idle OR of a
// zero (the LSU pipe is 14 % busy, the issue slots 77 %).
__device__ __forceinline__ void or_mask64(uint32_t plane, int y, unsigned long long m) {
    const uint32_t addr = plane + 4u * (uint32_t)y;
    sred_or(addr, (uint32_t)m);
    sred_or(addr + 256u, (uint32_t)(m >> 32));
}

// stage 2a: a triangle with all vertices inside the image: one interval and one atomic OR per row and word
template <int RES, bool SMALL>
__device__ __forceinline__ void draw_inside(uint32_t plane, int res, uint32_t rcp_sa, int x0, int y0, int x1, int y1,
                                            int x2, int y2) {
    tds::FastTri t;
    tds::fast_tri_setup<SMALL>(x0, y0, x1, y1, x2, y2, t, [&](int dy) { return slds_const(rcp_sa + 4u * (uint32_t)dy); });
    tds::fast_tri_rows(t, [&](int y, int lo, int hi) {
        if (RES == 64) or_mask64(plane, y, (~0ull >> (63 - (hi - lo))) << lo);
        else or_span(plane, res, y, lo, hi);
    });
}

// stage 2a of the 64x64 kernels: a triangle inside the image as three line walkers (tds_raster_rows.h): one interval and
// one atomic OR per row and word.  Vertices packed as x | y << 8, two per word.
__device__ __forceinline__ uint32_t pack_vertex8(int x, int y) { return (uint32_t)x | ((uint32_t)y << 8); }
__device__ __forceinline__ void draw_lines3_64(uint32_t plane, uint32_t rcp_sa, uint32_t w0, uint32_t w1) {
    tds::Lines3 q;
    tds::lines3_setup((int)(w0 & 0xffu), (int)((w0 >> 8) & 0xffu), (int)((w0 >> 16) & 0xffu), (int)(w0 >> 24), (int)(w1 & 0xffu),
                      (int)((w1 >> 8) & 0xffu), q, [&](int dy) { return slds_const(rcp_sa + 4u * (uint32_t)dy); });
    tds::lines3_rows(q, [&](int yy, int lo, int hi) { or_mask64(plane, yy, (~0ull >> (63 - (hi - lo))) << lo); });
}

// stage 2q: two faces of a strip that form a sliver quad inside the image: the rows of its coverage pattern
// (tds_quad_table.h), shifted to the quad's corner.  w0 = xmin | ymin << 8 | rows << 16 | plane << 24.
__device__ __forceinline__ void draw_quad_pattern64(uint32_t planes_sa, uint32_t plane_bytes, const uint4* __restrict__ table, uint32_t w0,
                                                    uint32_t index) {
    const int xmin = (int)(w0 & 0xffu), ymin = (int)((w0 >> 8) & 0xffu), h = (int)((w0 >> 16) & 0xffu);
    const uint32_t plane = planes_sa + (w0 >> 24) * plane_bytes;
    const uint4* tp = table + (size_t)index * (tds::kQuadRows / 4);
    // rows past the pattern hold zeros: OR-ed into the last image row at most.  The first two groups of four rows (most
    // quads are at most 8 rows tall) are requested together: one L2 latency instead of two.
    uint4 m = __ldg(tp);
    uint4 m_next = __ldg(tp + 1);
#pragma unroll 1
    for (int r = 0; r < h; r += 4) {
        const uint32_t rows[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
        for (int k = 0; k < 4; k++) or_mask64(plane, min(ymin + r + k, 63), (unsigned long long)rows[k] << xmin);
        m = m_next;
        if (r + 8 < h) m_next = __ldg(tp + (r >> 2) + 2);
    }
}

// stage 2b: a triangle that crosses the image border (|coordinates| < 8192), drawn by FOUR lanes (lane & 3 = part): the
// clipped runs of one outline edge each for parts 0..2, the fill set-up by part 3, then a fourth of the clamped fill rows
// each (tds_raster_rows.h: row_tri_part).  Called with the four lanes of a face converged.
template <int RES>
__device__ __forceinline__ void draw_clipped_part(uint32_t plane, int res, uint32_t rcp_sa, int x0, int y0, int x1, int y1,
                                                  int x2, int y2, int part, unsigned lanes) {
    const int first = threadIdx.x & 28;           // the part-0 lane of this face
    tds::row_tri_part(res, res, x0, y0, x1, y1, x2, y2, part, [&](int dy) { return slds_const(rcp_sa + 4u * (uint32_t)dy); },
        [&](int y, int lo, int hi) {
            if (RES == 64) or_mask64(plane, y, (~0ull >> (63 - (hi - lo))) << lo);
            else or_span(plane, res, y, lo, hi);
        },
        [&](int v, int w) { return __shfl_sync(lanes, v, first | w); });
}

// coordinates beyond +-8000 pixels (extreme zoom / giant rectangles): 64-bit rule, pixel by pixel.  Rare.
static __device__ __noinline__ void draw_huge(uint32_t plane, int res, int x0, int y0, int x1, int y1, int x2, int y2) {
    tds::draw_triangle(res, res, x0, y0, x1, y1, x2, y2,
        [&](int x, int y) { or_bit(plane, res, x, y); },
        [&](int y, int xa, int xb) { or_span(plane, res, y, xa, xb); });
}

struct RasterArgs {
    const int32_t* env_map;
    const float* cam_xy;
    const float* cam_sc;
    const uint8_t* present;
    const uint8_t* ws;
    void* out;
    int32_t B, Nc, N, T, present_per_camera, res;
    int32_t LR;                // traffic lights + extra rectangles of an environment (T = 3 N + 2 LR)
    int32_t ncam;
    float scale;
    int32_t* next_cam;         // work counter of the persistent grid (zeroed before the launch)
    const float* cam_tris;     // [B*Nc][Tc][6] world-space triangles of each camera (waypoint discs), or NULL
    const int32_t* cam_cls;    // [B*Nc][Tc] their classes (< 0: skipped)
    int32_t Tc;
    int32_t strip_mode;        // 1: strips take stage 1S, the face segments hold the other faces; 0: the face segments hold all faces
    const uint4* quad_table;   // coverage patterns of sliver quads (tds_quad_table.h), or NULL: pairs of strip faces are drawn one by one
    int32_t out_format;        // TDS_IMAGE_F32 / TDS_IMAGE_U8 / TDS_IMAGE_RANK
    const uint8_t* agent_cls;  // [B*Nc][N] class of each agent's rectangle as this camera sees it (custom colours), or NULL
    int32_t* redo;             // [0] = number of cameras in redo[4..]: LEAN kernels list the cameras they cannot finish
                               // (coordinates beyond +-8000 pixels); a general kernel launched with cam_list = redo
    const int32_t* cam_list;   // NULL: cameras 0..ncam-1; else the general kernel renders cam_list[4 + i], i < cam_list[0]
    // two-pass form of the 64x64 LEAN kernels: the draw pass (PHASE 1) renders cameras [cam_begin, ncam) except the faces
    // that cross the image border, which it lists per camera, and hands the bitplanes over; the finish pass (raster_finish_kernel)
    // draws the listed faces and resolves.  Each pass is a smaller program than the two together: instruction fetch, not
    // instruction count, limits the one-pass kernel (DESIGN.md section 9).  Indexed by camera - cam_begin.
    int32_t cam_begin;
    uint32_t* planes_io;       // [cameras][plane_stride] uint4: the K bitplanes of a camera
    int32_t plane_stride;      // uint4 per camera in planes_io (>= K * res * W32 / 4)
    uint4* clip_list;          // [cameras][kClipCap] faces: x | y << 16 per vertex, plane
    int32_t* clip_count;       // [cameras] listed faces; -1: the camera is on the redo list (the general kernel renders it)
    int32_t clip_cap;          // faces a camera may list before it goes on the redo list (<= kClipCap, the stride of clip_list)
};
constexpr int kClipCap = 192;  // border-crossing faces a camera can list (60 on average at 64x64 / 35 m, 150 at a junction); more: redo

constexpr int kRows = tds::kMaxRasterRows;
constexpr int kQueues = 3;                          // short inside, tall inside, clipped
constexpr int kQueueBytes = (64 + 64 + 40) * 16;    // inside queues: up to 31 left over + 32 new; clipped: 7 + 32
// dynamic primitives in view that a camera can list: 128 for the warp-per-camera kernels (shared memory is what limits
// their occupancy), 512 for the CTA-per-camera kernels of the large tiles (BASELINE config 4: a camera sees 100-200
// of 512 agents; without the list it would walk all 1 536 agent faces)
__host__ __device__ constexpr int cull_cap(int G) { return G == 32 ? 128 : 512; }
constexpr int kSlowCap = 40;                        // strips waiting for their faces to be classified (7 left over + 32 new)
// the warp-per-camera kernels of 64x64 tiles draw every face inside the image as an item of three lines, and pairs of
// strip faces that form a sliver quad as ONE such item (tds_raster_rows.h)
__host__ __device__ constexpr bool raster_quads(int G, int res) { return G == 32 && res == 64; }
// ... whose queue of sliver quads takes up to 31 left over + 64 new (two per strip and thread of stage 1S)
__host__ __device__ constexpr int raster_queue_bytes(int G, int res) { return raster_quads(G, res) ? (64 + 40 + 96) * 16 : kQueueBytes; }

__host__ __device__ constexpr int raster_group_bytes(int res, int n_planes, int G) {
    // planes of the camera | per warp of the group: the three face queues + the queue of strips | tables
    return n_planes * res * ((res + 31) / 32) * 4 + (G / 32) * (raster_queue_bytes(G, res) + kSlowCap * 32) + 16 + cull_cap(G) * 2;
}
// The 64x64 variants (the benchmark configuration) reserve KS = 5 or 7 planes per camera in STATIC shared memory:
// every address is then a compile-time offset and nothing has to be re-derived from the dynamic base.
__host__ __device__ constexpr bool raster_static_smem(int G, int RES, int KS) { return G == 32 && RES == 64 && KS > 0; }

// G = threads cooperating on one camera: 32 (one warp per camera, 4 cameras in flight per CTA, no block barriers)
// for tiles up to 64x64, or the whole CTA for larger tiles.  The warps of a CTA group share the camera's bitplanes
// (atomic ORs) but nothing else: each takes every (G/32)-th batch of 32 candidates and keeps its own three queues,
// so the only block barriers of a camera are after the set-up and before the resolve.
template <int G>
__device__ __forceinline__ void group_sync() {
    if (G == 32) __syncwarp();
    else __syncthreads();
}

// ---- packed fp32 pairs (FADD2 / FMUL2 of sm_100): two IEEE round-to-nearest operations per instruction, bit-identical
// to the scalar ones; the projection of a strip is 18 of them instead of 72 scalar operations.
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// project_f for two vertices at once: X = (xa, xb), Y = (ya, yb) world coordinates -> U, V pixel coordinates
template <bool POW2>
__device__ __forceinline__ void project2(const Camera& cam, uint64_t X, uint64_t Y, uint64_t& U, uint64_t& V) {
    const uint64_t c2 = pk2(cam.C, cam.C), s2 = pk2(cam.S, cam.S), ns2 = pk2(-cam.S, -cam.S);
    const uint64_t px = add2(X, pk2(cam.ncx, cam.ncx)), py = add2(Y, pk2(cam.ncy, cam.ncy));
    U = add2(mul2(c2, px), mul2(s2, py));
    V = add2(mul2(ns2, px), mul2(c2, py));
    const uint64_t h2 = pk2(cam.half, cam.half);
    if (POW2) {
        const uint64_t k2 = pk2(cam.kscale, cam.kscale);
        U = add2(mul2(U, k2), h2);
        V = add2(mul2(V, k2), h2);
    } else {
        // (-u) * scale == u * (-scale) and u / 2 == u * 0.5 exactly; otherwise rendering/base.py:102-115 operation by operation
        const uint64_t m2 = pk2(-cam.scale, -cam.scale), f2 = pk2(cam.fmin, cam.fmin), q2 = pk2(0.5f, 0.5f);
        U = add2(mul2(mul2(mul2(U, m2), f2), q2), h2);
        V = add2(mul2(mul2(mul2(V, m2), f2), q2), h2);
    }
}

// ---- resolve painter's order and expand through the colour LUT: out[cam][ch][x][y].
template <int G, int RES, int NS, bool F32>
__device__ __forceinline__ void resolve_camera(const RasterArgs& a, int camid, int tid, int res, int W32, int K, uint32_t planes_sa,
                                               uint32_t plane_bytes, uint32_t lut_sa) {
    // A thread owns 4 image rows y of one 32-pixel word column: it folds the K planes of those rows into bit
    // slices of the top-most draw rank (registers), then walks the 32 columns: one 128-bit store per channel
    // (float32), one 32-bit store per channel (uint8) or one 32-bit store (draw ranks).
    const int nyq = res >> 2;
    for (int item = tid; item < W32 * nyq; item += G) {
        const int w = item / nyq, yq = item - w * nyq;
        uint32_t sl[NS][4];
#pragma unroll
        for (int s = 0; s < NS; s++)
#pragma unroll
            for (int k = 0; k < 4; k++) sl[s][k] = 0u;
        uint32_t rem[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
#pragma unroll 1
        for (int p = K - 1; p >= 0; p--) {          // last drawn = on top
            const uint4 v = slds4(planes_sa + (uint32_t)p * plane_bytes + 4u * (uint32_t)(w * res + 4 * yq));
            const uint32_t pw[4] = {v.x, v.y, v.z, v.w};
            const int id = p + 1;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t e = pw[k] & rem[k];
                rem[k] &= ~e;
#pragma unroll
                for (int s = 0; s < NS; s++) sl[s][k] |= ((id >> s) & 1) ? e : 0u;
            }
        }
        const int nx = min(32, res - 32 * w);
        const int plane_stride = res * res;
        const int64_t pix = (int64_t)(32 * w) * res + 4 * yq;
        const bool rgb = F32 || a.out_format != TDS_IMAGE_RANK;
        uint8_t* o = reinterpret_cast<uint8_t*>(a.out) + ((int64_t)camid * (rgb ? 3 : 1) * plane_stride + pix) * (F32 ? 4 : 1);
        // draw rank of column x of the thread's row k = bit x of the NS slices.  NS = 3: the slices are interleaved once
        // into nibbles - column 4 j + t of row k is nibble j of nib[t][k] - so a column costs a shift and a mask.
        constexpr int NT = NS == 3 ? 4 : 1;
        uint32_t nib[NT][4];
        if (NS == 3) {
#pragma unroll
            for (int t = 0; t < NT; t++)
#pragma unroll
                for (int k = 0; k < 4; k++)
                    nib[t][k] = ((sl[0][k] >> t) & 0x11111111u) | (((sl[1][k] >> t) & 0x11111111u) << 1) |
                                (((sl[2 % NS][k] >> t) & 0x11111111u) << 2);
        }
        auto rank_of = [&](int x, int t, int k) -> uint32_t {
            if (NS == 3) return (nib[t % NT][k] >> (x - t)) & 7u;          // x - t = 4 j
            uint32_t v = 0u;
#pragma unroll
            for (int q = 0; q < NS; q++) v |= ((sl[q][k] >> x) & 1u) << q;
            return v;
        };
        if (F32) {
#pragma unroll 1
            for (int x0 = 0; x0 < nx; x0 += NT) {
#pragma unroll
                for (int t = 0; t < NT; t++) {
                    const int x = x0 + t;
                    float4 c[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const uint4 q = slds4(lut_sa + 16u * rank_of(x, t, k));
                        c[k] = make_float4(__uint_as_float(q.x), __uint_as_float(q.y), __uint_as_float(q.z), 0.f);
                    }
                    float* of = reinterpret_cast<float*>(o) + (int64_t)x * res;
                    tds::st_cs_f4(reinterpret_cast<float4*>(of), make_float4(c[0].x, c[1].x, c[2].x, c[3].x));
                    tds::st_cs_f4(reinterpret_cast<float4*>(of + plane_stride), make_float4(c[0].y, c[1].y, c[2].y, c[3].y));
                    tds::st_cs_f4(reinterpret_cast<float4*>(of + 2 * plane_stride), make_float4(c[0].z, c[1].z, c[2].z, c[3].z));
                }
            }
        } else {
#pragma unroll 1
            for (int x0 = 0; x0 < nx; x0 += NT) {
#pragma unroll
                for (int t = 0; t < NT; t++) {
                    const int x = x0 + t;
                    uint32_t c[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const uint32_t v = rank_of(x, t, k);
                        c[k] = rgb ? slds(lut_sa + 16u * v + 12u) : v;
                    }
                    // byte b of the four rows -> one word (rows 4 yq .. 4 yq + 3 are consecutive bytes of the output)
                    uint8_t* ob = o + (int64_t)x * res;
                    const uint32_t lo01 = __byte_perm(c[0], c[1], 0x5140), lo23 = __byte_perm(c[2], c[3], 0x5140);   // (r0 r1 g0 g1), (r2 r3 g2 g3)
                    tds::st_cs_u32(reinterpret_cast<uint32_t*>(ob), __byte_perm(lo01, lo23, 0x5410));
                    if (rgb) {
                        const uint32_t hi01 = __byte_perm(c[0], c[1], 0x7362), hi23 = __byte_perm(c[2], c[3], 0x7362);   // (b0 b1 - -), (b2 b3 - -)
                        tds::st_cs_u32(reinterpret_cast<uint32_t*>(ob + plane_stride), __byte_perm(lo01, lo23, 0x7632));
                        tds::st_cs_u32(reinterpret_cast<uint32_t*>(ob + 2 * plane_stride), __byte_perm(hi01, hi23, 0x5410));
                    }
                }
            }
        }
    }
}

#ifndef TDS_RASTER_MINB
#define TDS_RASTER_MINB 7
#endif
#ifndef TDS_FINISH_MINB
#define TDS_FINISH_MINB 8
#endif
#ifndef TDS_RASTER_MINB_BIG
#define TDS_RASTER_MINB_BIG 2
#endif
// NS = bits of the per-pixel draw rank (0 = background): 3 for up to 7 active classes, 5 for up to 31
// KS = planes reserved per camera in static shared memory (64x64 warp-per-camera variants), 0 = dynamic shared memory
// F32: float32 image (else uint8 RGB / draw ranks, a.out_format).  LEAN: the common case only - no
// per-camera triangles, no per-camera agent classes, and cameras that meet coordinates beyond +-8000 pixels are handed
// to the general kernel through a.redo: code that is never executed still costs instruction-cache reach (DESIGN.md section 9)
template <int G, int RES, int NS, bool SMALL, int KS_, bool F32, bool LEAN, int PHASE = 0>
__global__ void __launch_bounds__(G == 32 ? 128 : G, G <= 128 ? TDS_RASTER_MINB : (G == 256 ? 2 * TDS_RASTER_MINB_BIG : TDS_RASTER_MINB_BIG)) raster_kernel(MapSetDev maps, RasterArgs a, PaletteDev pal) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    constexpr int QN = 64;                      // queue capacity per warp and kind
    // SMALL: images up to 128 pixels, slopes through the reciprocal table
    constexpr bool POW2 = RES != 0 && (RES & (RES - 1)) == 0;     // compile-time tile size that is a power of two
    const int res = RES ? RES : a.res;          // RES = 64 is compiled with constant strides
    const int W32 = RES ? RES / 32 : (res + 31) >> 5;
    const int group = G == 32 ? (threadIdx.x >> 5) : 0;
    const int tid = G == 32 ? (threadIdx.x & 31) : threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int K = pal.n_classes;                // planes = draw ranks of the active classes
    // behind a LEAN kernel: the redo list is nearly always empty, and then every CTA leaves before it builds its tables
    if (!LEAN && a.cam_list && a.cam_list[0] == 0) return;

    // CTA-wide tables: colour per draw rank (0 = background), reciprocals of the row runs, class -> plane
    __shared__ float4 s_lut[TDS_MAX_CLASSES + 1];
    constexpr bool STATIC = raster_static_smem(G, RES, KS_);
    constexpr int STATIC_RCP = ((64 + 1) * 4 + 15) & ~15;
    constexpr int STATIC_BYTES = STATIC ? STATIC_RCP + 4 * raster_group_bytes(64, KS_, 32) : 16;
    __shared__ __align__(16) uint8_t smem_static[STATIC_BYTES];
    uint8_t* const smem = STATIC ? smem_static : smem_raw;
    const int KS = STATIC ? KS_ : K;                                         // planes reserved per camera
    uint32_t* s_rcp = reinterpret_cast<uint32_t*>(smem);                     // [res + 1]
    const int rcp_bytes = ((res + 1) * 4 + 15) & ~15;
    for (int i = threadIdx.x; i <= K; i += blockDim.x) {
        const float* c = pal.rgb[i == 0 ? 0 : pal.order[i - 1] + 1];
        // .w = the colour packed as bytes r | g << 8 | b << 16 (uint8 output)
        s_lut[i] = make_float4(c[0], c[1], c[2], __uint_as_float((uint32_t)c[0] | ((uint32_t)c[1] << 8) | ((uint32_t)c[2] << 16)));
    }
    for (int i = threadIdx.x; i <= res; i += blockDim.x) s_rcp[i] = g_rcp.v[i];
    __syncthreads();
    const int plane_tbl = pal.plane_of_class[lane];     // lane c holds the plane of class c (TDS_MAX_CLASSES == 32)

    // per-group shared memory: planes | queues | counters, edge functions, list of dynamic primitives
    const int plane_words = res * W32;
    const int group_bytes = raster_group_bytes(res, KS, G);
    uint8_t* base = smem + rcp_bytes + group * group_bytes;
    const uint32_t planes_sa = smem_addr(base);                            // [KS][W32][res] words
    const uint32_t rcp_sa = planes_sa - (uint32_t)(rcp_bytes + group * group_bytes);
    const uint32_t plane_bytes = 4u * (uint32_t)plane_words;
    constexpr int WARPS = G / 32;
    const uint32_t queues_sa = planes_sa + (uint32_t)KS * plane_bytes;     // [WARPS] x (3 queues of QN x 16 B + the strip queue)
    constexpr bool QUADS = raster_quads(G, RES);
    constexpr int QUEUE_BYTES = raster_queue_bytes(G, RES);
    constexpr int WARP_Q = QUEUE_BYTES + kSlowCap * 32;
    // queue 0: short faces inside the image (QUADS: all of them), queue 1: tall ones (QUADS: sliver quads, 96 entries), queue 2: clipped
    constexpr int Q1 = QUADS ? QN + 40 : QN, Q2 = QUADS ? QN : 2 * QN;
    const uint32_t queue_sa = queues_sa + (G == 32 ? 0u : (uint32_t)(threadIdx.x >> 5) * WARP_Q);   // this warp's
    const uint32_t slow_sa = queue_sa + QUEUE_BYTES;                        // [kSlowCap] x 32 B
    int* s_cnt = reinterpret_cast<int*>(base + KS * plane_words * 4 + WARPS * WARP_Q);   // [3] = next camera (G > 32)
    constexpr int kCullCap = cull_cap(G);
    uint16_t* s_list = reinterpret_cast<uint16_t*>(s_cnt + 4);             // [kCullCap] dynamic primitives in view

    // persistent grid: every group (warp or CTA) pulls the next camera from a global counter, so uneven cameras
    // (a junction full of lane markings next to an empty field) do not leave SMs idle at the end
    while (true) {
        int camid = 0;
        if (G == 32) {
            if (lane == 0) camid = atomicAdd(a.next_cam, 1);
            camid = __shfl_sync(0xffffffffu, camid, 0);
        } else {
            __syncthreads();                        // previous camera completely done (s_cnt is reused below)
            if (tid == 0) s_cnt[3] = atomicAdd(a.next_cam, 1);
            __syncthreads();
            camid = s_cnt[3];
        }
        if (!LEAN && a.cam_list) {
            if (camid >= a.cam_list[0]) break;
            camid = a.cam_list[4 + camid];
        } else {
            if (PHASE == 1) camid += a.cam_begin;
            if (camid >= a.ncam) break;
        }
        // environment of the camera: camid / Nc through the fp32 reciprocal, fixed with the remainder (exact below 2^22
        // environments, which the launcher checks)
        int b = __float2int_rz(__fdividef((float)camid, (float)a.Nc));
        {
            const int r = camid - b * a.Nc;
            b += r < 0 ? -1 : (r >= a.Nc ? 1 : 0);
        }
        const MapDev& map = maps.m[a.env_map ? a.env_map[b] : 0];
        Camera cam;
        const float2 cxy = reinterpret_cast<const float2*>(a.cam_xy)[camid];
        const float2 csc = reinterpret_cast<const float2*>(a.cam_sc)[camid];
        group_sync<G>();                            // previous camera of this group is completely done
        make_camera(cam, cxy.x, cxy.y, csc.x, csc.y, a.scale, res);
        {
#pragma unroll 1
            for (int i = tid; i < K * plane_words / 4; i += G) ssts4(planes_sa + 16u * (uint32_t)i, make_uint4(0u, 0u, 0u, 0u));
            if (G != 32 && tid < 3) s_cnt[tid] = 0;
        }

        // ---- grid cells touched by the bounding box of the view quad: the quad is a square of half-side 1.05 / scale
        // rotated by the camera heading, so its bounding box reaches 1.05 / scale * (|sin| + |cos|) from the camera
        // (+ 1e-4 relative and 10 cm for the rounding of the reference's own corner arithmetic).  With 16 m cells the
        // box touches 3-5 rows and columns; candidates of the few extra corner cells are rejected after ~40
        // instructions, which is cheaper than intersecting the quad with every row - and much less code.  One grid row
        // = one contiguous record range (strips: scell, single faces: rcell), looked up when the walk below reaches it.
        const float margin = 0.10f;
        const float ext = (1.05f / a.scale) * (fabsf(csc.x) + fabsf(csc.y)) * 1.0001f + margin;
        const float xmin = cxy.x - ext, xmax = cxy.x + ext, ymin = cxy.y - ext, ymax = cxy.y + ext;
        int r0 = (int)floorf((ymin - map.ry0) * map.rinv), r1 = (int)floorf((ymax - map.ry0) * map.rinv);
        r0 = max(r0, 0);
        r1 = min(r1, map.rgy - 1);
        const int gc0 = max((int)floorf((xmin - map.rx0) * map.rinv), 0);
        const int gc1 = min((int)floorf((xmax - map.rx0) * map.rinv), map.rgx - 1);
        const int nrows = (xmin <= xmax && gc1 >= gc0) ? min(max(r1 - r0 + 1, 0), kRows) : 0;     // NaN camera: nothing
        group_sync<G>();

        const int T = a.T;
        const float* dtri = reinterpret_cast<const float*>(a.ws + (int64_t)b * ws_env_bytes(T));
        const uint8_t* dcls = reinterpret_cast<const uint8_t*>(dtri + (int64_t)T * 6);
        const uint8_t* pres = a.present ? (a.present_per_camera ? a.present + (int64_t)camid * a.N : a.present + (int64_t)b * a.N)
                                        : nullptr;

        // ---- dynamic primitives in view.  An agent (rectangle + direction triangle, 3 faces) or a traffic light /
        // sign (2 faces) lies within the circle around its rectangle's diagonal (the corners 1 and 3 of its first
        // face); if that circle misses the quad none of its vertices is inside and all its faces are culled, so
        // only the primitives that pass are listed (in any order: the bitplanes do not depend on it).  Absent
        // agents are not listed: they all draw the SAME degenerate face (mesh.py:1083-1089), added once below.
        const int items = a.N + a.LR;
        int n_view = 0;
        bool any_absent = false;
#pragma unroll 1
        for (int i0 = 0; i0 < items; i0 += G) {
            const int i = i0 + tid;
            bool keep = false;
            if (i < items) {
                const bool agent = i < a.N;
                if (agent && pres && !pres[i]) {
                    any_absent = true;
                } else {
                    const float* p = dtri + (int64_t)(agent ? 3 * i : 3 * a.N + 2 * (i - a.N)) * 6;
                    const float mx = 0.5f * (p[2] + p[4]), my = 0.5f * (p[3] + p[5]);
                    const float hx = p[2] - mx, hy = p[3] - my;
                    float u, v;
                    project_f<POW2>(cam, mx + cam.ncx, my + cam.ncy, u, v);
                    const float dd = fmaxf(fabsf(u - cam.half), fabsf(v - cam.half));
                    // |hx| + |hy| >= the radius: a looser circle, no square root
                    keep = !(dd > (cam.r_out + 0.05f) + (fabsf(hx) + fabsf(hy)) * (a.scale * cam.half) * 1.0001f);   // NaN: kept
                }
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            int base = n_view;
            if (G == 32) {
                n_view += __popc(m);
            } else {
                if (lane == 0 && m) base = atomicAdd(&s_cnt[0], __popc(m));
                base = __shfl_sync(0xffffffffu, base, 0);
            }
            const int pos = base + __popc(m & ((1u << lane) - 1u));
            if (keep && pos < kCullCap) s_list[pos] = (uint16_t)i;
        }
        any_absent = __any_sync(0xffffffffu, any_absent);
        if (G != 32) {
            if (any_absent && lane == 0) s_cnt[1] = 1;
            __syncthreads();
            n_view = s_cnt[0];
            any_absent = s_cnt[1] != 0;
        } else {
            __syncwarp();
        }
        // more primitives in view than the list holds (or more than 65535 of them): take them all, in order
        const bool listed = n_view <= kCullCap && items <= 65535;
        const int n_dyn = 3 * (listed ? n_view : items);
        const int dyn_count = n_dyn + (LEAN ? 0 : a.Tc) + (any_absent ? 1 : 0);

        // ---- ONE pass over the candidates.  Segments 0 .. nrows-1 = the strip records of the touched grid rows,
        // nrows .. 2 nrows - 1 = their single-face records, segment 2 nrows = the dynamic primitives of the
        // environment.  Stage 1 plots what is just vertices and queues the other faces by kind; whenever a warp has
        // queued 32 faces of a kind, stage 2 turns them into row intervals, one face per thread, so stage 2 always
        // runs with full warps.  Strips that need more than their vertices wait in a queue of their own until 8 of
        // them make a full warp of faces (4 lanes per strip).  The last iterations (seg > 2 nrows) only drain the queues.
        const int seg_dyn = 2 * nrows;
        const int strip_rows = nrows;                  // segments below this one take stage 1S (empty without strip mode)
        bool redo = false;                             // LEAN: something this kernel leaves to the general one
        int seg = -1, j0 = 0, seg_start = 0, seg_count = 0;
        int nq0 = 0, nq1 = 0, nq2 = 0;                 // fill levels of this warp's queues (uniform over the warp)
        int nslow = 0;                                 // strips whose faces are still to be classified
        while (true) {
            if (nslow < 8) {
                while (j0 >= seg_count && seg <= seg_dyn) {
                    seg++;
                    j0 = 0;
                    if (seg < seg_dyn) {
                        // without strip mode the strip segments are empty and the face segments hold EVERY face
                        const bool strips = seg < nrows;
                        const int32_t* cell = (strips ? map.scell : (a.strip_mode ? map.rcell : map.rcell_all)) +
                                              (r0 + (strips ? seg : seg - nrows)) * map.rgx;
                        seg_start = __ldg(cell + gc0);
                        seg_count = (strips && !a.strip_mode) ? 0 : __ldg(cell + gc1 + 1) - seg_start;
                    } else {
                        seg_start = 0;
                        seg_count = seg == seg_dyn ? dyn_count : 0;
                    }
                }
            }
            // kind and truncated vertices of the face this lane hands to the queues in this iteration (if any)
            int kind = kCulled, plane = -1;
            int xy[6];
            if (nslow >= 8 || (nslow > 0 && seg >= strip_rows)) {
                // ================= faces of queued strips: 4 lanes per strip, face f = vertices f, f+1, f+2
                const int take = min(nslow, 8);
                const int s = lane >> 2, f = lane & 3;
                const bool act = s < take;
                const uint32_t ea = slow_sa + 32u * (uint32_t)(nslow - take + (act ? s : 0));
                const uint32_t w0 = slds(ea + 4u * f), w1 = slds(ea + 4u * f + 4u), w2 = slds(ea + 4u * f + 8u), m = slds(ea + 24u);
                nslow -= take;
                xy[0] = (int16_t)(w0 & 0xffff); xy[1] = (int32_t)w0 >> 16;
                xy[2] = (int16_t)(w1 & 0xffff); xy[3] = (int32_t)w1 >> 16;
                xy[4] = (int16_t)(w2 & 0xffff); xy[5] = (int32_t)w2 >> 16;
                plane = (int)((m >> 8) & 0xffu);
                const int fxmin = min(min(xy[0], xy[2]), xy[4]), fxmax = max(max(xy[0], xy[2]), xy[4]);
                const int fymin = min(min(xy[1], xy[3]), xy[5]), fymax = max(max(xy[1], xy[3]), xy[5]);
                const bool off = ((fxmax | fymax) < 0) | (fxmin >= res) | (fymin >= res);
                const bool tiny = ((fxmax - fxmin) | (fymax - fymin)) <= 1;      // its vertices: plotted by stage 1S
                const bool inside = ((fxmin | fymin) >= 0) & (fxmax < res) & (fymax < res);
                // some vertex inside the view quad, and not already drawn as half of a sliver quad (stage 1S)
                const bool kept = ((m >> f) & 7u) != 0u && !((m >> (16 + f)) & 1u);
                kind = (!act | off | tiny | !kept) ? kCulled : (!inside ? kClipped : (fymax - fymin <= kShortRows ? kShort : kTall));
            } else if (seg <= seg_dyn) {
                // uniform control flow: every lane fetches a valid record (the last one of the segment past its end)
                const int j = j0 + tid;
                const bool warp_has_work = j0 + (tid & ~31) < seg_count;
                j0 += G;
                if (G != 32 && !warp_has_work) continue;      // this warp's slice of the batch is past the segment's end
                const bool valid = j < seg_count;
                const int jj = valid ? j : seg_count - 1;
                if (seg < strip_rows) {
                    // ================= stage 1S: one strip (6 vertices, faces (k, k+1, k+2), k = 0..3) per thread
                    const int idx = seg_start + jj;
                    const float4* sp = map.srec + (int64_t)(idx >> 5) * 96 + (idx & 31);
                    const float4 va = __ldg(sp), vb = __ldg(sp + 32), vc = __ldg(sp + 64);
                    const uint32_t meta = __ldg(map.smeta + idx);
                    // a copy binned outside the cell of vertex 0 is redundant when that cell is scanned as well
                    const int pc = (int)((meta >> 6) & 8191u), pr = (int)(meta >> 19);
                    const bool dup = (meta & 32u) && pc >= gc0 && pc <= gc1 && pr >= r0 && pr < r0 + nrows;
                    int spl = __shfl_sync(0xffffffffu, plane_tbl, (int)(meta & 31u));
                    spl = (valid && !dup) ? spl : -1;
                    float u[6], v[6];
                    {
                        uint64_t U, V;
                        project2<POW2>(cam, pk2(va.x, va.y), pk2(va.z, va.w), U, V);
                        upk2(U, u[0], u[1]); upk2(V, v[0], v[1]);
                        project2<POW2>(cam, pk2(vb.x, vb.y), pk2(vb.z, vb.w), U, V);
                        upk2(U, u[2], u[3]); upk2(V, v[2], v[3]);
                        project2<POW2>(cam, pk2(vc.x, vc.y), pk2(vc.z, vc.w), U, V);
                        upk2(U, u[4], u[5]); upk2(V, v[4], v[5]);
                    }
                    // inside / outside the 1.05x quad per vertex (bit k of cb), undecided ones in ub (see setup_triangle)
                    int xi[6], yi[6];
                    uint32_t cb = 0u, ub = 0u;
                    float dmax = 0.0f;              // NaN vertices: undecided (ub), truncated to 0, not "huge"
#pragma unroll
                    for (int k = 0; k < 6; k++) {
                        const float d = fmaxf(fabsf(u[k] - cam.half), fabsf(v[k] - cam.half));
                        const bool in = d < cam.r_in;
                        cb |= in ? 1u << k : 0u;
                        ub |= (!in && !(d > cam.r_out)) ? 1u << k : 0u;
                        dmax = fmaxf(dmax, d);
                        xi[k] = __float2int_rz(u[k]);
                        yi[k] = __float2int_rz(v[k]);
                    }
                    const uint32_t pl = planes_sa + (uint32_t)max(spl, 0) * plane_bytes;
                    // every vertex inside the image is a pixel of each kept face it belongs to (the outline of a face
                    // contains its end points), and such a face IS kept: the image lies inside the view quad with a
                    // margin of more than one pixel (strip_mode).  A vertex outside the image ORs a zero into
                    // pixel (0, 0): no branch around the reduction.  (The kernels with sliver quads plot further down,
                    // and only the strips that need it.)
                    if (!QUADS) {
#pragma unroll
                        for (int k = 0; k < 6; k++) {
                            const bool in = spl >= 0 && (POW2 ? (unsigned)(xi[k] | yi[k]) < (unsigned)res
                                                              : ((unsigned)xi[k] < (unsigned)res && (unsigned)yi[k] < (unsigned)res));
                            const int x = in ? xi[k] : 0, y = in ? yi[k] : 0;
                            sred_or(pl + 4u * (uint32_t)((x >> 5) * res + y), in ? 1u << (x & 31) : 0u);
                        }
                    }
                    const int sxmin = min(min(min(xi[0], xi[1]), min(xi[2], xi[3])), min(xi[4], xi[5]));
                    const int sxmax = max(max(max(xi[0], xi[1]), max(xi[2], xi[3])), max(xi[4], xi[5]));
                    const int symin = min(min(min(yi[0], yi[1]), min(yi[2], yi[3])), min(yi[4], yi[5]));
                    const int symax = max(max(max(yi[0], yi[1]), max(yi[2], yi[3])), max(yi[4], yi[5]));
                    // nothing left to draw: all six vertices within 2x2 pixels (every face is its vertices), or the
                    // strip's bounding box off the image, or no vertex inside the quad
                    bool slow = spl >= 0 && (((sxmax - sxmin) | (symax - symin)) > 1) &&
                                !(((sxmax | symax) < 0) | (sxmin >= res) | (symin >= res)) && ((cb | ub) != 0u);
                    if (slow && ub) {
                        // vertices in the thin band around the quad's boundary: the reference's fp32 edge functions
#pragma unroll 1
                        for (int k = 0; k < 6; k++) {
                            if ((ub >> k) & 1u) {
                                const float* fp = reinterpret_cast<const float*>(sp + (k >> 1) * 32);
                                if (inside_quad(cam, fp[k & 1] + cam.ncx, fp[2 + (k & 1)] + cam.ncy)) cb |= 1u << k;
                            }
                        }
                    }
                    if (slow && !(dmax < 8000.0f - cam.half)) {
                        // |coordinates| >= 8000: 64-bit rule, face by face (LEAN: the general kernel redoes the camera)
                        if (LEAN) {
                            redo = true;
                        } else {
                            if (cb & 7u) draw_huge(pl, res, xi[0], yi[0], xi[1], yi[1], xi[2], yi[2]);
                            if (cb & 14u) draw_huge(pl, res, xi[1], yi[1], xi[2], yi[2], xi[3], yi[3]);
                            if (cb & 28u) draw_huge(pl, res, xi[2], yi[2], xi[3], yi[3], xi[4], yi[4]);
                            if (cb & 56u) draw_huge(pl, res, xi[3], yi[3], xi[4], yi[4], xi[5], yi[5]);
                        }
                        slow = false;
                    }
                    uint32_t done = 0u;              // faces that need nothing more: half of a sliver quad (queued, or just its vertices)
                    uint32_t queued = 0u;            // faces of the quads that were queued
                    if (QUADS && a.quad_table) {
                        // The strip is two quads: faces (0, 1) over vertices 0..3 and faces (2, 3) over vertices 2..5.  A quad
                        // whose faces are both kept, with its four vertices inside the image and a shape of the pattern
                        // table, is queued as ONE item right here (tds_quad_table.h: the union of the two triangles by the
                        // reference's rule, so it does not matter that one of them may be tiny); within 2x2 pixels it is just
                        // its vertices, which are plotted already.
#pragma unroll
                        for (int qd = 0; qd < 2; qd++) {
                            const int k = 2 * qd;
                            const bool both = ((cb >> k) & 7u) != 0u && ((cb >> (k + 1)) & 7u) != 0u;
                            const int qxmin = min(min(xi[k], xi[k + 1]), min(xi[k + 2], xi[k + 3])), qxmax = max(max(xi[k], xi[k + 1]), max(xi[k + 2], xi[k + 3]));
                            const int qymin = min(min(yi[k], yi[k + 1]), min(yi[k + 2], yi[k + 3])), qymax = max(max(yi[k], yi[k + 1]), max(yi[k + 2], yi[k + 3]));
                            const bool allin = (unsigned)(qxmin | qymin) < 64u && (unsigned)(qxmax | qymax) < 64u;
                            // rungs (v0, v1), (v2, v3) with rails (v0, v2), (v1, v3) - or the other way round
                            int gx = xi[k + 1] - xi[k], gy = yi[k + 1] - yi[k], r1x = xi[k + 2] - xi[k], r1y = yi[k + 2] - yi[k];
                            int r2x = xi[k + 3] - xi[k + 1], r2y = yi[k + 3] - yi[k + 1];
                            const bool cand = slow && both && allin;
                            bool tab = tds::quad_in_table(gx, gy, r1x, r1y, r2x, r2y);
                            if (__any_sync(0xffffffffu, cand && !tab)) {        // rare: the first naming fits almost every quad
                                if (!tab) {
                                    int t = gx; gx = r1x; r1x = t; t = gy; gy = r1y; r1y = t;
                                    r2x = xi[k + 3] - xi[k + 2]; r2y = yi[k + 3] - yi[k + 2];
                                    tab = tds::quad_in_table(gx, gy, r1x, r1y, r2x, r2y);
                                }
                            }
                            const bool covered = cand && tab;
                            const bool quad = covered && (((qxmax - qxmin) | (qymax - qymin)) > 1);
                            done |= covered ? 3u << k : 0u;
                            queued |= quad ? 3u << k : 0u;
                            const unsigned mq = __ballot_sync(0xffffffffu, quad);
                            if (quad) {
                                const int pos = Q1 + nq1 + __popc(mq & ((1u << lane) - 1));
                                ssts4(queue_sa + 16u * (uint32_t)pos,
                                      make_uint4((uint32_t)qxmin | ((uint32_t)qymin << 8) | ((uint32_t)(qymax - qymin + 1) << 16) | ((uint32_t)spl << 24),
                                                 (uint32_t)tds::quad_pattern_index(gx, gy, r1x, r1y, r2x, r2y), 0u, 0u));
                            }
                            nq1 += __popc(mq);
                        }
                        // faces that are kept and not covered by a quad still go through the strip queue
                        uint32_t left = 0u;
#pragma unroll
                        for (int f = 0; f < 4; f++) left |= (((cb >> f) & 7u) != 0u && !((done >> f) & 1u)) ? 1u << f : 0u;
                        slow = slow && left != 0u;
                    }
                    // QUADS: the vertices are plotted here, unless the strip's four faces went on as quads (road surfaces,
                    // batch after batch: the records of a cell are sorted by class)
                    if (QUADS && __any_sync(0xffffffffu, spl >= 0 && queued != 15u)) {
#pragma unroll
                        for (int k = 0; k < 6; k++) {
                            // 64x64: the address is formed from the low six bits (always inside the plane), the bit is
                            // zero for a vertex outside the image
                            const bool in = spl >= 0 && (unsigned)(xi[k] | yi[k]) < 64u;
                            sred_or(pl + (((uint32_t)xi[k] & 32u) << 3) + (((uint32_t)yi[k] & 63u) << 2), in ? 1u << (xi[k] & 31) : 0u);
                        }
                    }
                    // the others wait in the strip queue until 8 of them make a full warp of faces
                    const unsigned ms = __ballot_sync(0xffffffffu, slow);
                    if (slow) {
                        const uint32_t ea = slow_sa + 32u * (uint32_t)(nslow + __popc(ms & ((1u << lane) - 1)));
                        ssts4(ea, make_uint4((uint32_t)(xi[0] & 0xffff) | ((uint32_t)yi[0] << 16), (uint32_t)(xi[1] & 0xffff) | ((uint32_t)yi[1] << 16),
                                             (uint32_t)(xi[2] & 0xffff) | ((uint32_t)yi[2] << 16), (uint32_t)(xi[3] & 0xffff) | ((uint32_t)yi[3] << 16)));
                        ssts4(ea + 16u, make_uint4((uint32_t)(xi[4] & 0xffff) | ((uint32_t)yi[4] << 16), (uint32_t)(xi[5] & 0xffff) | ((uint32_t)yi[5] << 16),
                                                   cb | ((uint32_t)spl << 8) | (done << 16), 0u));
                    }
                    nslow += __popc(ms);
                } else {
                    // ================= stage 1F: one face per thread
                    float x0, y0, x1, y1, x2, y2;
                    int own = 7, cls;
                    if (seg < seg_dyn) {
                        const float4* rp = (a.strip_mode ? map.rec : map.rec_all) + 2 * (int64_t)(seg_start + jj);
                        const float4 v01 = __ldg(rp);
                        const float4 v2o = __ldg(rp + 1);
                        x0 = v01.x; y0 = v01.y; x1 = v01.z; y1 = v01.w; x2 = v2o.x; y2 = v2o.y;
                        const int meta = __float_as_int(v2o.z);
                        own = meta & 7;
                        cls = meta >> 8;
                    } else if (!LEAN && jj >= n_dyn && jj < n_dyn + a.Tc) {
                        // triangles of this camera only (goal-waypoint discs, mesh.py:1120-1145)
                        const int64_t ct = (int64_t)camid * a.Tc + (jj - n_dyn);
                        const int c = a.cam_cls[ct];
                        cls = c < 0 ? 255 : c;
                        const float* p = a.cam_tris + ct * 6;
                        x0 = p[0]; y0 = p[1]; x1 = p[2]; y1 = p[3]; x2 = p[4]; y2 = p[5];
                    } else {
                        // dynamic primitives in view: slot 3 k + f = face f of the k-th listed agent / light / sign; the
                        // last slot is the degenerate face of the absent agents: actor vertex 0 with agent 0's class
                        const bool degenerate = jj >= n_dyn;
                        const int k = jj / 3, f = jj - 3 * k;
                        const int item = degenerate ? 0 : (listed ? (int)s_list[k] : k);
                        const bool agent = item < a.N;
                        const int t = degenerate ? 0 : (agent ? 3 * item + f : 3 * a.N + 2 * (item - a.N) + f);
                        // a sign has two faces; without the list an absent agent shows up here as well
                        const bool skip = !degenerate && ((!agent && f == 2) || (!listed && agent && pres && !pres[item]));
                        const int ts = skip ? 0 : t;
                        cls = skip ? 255 : dcls[ts];
                        // generate(custom_agent_colors=...), mesh.py:1092-1099: the four rectangle vertices of an agent
                        // take the colour this camera was given for it (the direction triangle keeps its own)
                        if (!LEAN && a.agent_cls && !skip && agent && (degenerate || f < 2)) cls = a.agent_cls[(int64_t)camid * a.N + item];
                        const float* p = dtri + (int64_t)ts * 6;
                        x0 = p[0]; y0 = p[1];
                        x1 = degenerate ? x0 : p[2]; y1 = degenerate ? y0 : p[3];
                        x2 = degenerate ? x0 : p[4]; y2 = degenerate ? y0 : p[5];
                    }
                    // class -> plane through the lane-resident table (lane c holds the plane of class c)
                    plane = __shfl_sync(0xffffffffu, plane_tbl, cls & 31);
                    plane = (valid && (unsigned)cls < (unsigned)TDS_MAX_CLASSES) ? plane : -1;
                    if (plane >= 0) kind = setup_triangle<POW2>(cam, x0, y0, x1, y1, x2, y2, own, xy);
                    if (kind == kVerts) {
                        // a vertex outside the image ORs a zero into pixel (0, 0): no branch around the reduction
                        const uint32_t pl = planes_sa + (uint32_t)plane * plane_bytes;
#pragma unroll
                        for (int k = 0; k < 3; k++) {
                            const bool in = (unsigned)xy[2 * k] < (unsigned)res && (unsigned)xy[2 * k + 1] < (unsigned)res;
                            const int x = in ? xy[2 * k] : 0, y = in ? xy[2 * k + 1] : 0;
                            sred_or(pl + 4u * (uint32_t)((x >> 5) * res + y), in ? 1u << (x & 31) : 0u);
                        }
                    } else if (kind == kHuge) {
                        if (LEAN) redo = true;
                        else draw_huge(planes_sa + (uint32_t)plane * plane_bytes, res, xy[0], xy[1], xy[2], xy[3], xy[4], xy[5]);
                    }
                }
            }
            const bool drain = seg > seg_dyn && nslow == 0;
            // queue the faces by kind (warp-aggregated append)
            if (__any_sync(0xffffffffu, kind >= kShort)) {
                if (QUADS) {
                    // queue 0: triangles inside the image (three line walkers), queue 2: faces that cross the border
                    // (queue 1, the sliver quads, is filled by stage 1S)
                    const bool ins = kind == kShort || kind == kTall;
                    const unsigned m0 = __ballot_sync(0xffffffffu, ins), m2 = __ballot_sync(0xffffffffu, kind == kClipped);
                    const int b0 = nq0, b2 = nq2;
                    nq0 += __popc(m0); nq2 += __popc(m2);
                    if (kind >= kShort) {
                        const int pos = (ins ? b0 : (PHASE == 1 ? b2 : Q2 + b2)) + __popc((ins ? m0 : m2) & ((1u << lane) - 1));
                        const uint4 item = ins ? make_uint4(pack_vertex8(xy[0], xy[1]) | (pack_vertex8(xy[2], xy[3]) << 16), pack_vertex8(xy[4], xy[5]),
                                                            (uint32_t)plane, 0u)
                                               : make_uint4((uint32_t)(xy[0] & 0xffff) | ((uint32_t)xy[1] << 16),
                                                            (uint32_t)(xy[2] & 0xffff) | ((uint32_t)xy[3] << 16),
                                                            (uint32_t)(xy[4] & 0xffff) | ((uint32_t)xy[5] << 16), (uint32_t)plane);
                        if (PHASE == 1 && !ins) {
                            // the finish pass draws the faces that cross the border (nq2 counts them over the whole camera)
                            if (pos < a.clip_cap) a.clip_list[(int64_t)(camid - a.cam_begin) * kClipCap + pos] = item;
                        } else {
                            ssts4(queue_sa + 16u * (uint32_t)pos, item);
                        }
                    }
                    if (PHASE == 1 && nq2 > a.clip_cap) redo = true;
                } else {
                    const unsigned m0 = __ballot_sync(0xffffffffu, kind == kShort), m1 = __ballot_sync(0xffffffffu, kind == kTall),
                                   m2 = __ballot_sync(0xffffffffu, kind == kClipped);
                    const int b0 = nq0, b1 = nq1, b2 = nq2;
                    nq0 += __popc(m0); nq1 += __popc(m1); nq2 += __popc(m2);
                    if (kind >= kShort) {
                        const unsigned mine = kind == kShort ? m0 : (kind == kTall ? m1 : m2);
                        const int qb = kind == kShort ? b0 : (kind == kTall ? Q1 + b1 : Q2 + b2);
                        const int pos = qb + __popc(mine & ((1u << lane) - 1));
                        ssts4(queue_sa + 16u * (uint32_t)pos,
                              make_uint4((uint32_t)(xy[0] & 0xffff) | ((uint32_t)xy[1] << 16),
                                         (uint32_t)(xy[2] & 0xffff) | ((uint32_t)xy[3] << 16),
                                         (uint32_t)(xy[4] & 0xffff) | ((uint32_t)xy[5] << 16), (uint32_t)plane));
                    }
                }
            }
            __syncwarp();
            if (!(drain | (nq0 >= 32) | (nq1 >= 32) | (PHASE != 1 && nq2 >= 8))) continue;
            // stage 2: a queue is drawn when it holds a full group (or, at the end, whatever is left)
            if (QUADS) {
                while (nq1 >= 32 || (drain && nq1 > 0)) {
                    const int take = min(nq1, 32);
                    if (lane < take) {
                        const uint4 q = slds4(queue_sa + 16u * (uint32_t)(Q1 + nq1 - take + lane));
                        draw_quad_pattern64(planes_sa, plane_bytes, a.quad_table, q.x, q.y);
                    }
                    nq1 -= take;
                    __syncwarp();
                }
                if (nq0 >= 32 || (drain && nq0 > 0)) {
                    const int take = min(nq0, 32);
                    if (lane < take) {
                        const uint4 q = slds4(queue_sa + 16u * (uint32_t)(nq0 - take + lane));
                        draw_lines3_64(planes_sa + q.z * plane_bytes, rcp_sa, q.x, q.y);
                    }
                    nq0 -= take;
                    __syncwarp();
                }
            } else {
#pragma unroll 1
                for (int which = 0; which < 2; which++) {
                    const int nq = which ? nq1 : nq0;
                    if (nq >= 32 || (drain && nq > 0)) {
                        const int take = min(nq, 32);
                        if (lane < take) {
                            const uint4 q = slds4(queue_sa + 16u * (uint32_t)(which * Q1 + nq - take + lane));
                            draw_inside<RES, SMALL>(planes_sa + q.w * plane_bytes, res, rcp_sa,
                                                    (int16_t)(q.x & 0xffff), (int32_t)q.x >> 16, (int16_t)(q.y & 0xffff),
                                                    (int32_t)q.y >> 16, (int16_t)(q.z & 0xffff), (int32_t)q.z >> 16);
                        }
                        if (which) nq1 -= take; else nq0 -= take;
                        __syncwarp();
                    }
                }
            }
            // faces that cross the border: 4 lanes per face (its three outline edges and its fill), 8 faces per round
#ifdef TDS_EXP_NOCLIP
            if (PHASE != 1) nq2 = 0;                   // experiment: border-crossing faces are not drawn (wrong images)
#endif
            while (PHASE != 1 && (nq2 >= 8 || (drain && nq2 > 0))) {
                const int take = min(nq2, 8);
                const unsigned lanes = take >= 8 ? 0xffffffffu : (1u << (4 * take)) - 1u;
                if ((lane >> 2) < take) {
                    const uint4 q = slds4(queue_sa + 16u * (uint32_t)(Q2 + nq2 - take + (lane >> 2)));
                    draw_clipped_part<RES>(planes_sa + q.w * plane_bytes, res, rcp_sa,
                                           (int16_t)(q.x & 0xffff), (int32_t)q.x >> 16, (int16_t)(q.y & 0xffff),
                                           (int32_t)q.y >> 16, (int16_t)(q.z & 0xffff), (int32_t)q.z >> 16, lane & 3, lanes);
                }
                nq2 -= take;
                __syncwarp();
            }
            if (drain) {
                if ((nq0 | nq1 | (PHASE == 1 ? 0 : nq2)) == 0) break;     // a queue held more than one group: drain again
            }
        }
        group_sync<G>();
        bool any_redo = false;
        if (LEAN || PHASE == 1) {
            // a camera this kernel could not finish exactly goes on the list of the general kernel (which overwrites its image)
            any_redo = G == 32 ? __any_sync(0xffffffffu, redo) : (__syncthreads_or(redo) != 0);
            if (any_redo && tid == 0) a.redo[4 + atomicAdd(a.redo, 1)] = camid;
        }
        group_sync<G>();

        // ---- resolve painter's order and expand through the colour LUT (or hand the bitplanes to the finish kernel)
        if (PHASE == 1) {
            const int li = camid - a.cam_begin;
            uint4* po = reinterpret_cast<uint4*>(a.planes_io) + (int64_t)li * a.plane_stride;
#pragma unroll 1
            for (int i = tid; i < K * plane_words / 4; i += G) po[i] = slds4(planes_sa + 16u * (uint32_t)i);
            if (tid == 0) a.clip_count[li] = any_redo ? -1 : nq2;   // -1: the general kernel renders this camera
        } else {
#ifdef TDS_EXP_NORESOLVE
            if (a.ncam < 0)                            // experiment: the resolve is compiled in but never executed (no images)
#endif
            resolve_camera<G, RES, NS, F32>(a, camid, tid, res, W32, K, planes_sa, plane_bytes, smem_addr(s_lut));
        }
    }
}


// ---- finish pass of the two-pass 64x64 form: bitplanes of the draw pass + its list of border-crossing faces -> image.
// A warp per camera, 4 cameras in flight per CTA; the program is the clipped-face path and the resolve, nothing else.
// The hand-over data of the NEXT camera (bitplanes by cp.async into the other half of a double buffer, face count and
// the first eight faces into registers) is requested before the current camera is drawn: the pass is bound by the
// latency of these loads and by the 3.2 GB of image it writes, not by instructions.
__device__ __forceinline__ void cp_async16(uint32_t dst_sa, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_sa), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int NS, int KS, bool F32>
__global__ void __launch_bounds__(128, TDS_FINISH_MINB) raster_finish_kernel(RasterArgs a, PaletteDev pal) {
    constexpr int RES = 64, W32 = 2, PLANE_WORDS = RES * W32;
    __shared__ float4 s_lut[TDS_MAX_CLASSES + 1];
    __shared__ __align__(16) uint32_t s_rcp[RES + 4];
    constexpr int NB = KS <= 7 ? 2 : 1;          // double buffer while it fits the 48 KB of static shared memory
    __shared__ __align__(16) uint32_t s_planes[4][NB][KS * PLANE_WORDS];
    const int K = pal.n_classes;
    for (int i = threadIdx.x; i <= K; i += blockDim.x) {
        const float* c = pal.rgb[i == 0 ? 0 : pal.order[i - 1] + 1];
        s_lut[i] = make_float4(c[0], c[1], c[2], __uint_as_float((uint32_t)c[0] | ((uint32_t)c[1] << 8) | ((uint32_t)c[2] << 16)));
    }
    for (int i = threadIdx.x; i <= RES; i += blockDim.x) s_rcp[i] = g_rcp.v[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t buf_sa[2] = {smem_addr(s_planes[threadIdx.x >> 5][0]), smem_addr(s_planes[threadIdx.x >> 5][NB - 1])};
    const uint32_t rcp_sa = smem_addr(s_rcp), lut_sa = smem_addr(s_lut);
    constexpr uint32_t plane_bytes = 4u * PLANE_WORDS;
    const int n_local = a.ncam - a.cam_begin;

    // planes of camera li -> buffer b (one commit group)
    auto request_planes = [&](int li, int b) {
        if (li < n_local) {
            const uint4* pi = reinterpret_cast<const uint4*>(a.planes_io) + (int64_t)li * a.plane_stride;
#pragma unroll 1
            for (int i = lane; i < K * PLANE_WORDS / 4; i += 32) cp_async16(buf_sa[b] + 16u * (uint32_t)i, pi + i);
        }
        cp_async_commit();
    };
    // next camera of this warp: its face count and first faces -> registers (and, with two buffers, its planes -> buffer b)
    auto fetch = [&](int& li, int& count, uint4& q0, int b) {
        li = 0;
        if (lane == 0) li = atomicAdd(a.next_cam, 1);
        li = __shfl_sync(0xffffffffu, li, 0);
        count = -1;
        q0 = make_uint4(0u, 0u, 0u, 0u);
        if (li < n_local) {
            count = a.clip_count[li];
            q0 = a.clip_list[(int64_t)li * kClipCap + (lane >> 2)];     // slots past the count hold stale data: not used
        }
        if (NB == 2) request_planes(li, b);
    };

    int li, count, b = 0;
    uint4 q0;
    fetch(li, count, q0, 0);
    while (li < n_local) {
        int li_next, count_next;
        uint4 q0_next;
        __syncwarp();                               // the resolve of the camera before (last) has read the buffer that is filled next
        fetch(li_next, count_next, q0_next, b ^ 1);
        if (NB == 2) {
            cp_async_wait<1>();                     // this camera's planes have landed (the next one's may be in flight)
        } else {
            request_planes(li, 0);
            cp_async_wait<0>();
        }
        __syncwarp();
        if (count >= 0) {                           // -1: on the redo list, the general kernel renders this camera
            const int camid = li + a.cam_begin;
            const uint32_t planes_sa = buf_sa[NB == 2 ? b : 0];
            const uint4* faces = a.clip_list + (int64_t)li * kClipCap;
#pragma unroll 1
            for (int i0 = 0; i0 < count; i0 += 8) {
                const int take = min(count - i0, 8);
                uint4 q_after = q0;
                if (i0 + 8 < count) q_after = faces[i0 + 8 + (lane >> 2)];          // the next round's faces, ahead of the draw
                // every lane takes part (full-mask shuffles: one instruction each); the lanes past the last face draw a face that
                // lies off the image - all its edges are rejected by clipLine, its bounding box misses the image
                if ((lane >> 2) >= take) q0 = make_uint4(0xff9cff9cu, 0xff9cff9cu, 0xff9cff9cu, 0u);          // (-100, -100) x 3
                draw_clipped_part<RES>(planes_sa + q0.w * plane_bytes, RES, rcp_sa, (int16_t)(q0.x & 0xffff), (int32_t)q0.x >> 16,
                                       (int16_t)(q0.y & 0xffff), (int32_t)q0.y >> 16, (int16_t)(q0.z & 0xffff), (int32_t)q0.z >> 16, lane & 3,
                                       0xffffffffu);
                q0 = q_after;
                __syncwarp();
            }
            resolve_camera<32, RES, NS, F32>(a, camid, lane, RES, W32, K, planes_sa, plane_bytes, lut_sa);
        }
        li = li_next; count = count_next; q0 = q0_next; b ^= 1;
    }
    cp_async_wait<0>();
}

// ---- launch of one kernel variant (shared by the translation units that instantiate the variants)
struct LaunchCfg {
    MapSetDev set;
    RasterArgs a;
    PaletteDev pal;
    int K, res, sms;
    int64_t ncam;
    cudaStream_t st;
    cudaEvent_t ev_start, ev_stop;      // recorded around the launch when both are set
};

template <class Kernel>
int launch_variant(Kernel kernel, const LaunchCfg& c, int groups, int threads, bool static_smem) {
    const size_t rcp_bytes = (((size_t)c.res + 1) * 4 + 15) & ~(size_t)15;
    size_t smem = static_smem ? 0 : rcp_bytes + (size_t)raster_group_bytes(c.res, c.K, threads / groups) * groups;
    if (const char* e = getenv("TDS_RASTER_PAD_SMEM")) smem += (size_t)atoi(e);      // profiling aid: fewer resident CTAs
    TDS_REQUIRE(smem <= 227 * 1024, "raster: res=%d with %d active classes needs %zu bytes of shared memory", c.res, c.K, smem);
    if (smem > 40 * 1024) TDS_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    TDS_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    TDS_REQUIRE(per_sm >= 1, "raster: kernel does not fit an SM (res=%d, %d classes)", c.res, c.K);
    // persistent grid: every resident CTA slot of the GPU, cameras pulled from a global counter
    const int64_t want = (c.ncam - c.a.cam_begin + groups - 1) / groups;
    const unsigned grid = (unsigned)std::min<int64_t>(want, (int64_t)c.sms * per_sm);
    if (c.ev_start && c.ev_stop) cudaEventRecord(c.ev_start, c.st);
    kernel<<<grid, threads, smem, c.st>>>(c.set, c.a, c.pal);
    if (c.ev_start && c.ev_stop) cudaEventRecord(c.ev_stop, c.st);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

template <class Kernel>
int launch_finish(Kernel kernel, const LaunchCfg& c) {
    int per_sm = 0;
    TDS_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 128, 0));
    TDS_REQUIRE(per_sm >= 1, "raster: finish kernel does not fit an SM");
    const int64_t cams = c.ncam - c.a.cam_begin;
    const unsigned grid = (unsigned)std::min<int64_t>((cams + 3) / 4, (int64_t)c.sms * per_sm);
    kernel<<<grid, 128, 0, c.st>>>(c.a, c.pal);
    TDS_LAUNCH_OK();
    return TDS_OK;
}

// two-pass form (64x64 tiles, K <= 15): launch_g32_draw = pass 1, launch_g32_finish = pass 2 (raster_g32.cu)
bool g32_two_pass_available(const LaunchCfg& c);
int launch_g32_draw(const LaunchCfg& c, bool lean);
int launch_g32_finish(const LaunchCfg& c, bool f32);
// bytes per camera of the hand-over buffers: bitplanes, face list, face count
inline int two_pass_planes(int K) { return K <= 5 ? 5 : (K <= 7 ? 7 : K); }      // planes stored per camera
inline int64_t two_pass_bytes_per_camera(int K) { return (int64_t)two_pass_planes(K) * 512 + (int64_t)kClipCap * 16 + 4; }

// defined in raster_g32.cu / raster_g128.cu / raster_g256.cu: picks the instantiation for (G, res, K, format, lean)
int launch_g32(const LaunchCfg& c, bool f32, bool lean);
int launch_g128(const LaunchCfg& c, bool f32, bool lean);
int launch_g256(const LaunchCfg& c, int G, bool f32, bool lean);

}  // namespace tds_raster
