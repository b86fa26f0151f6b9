// Static map acceleration structures (device view).  Built once per map by tds_map_create.
#pragma once
#include <math_constants.h>

#include "tds_common.cuh"

namespace tds {

constexpr int kMaxSlots = 8;        // distinct palette classes among the static faces of one map
constexpr int kMaxRasterRows = 64;  // grid rows a single camera may touch

struct MapDev {
    // ---- raster grid: triangles binned by the cell of each VERTEX (the reference keeps a face
    // iff any vertex is inside the view quad, mesh.py:311-313).  A record is two float4:
    //   (x0, y0, x1, y1), (x2, y2, meta, unused); meta = own_bits | class << 8, own bit i set = vertex i lies
    //   in this cell.  Records are sorted by cell (row-major), so one grid row is one contiguous range.
    const float4* rec;
    const int32_t* rcell;           // [rgx * rgy + 1] CSR offsets into rec (in records)
    // ---- strips: four consecutive faces (a,b,c), (b,c,d), (c,d,e), (d,e,f) of one class - what the reference's
    // line_segments_to_mesh (lanelet2.py:253-283) emits for every lane-marking segment - are kept as ONE record of
    // six vertices instead of four face records, binned by the cell of each of the six vertices.  Vertex data in
    // blocks of 32 strips, structure of arrays: block b = 3 x 32 float4, strip j of the block at float4 index
    // b * 96 + p * 32 + j, p = 0: (x0, x1, y0, y1), p = 1: (x2, x3, y2, y3), p = 2: (x4, x5, y4, y5).
    // smeta = class | secondary << 5 | primary cell column << 6 | primary cell row << 19: a copy outside the cell of
    // vertex 0 (secondary) is skipped when the camera also scans that primary cell.
    const float4* srec;
    const uint32_t* smeta;
    const int32_t* scell;           // [rgx * rgy + 1] CSR offsets into srec / smeta (in strips)
    // rec / rcell hold the faces that are NOT part of a strip; rec_all / rcell_all hold every face in the same record
    // format: what a camera walks when strips do not pay (large tiles / close zoom, where no strip is a handful of
    // pixels and every face of a strip would have to be classified on its own anyway).
    const float4* rec_all;
    const int32_t* rcell_all;
    float strip_len;                // median length (metres) of the long side of the strips, 0 without strips
    float rx0, ry0, rcs, rinv;
    int32_t rgx, rgy, n_slots;
    int32_t slot_of_class[TDS_MAX_CLASSES];   // -1: the map has no face of that class
    // ---- offroad grid: triangles binned by bounding box overlap
    const float* tri;               // [nf][6] x0,y0,x1,y1,x2,y2 (indexed by face, for the backward)
    const int32_t* ocell;           // [ogx * ogy + 1] CSR offsets into orec (in records)
    const float4* orec;             // per cell entry: (x0,y0,x1,y1), (x2,y2, face index bits, unused); within a
                                    // cell the faces are sorted by decreasing area (a containing face is found early)
    float ox0, oy0, ocs, oinv;
    int32_t ogx, ogy, nf;
    // ---- offroad distance bound: one byte per subcell of a fine grid over the map's bounding box (1 m margin),
    // row-major.  Code q < 255: every point of the subcell is within q / kBoundPerMetre metres of the road mesh by the
    // reference's own fp32 distance (offroad.cu, offroad_bound_kernel); 255: unknown.  Subcells are 0.25 m (a power of
    // two, so the lookup is exact), coarser for maps too large for 16 M subcells.
    const uint8_t* obound;
    float bx0, by0, bcs, binv;
    int32_t bgx, bgy;
};

constexpr int kBoundPerMetre = 64;  // bound codes are multiples of 1/64 m: (q/64)^2 <= thr is exact as q*q <= thr*4096
constexpr int kBoundUnknown = 255;

struct MapSetDev {
    MapDev m[TDS_MAX_MAPS];
};

// ---- lane-marking segments (tds_nearest_map_segments): segment s is the s-th strip of the map whose faces are listed
// as (a,b,c),(b,c,d),(c,d,e),(d,e,f), in face order; its endpoints are (c, d).  Kept apart from MapDev, so the raster
// and offroad kernels see the same map struct as without them.  Grid: square cells of `cs` metres over the bounding
// box of the segment midpoints, row-major, CSR; each segment is listed once, in the cell of its midpoint, so every
// point of a segment listed in a cell lies within `slack` (the largest half-length) of that cell.
struct SegDev {
    const float4* seg;              // [n] x0, y0, x1, y1
    const uint8_t* kind;            // [n] palette class of the strip
    const int32_t* cell;            // [gx * gy + 1] CSR offsets into ent
    const int32_t* ent;             // [n] segment indices, by cell, ascending within a cell
    float x0, y0, cs, inv, slack;
    int32_t gx, gy, n;
};

struct SegSetDev {
    SegDev m[TDS_MAX_MAPS];
};

// One warp's walk over the segment grid around (x, y), what the map-segment and range-scan kernels search it with.
// The cells are taken ring by ring around the point's cell (clamped into the grid, so a point off the map starts at the
// nearest border cell): ring r is the 8 r cells at Chebyshev distance r, in side order.  The lanes take 32 cells of a
// ring at a time, and a scan of their entry counts deals the cells' entries to the lanes, 32 at a time, whatever the
// cells hold.  After ring r every unsearched cell lies outside the searched square, at distance >= dmin from (x, y),
// and every point of a segment listed in it at distance >= dmin - slack.
// visit(s): called by all 32 lanes once per round of 32 entries; s = segment index, or -1 for a lane with no entry
//           (so visit may contain warp collectives such as tds::near_insert).
// done(dmin): called by all 32 lanes after each ring with the double-precision distance from (x, y) to the unsearched
//           cells (CUDART_INF when none is left on any side); returns a warp-uniform bool: stop.
// Precondition: x, y finite and m.n > 0.
template <class Visit, class Done>
__device__ __forceinline__ void seg_grid_walk(const SegDev& m, float x, float y, int lane, Visit visit, Done done) {
    const int cx = (int)fminf(fmaxf(floorf((x - m.x0) * m.inv), 0.0f), (float)(m.gx - 1));
    const int cy = (int)fminf(fmaxf(floorf((y - m.y0) * m.inv), 0.0f), (float)(m.gy - 1));
    const int rmax = max(max(cx, m.gx - 1 - cx), max(cy, m.gy - 1 - cy));
    for (int r = 0; r <= rmax; r++) {
        const int ncells = r == 0 ? 1 : 8 * r;
        for (int c0 = 0; c0 < ncells; c0 += 32) {
            int beg = 0, cnt = 0;
            const int q = c0 + lane;
            if (q < ncells) {
                int px = cx, py = cy;
                if (r > 0) {
                    const int side = q / (2 * r), off = q - side * 2 * r;
                    px = side == 0 ? cx - r + off : side == 1 ? cx + r : side == 2 ? cx + r - off : cx - r;
                    py = side == 0 ? cy - r : side == 1 ? cy - r + off : side == 2 ? cy + r : cy + r - off;
                }
                if (px >= 0 && px < m.gx && py >= 0 && py < m.gy) {
                    const int cell = py * m.gx + px;
                    beg = m.cell[cell];
                    cnt = m.cell[cell + 1] - beg;
                }
            }
            int incl = cnt;                                        // inclusive scan of the lanes' counts
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            for (int t0 = 0; t0 < total; t0 += 32) {
                const int t = t0 + lane;
                int pos = 0;                                       // the lane whose cell holds entry t: first incl > t
#pragma unroll
                for (int step = 16; step > 0; step >>= 1)
                    if (__shfl_sync(0xffffffffu, incl, pos + step - 1) <= t) pos += step;
                const int cbeg = __shfl_sync(0xffffffffu, beg, pos), cfirst = __shfl_sync(0xffffffffu, incl - cnt, pos);
                int s = -1;
                if (t < total) {
                    s = m.ent[cbeg + t - cfirst];
                    __builtin_assume(s >= 0);                      // so that visit's s >= 0 folds into t < total
                }
                visit(s);
            }
        }
        // distance to the unsearched cells (double: exact for float inputs, whatever the map's coordinates)
        double dmin = CUDART_INF;
        if (cx - r > 0) dmin = fmin(dmin, (double)x - ((double)m.x0 + (double)(cx - r) * m.cs));
        if (cx + r < m.gx - 1) dmin = fmin(dmin, ((double)m.x0 + (double)(cx + r + 1) * m.cs) - (double)x);
        if (cy - r > 0) dmin = fmin(dmin, (double)y - ((double)m.y0 + (double)(cy - r) * m.cs));
        if (cy + r < m.gy - 1) dmin = fmin(dmin, ((double)m.y0 + (double)(cy + r + 1) * m.cs) - (double)y);
        if (done(dmin)) break;
    }
}

}  // namespace tds

struct tds_map {
    tds::MapDev dev;
    tds::SegDev seg;
    tds_map_info_t info;
    void* allocations[15];
    int device;
};

namespace tds {
int gather_maps(const tds_map_t* const* maps, int32_t n_maps, MapSetDev& out);
int gather_segments(const tds_map_t* const* maps, int32_t n_maps, SegSetDev& out);
// coverage patterns of sliver quads (tds_quad_table.h) on the current device: built and uploaded by the first
// tds_map_create on that device (never inside a raster call, which may be under CUDA-graph capture); NULL before that
const void* quad_table_device();
// fills d.obound (d.bgx * d.bgy bytes, device) from the offroad grid of d; synchronous (offroad.cu)
int offroad_bound_build(const MapDev& d, uint8_t* obound);
}
