// Static map acceleration structures (device view).  Built once per map by tds_map_create.
#pragma once
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

}  // namespace tds

struct tds_map {
    tds::MapDev dev;
    tds_map_info_t info;
    void* allocations[11];
    int device;
};

namespace tds {
int gather_maps(const tds_map_t* const* maps, int32_t n_maps, MapSetDev& out);
// coverage patterns of sliver quads (tds_quad_table.h) on the current device: built and uploaded by the first
// tds_map_create on that device (never inside a raster call, which may be under CUDA-graph capture); NULL before that
const void* quad_table_device();
// fills d.obound (d.bgx * d.bgy bytes, device) from the offroad grid of d; synchronous (offroad.cu)
int offroad_bound_build(const MapDev& d, uint8_t* obound);
}
