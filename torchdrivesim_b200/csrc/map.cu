// Host-side construction of the per-map grids (tds_map_create).  Runs once per map; nothing here
// is on the per-step path.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include <mutex>

#include "tds_map.cuh"
#include "tds_quad_table.h"

namespace tds {

int gather_maps(const tds_map_t* const* maps, int32_t n_maps, MapSetDev& out) {
    TDS_REQUIRE(maps && n_maps >= 1 && n_maps <= TDS_MAX_MAPS, "n_maps must be in [1,%d]", TDS_MAX_MAPS);
    int dev = -1;
    cudaGetDevice(&dev);
    for (int i = 0; i < n_maps; i++) {
        TDS_REQUIRE(maps[i], "null map handle at index %d", i);
        TDS_REQUIRE(maps[i]->device == dev, "map %d lives on device %d, current device is %d", i, maps[i]->device, dev);
        out.m[i] = maps[i]->dev;
    }
    for (int i = n_maps; i < TDS_MAX_MAPS; i++) out.m[i] = maps[0]->dev;
    return TDS_OK;
}

}  // namespace tds

namespace {

template <class T>
bool upload(const std::vector<T>& h, void** d, int64_t& bytes) {
    const size_t n = std::max<size_t>(h.size(), 1) * sizeof(T);
    if (cudaMalloc(d, n) != cudaSuccess) return false;
    if (!h.empty() && cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) return false;
    bytes += (int64_t)n;
    return true;
}

constexpr int kMaxDevices = 64;
std::mutex g_quad_mu;
void* g_quad_table[kMaxDevices] = {};

// library-owned, one per device, lives until the process ends
bool quad_table_ensure() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return false;
    std::lock_guard<std::mutex> lock(g_quad_mu);
    if (g_quad_table[dev]) return true;
    static std::vector<uint32_t> host;          // generated once per process by the reference's triangle rule
    if (host.empty()) {
        host.resize((size_t)tds::kQuadPatterns * tds::kQuadRows);
        tds::quad_table_fill(host.data());
    }
    void* d = nullptr;
    const size_t n = host.size() * sizeof(uint32_t);
    if (cudaMalloc(&d, n) != cudaSuccess) return false;
    if (cudaMemcpy(d, host.data(), n, cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(d); return false; }
    g_quad_table[dev] = d;
    return true;
}

}  // namespace

const void* tds::quad_table_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return nullptr;
    std::lock_guard<std::mutex> lock(g_quad_mu);
    return g_quad_table[dev];
}

extern "C" tds_map_t* tds_map_create(const float* h_verts, int32_t nv, const int32_t* h_faces, int32_t nf,
                                     const uint8_t* h_face_class, float raster_cell, float offroad_cell) {
    using namespace tds;
    if (!h_verts || !h_faces || !h_face_class || nv < 0 || nf < 0) {
        fail(TDS_ERR_INVALID_ARGUMENT, "map_create: null pointer or negative size");
        return nullptr;
    }
    if (raster_cell <= 0.f) raster_cell = 16.0f;
    if (offroad_cell <= 0.f) offroad_cell = 2.0f;
    for (int f = 0; f < nf; f++) {
        for (int k = 0; k < 3; k++) {
            const int v = h_faces[3 * f + k];
            if (v < 0 || v >= nv) {
                fail(TDS_ERR_INVALID_ARGUMENT, "map_create: face %d references vertex %d (nv=%d)", f, v, nv);
                return nullptr;
            }
        }
        if (h_face_class[f] >= TDS_MAX_CLASSES) {
            fail(TDS_ERR_INVALID_ARGUMENT, "map_create: face class %d >= %d", (int)h_face_class[f], TDS_MAX_CLASSES);
            return nullptr;
        }
    }
    float minx = 0.f, miny = 0.f, maxx = 1.f, maxy = 1.f;
    if (nv > 0) {
        minx = maxx = h_verts[0];
        miny = maxy = h_verts[1];
        for (int v = 0; v < nv; v++) {
            minx = std::min(minx, h_verts[2 * v]); maxx = std::max(maxx, h_verts[2 * v]);
            miny = std::min(miny, h_verts[2 * v + 1]); maxy = std::max(maxy, h_verts[2 * v + 1]);
        }
    }
    if (!quad_table_ensure()) {
        fail(TDS_ERR_CUDA, "map_create: could not build the quad pattern table: %s", cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    tds_map* m = new tds_map();
    MapDev& d = m->dev;
    for (auto& a : m->allocations) a = nullptr;
    cudaGetDevice(&m->device);
    int64_t bytes = 0;

    // ---------------- distinct static classes (informational; the raster keeps the class in each record)
    int slot_of[TDS_MAX_CLASSES];
    std::fill(slot_of, slot_of + TDS_MAX_CLASSES, -1);
    int n_slots = 0;
    for (int f = 0; f < nf; f++)
        if (slot_of[h_face_class[f]] < 0) slot_of[h_face_class[f]] = n_slots++;
    // ---------------- raster grid (vertex binning)
    d.rcs = raster_cell;
    d.rinv = 1.0f / raster_cell;
    d.rx0 = minx - 0.5f * raster_cell;
    d.ry0 = miny - 0.5f * raster_cell;
    d.rgx = std::max(1, (int)std::floor((maxx - d.rx0) / raster_cell) + 1);
    d.rgy = std::max(1, (int)std::floor((maxy - d.ry0) / raster_cell) + 1);
    d.n_slots = n_slots;
    for (int c = 0; c < TDS_MAX_CLASSES; c++) d.slot_of_class[c] = slot_of[c];
    const int nc = d.rgx * d.rgy;
    auto rcell_of = [&](float x, float y) {
        int cx = (int)std::floor(((double)x - d.rx0) / raster_cell), cy = (int)std::floor(((double)y - d.ry0) / raster_cell);
        cx = std::min(std::max(cx, 0), d.rgx - 1);
        cy = std::min(std::max(cy, 0), d.rgy - 1);
        return cy * d.rgx + cx;
    };
    // ---- strips of four faces over six vertices (see tds_map.cuh); the other faces become face records
    std::vector<uint8_t> in_strip((size_t)nf, 0);
    struct Strip { int v[6]; int cls; bool ordered; };
    std::vector<Strip> strips;
    auto finite_v = [&](int v) { return std::isfinite(h_verts[2 * v]) && std::isfinite(h_verts[2 * v + 1]); };
    // Faces f .. f+3 form a strip when, AS SETS, face k = {v_k, v_k+1, v_k+2} for six distinct vertices v_0 .. v_5 (the
    // pixels of a face do not depend on the order of its vertices).  Lane markings list their faces as
    // (a,b,c),(b,c,d),(c,d,e),(d,e,f) (lanelet2.py:253-283), road surfaces as (a,b,c),(c,b,d),(c,d,e),(e,d,f).
    auto has = [](const int32_t* q, int v) { return q[0] == v || q[1] == v || q[2] == v; };
    auto strip_of = [&](const int32_t* q, int* v) {
        const int32_t *f0 = q, *f1 = q + 3, *f2 = q + 6, *f3 = q + 9;
        int shared[2], ns = 0, v0 = -1;
        for (int k = 0; k < 3; k++) { if (has(f1, f0[k])) { if (ns < 2) shared[ns] = f0[k]; ns++; } else v0 = f0[k]; }
        if (ns != 2 || v0 < 0) return false;
        int v3 = -1, n3 = 0;
        for (int k = 0; k < 3; k++) if (!has(f0, f1[k])) { v3 = f1[k]; n3++; }
        if (n3 != 1) return false;
        // v2 = the shared vertex that face 2 keeps, v1 = the one it drops
        const bool k0 = has(f2, shared[0]), k1 = has(f2, shared[1]);
        if (k0 == k1) return false;
        const int v2 = k0 ? shared[0] : shared[1], v1 = k0 ? shared[1] : shared[0];
        if (!has(f2, v3)) return false;
        int v4 = -1, n4 = 0;
        for (int k = 0; k < 3; k++) if (f2[k] != v2 && f2[k] != v3) { v4 = f2[k]; n4++; }
        if (n4 != 1) return false;
        if (!has(f3, v3) || !has(f3, v4) || has(f3, v2)) return false;
        int v5 = -1, n5 = 0;
        for (int k = 0; k < 3; k++) if (f3[k] != v3 && f3[k] != v4) { v5 = f3[k]; n5++; }
        if (n5 != 1) return false;
        v[0] = v0; v[1] = v1; v[2] = v2; v[3] = v3; v[4] = v4; v[5] = v5;
        for (int a = 0; a < 6; a++)
            for (int b = a + 1; b < 6; b++)
                if (v[a] == v[b]) return false;
        return true;
    };
    for (int f = 0; f + 3 < nf;) {
        const int32_t* q = h_faces + 3 * (size_t)f;
        bool ok = h_face_class[f] == h_face_class[f + 1] && h_face_class[f] == h_face_class[f + 2] &&
                  h_face_class[f] == h_face_class[f + 3];
        Strip s;
        ok = ok && strip_of(q, s.v);
        if (ok) {
            s.cls = h_face_class[f];
            s.ordered = true;
            for (int k = 0; s.ordered && k < 3; k++) s.ordered = q[3 * (k + 1)] == q[3 * k + 1] && q[3 * (k + 1) + 1] == q[3 * k + 2];
            for (int k = 0; ok && k < 6; k++) ok = finite_v(s.v[k]);
            if (ok) {
                strips.push_back(s);
                for (int k = 0; k < 4; k++) in_strip[f + k] = 1;
                f += 4;
                continue;
            }
        }
        f++;
    }
    const bool dedupe_ok = d.rgx <= 8191 && d.rgy <= 8191;
    struct SRec { int key; int strip; uint32_t meta; };
    std::vector<SRec> srecs;
    srecs.reserve(strips.size() * 2);
    for (size_t s = 0; s < strips.size(); s++) {
        int cell[6];
        for (int k = 0; k < 6; k++) cell[k] = rcell_of(h_verts[2 * strips[s].v[k]], h_verts[2 * strips[s].v[k] + 1]);
        for (int k = 0; k < 6; k++) {
            bool seen = false;
            for (int j = 0; j < k; j++) seen |= cell[j] == cell[k];
            if (seen) continue;
            uint32_t meta = (uint32_t)strips[s].cls;
            if (dedupe_ok && k > 0) meta |= 32u | ((uint32_t)(cell[0] % d.rgx) << 6) | ((uint32_t)(cell[0] / d.rgx) << 19);
            srecs.push_back({cell[k], (int)s, meta});
        }
    }
    std::stable_sort(srecs.begin(), srecs.end(), [&](const SRec& a, const SRec& b) {
        if (a.key != b.key) return a.key < b.key;
        return strips[a.strip].cls < strips[b.strip].cls;
    });
    std::vector<int32_t> scell((size_t)nc + 1, 0);
    for (const SRec& r : srecs) scell[r.key + 1]++;
    for (size_t i = 0; i + 1 < scell.size(); i++) scell[i + 1] += scell[i];
    const size_t sblocks = (srecs.size() + 31) / 32;
    std::vector<float> srecdata(sblocks * 96 * 4, 0.f);
    std::vector<uint32_t> smeta(std::max<size_t>(srecs.size(), 1), 0u);
    for (size_t i = 0; i < srecs.size(); i++) {
        const Strip& s = strips[srecs[i].strip];
        float* base = &srecdata[(i >> 5) * 96 * 4 + (i & 31) * 4];
        for (int k = 0; k < 6; k++) {
            float* p = base + (k >> 1) * 32 * 4;
            p[k & 1] = h_verts[2 * s.v[k]];
            p[2 + (k & 1)] = h_verts[2 * s.v[k] + 1];
        }
        smeta[i] = srecs[i].meta;
    }
    struct Rec { int key; int face; int own; };
    auto build_face_records = [&](bool all, std::vector<int32_t>& cells, std::vector<float>& data) {
        std::vector<Rec> recs;
        recs.reserve((size_t)nf * 2);
        for (int f = 0; f < nf; f++) {
            if (!all && in_strip[f]) continue;
            int cell[3];
            for (int k = 0; k < 3; k++) cell[k] = rcell_of(h_verts[2 * h_faces[3 * f + k]], h_verts[2 * h_faces[3 * f + k] + 1]);
            for (int k = 0; k < 3; k++) {
                bool seen = false;
                for (int j = 0; j < k; j++) seen |= cell[j] == cell[k];
                if (seen) continue;
                int own = 0;
                for (int j = 0; j < 3; j++) own |= (cell[j] == cell[k]) << j;
                recs.push_back({cell[k], f, own});
            }
        }
        // cell-major (all classes of a cell together: the kernel makes ONE pass over the candidates and keeps
        // painter's order in per-class bitplanes); inside a cell by class, then by face
        std::stable_sort(recs.begin(), recs.end(), [&](const Rec& a, const Rec& b) {
            if (a.key != b.key) return a.key < b.key;
            return h_face_class[a.face] < h_face_class[b.face];
        });
        cells.assign((size_t)nc + 1, 0);
        for (const Rec& r : recs) cells[r.key + 1]++;
        for (size_t i = 0; i + 1 < cells.size(); i++) cells[i + 1] += cells[i];
        data.assign(recs.size() * 8, 0.f);
        for (size_t i = 0; i < recs.size(); i++) {
            const int f = recs[i].face;
            for (int k = 0; k < 3; k++) {
                data[8 * i + 2 * k] = h_verts[2 * h_faces[3 * f + k]];
                data[8 * i + 2 * k + 1] = h_verts[2 * h_faces[3 * f + k] + 1];
            }
            const int meta = recs[i].own | ((int)h_face_class[f] << 8);
            memcpy(&data[8 * i + 6], &meta, sizeof(int));
        }
        return (int32_t)recs.size();
    };
    std::vector<int32_t> rcell, rcell_all;
    std::vector<float> recdata, recdata_all;
    const int32_t n_recs = build_face_records(false, rcell, recdata);
    if (strips.empty()) { rcell_all = rcell; recdata_all = recdata; }
    else build_face_records(true, rcell_all, recdata_all);
    // median length of the long side of a lane-marking strip (vertex 0 -> vertex 1 of the strips whose faces are listed
    // as (a,b,c),(b,c,d),...): the host side decides from it whether such a strip is a handful of pixels at the
    // requested zoom.  Road-surface strips are not counted: their faces are always drawn.
    d.strip_len = 0.f;
    {
        std::vector<float> len;
        for (size_t i = 0; i < strips.size(); i++) {
            if (!strips[i].ordered) continue;
            const float dx = h_verts[2 * strips[i].v[1]] - h_verts[2 * strips[i].v[0]];
            const float dy = h_verts[2 * strips[i].v[1] + 1] - h_verts[2 * strips[i].v[0] + 1];
            len.push_back(std::sqrt(dx * dx + dy * dy));
        }
        if (!len.empty()) {
            std::nth_element(len.begin(), len.begin() + len.size() / 2, len.end());
            d.strip_len = len[len.size() / 2];
        }
    }
    // ---------------- offroad grid (bounding-box binning)
    d.ocs = offroad_cell;
    d.oinv = 1.0f / offroad_cell;
    d.ox0 = minx - 0.5f * offroad_cell;
    d.oy0 = miny - 0.5f * offroad_cell;
    d.ogx = std::max(1, (int)std::floor((maxx - d.ox0) / offroad_cell) + 1);
    d.ogy = std::max(1, (int)std::floor((maxy - d.oy0) / offroad_cell) + 1);
    d.nf = nf;
    const int onc = d.ogx * d.ogy;
    auto oc = [&](float v, float o, int g) {
        int c = (int)std::floor(((double)v - o) / offroad_cell);
        return std::min(std::max(c, 0), g - 1);
    };
    std::vector<int32_t> ocell((size_t)onc + 1, 0);
    std::vector<float> tri((size_t)nf * 6);
    const float eps = 1e-3f;
    std::vector<int32_t> oidx, cursor;
    for (int pass = 0; pass < 2; pass++) {
        if (pass == 1) {
            for (int i = 0; i < onc; i++) ocell[i + 1] += ocell[i];
            cursor.assign(ocell.begin(), ocell.end() - 1);
            oidx.assign((size_t)ocell[onc], 0);
        }
        for (int f = 0; f < nf; f++) {
            float x[3], y[3];
            for (int k = 0; k < 3; k++) { x[k] = h_verts[2 * h_faces[3 * f + k]]; y[k] = h_verts[2 * h_faces[3 * f + k] + 1]; }
            if (pass == 0) for (int k = 0; k < 3; k++) { tri[6 * f + 2 * k] = x[k]; tri[6 * f + 2 * k + 1] = y[k]; }
            const int cx0 = oc(std::min({x[0], x[1], x[2]}) - eps, d.ox0, d.ogx), cx1 = oc(std::max({x[0], x[1], x[2]}) + eps, d.ox0, d.ogx);
            const int cy0 = oc(std::min({y[0], y[1], y[2]}) - eps, d.oy0, d.ogy), cy1 = oc(std::max({y[0], y[1], y[2]}) + eps, d.oy0, d.ogy);
            for (int cy = cy0; cy <= cy1; cy++)
                for (int cx = cx0; cx <= cx1; cx++) {
                    if (pass == 0) ocell[cy * d.ogx + cx + 1]++;
                    else oidx[cursor[cy * d.ogx + cx]++] = f;
                }
        }
    }
    m->info.offroad_entries = (int32_t)oidx.size();
    // inline the triangle data per cell entry, largest faces first
    auto area2 = [&](int f) {
        const float* t = &tri[6 * (size_t)f];
        return std::fabs((t[2] - t[0]) * (t[5] - t[1]) - (t[3] - t[1]) * (t[4] - t[0]));
    };
    std::vector<float> orec(oidx.size() * 8, 0.f);
    for (int c = 0; c < onc; c++) {
        std::stable_sort(oidx.begin() + ocell[c], oidx.begin() + ocell[c + 1],
                         [&](int a, int b) { return area2(a) > area2(b); });
        for (int e = ocell[c]; e < ocell[c + 1]; e++) {
            const int f = oidx[e];
            for (int k = 0; k < 6; k++) orec[8 * (size_t)e + k] = tri[6 * (size_t)f + k];
            memcpy(&orec[8 * (size_t)e + 6], &f, sizeof(int));
        }
    }
    if (!(upload(recdata, &m->allocations[0], bytes) && upload(rcell, &m->allocations[1], bytes) &&
          upload(tri, &m->allocations[2], bytes) && upload(ocell, &m->allocations[3], bytes) &&
          upload(orec, &m->allocations[4], bytes) && upload(srecdata, &m->allocations[5], bytes) &&
          upload(smeta, &m->allocations[6], bytes) && upload(scell, &m->allocations[7], bytes) &&
          upload(recdata_all, &m->allocations[8], bytes) && upload(rcell_all, &m->allocations[9], bytes))) {
        fail(TDS_ERR_CUDA, "map_create: device allocation/upload failed: %s", cudaGetErrorString(cudaGetLastError()));
        tds_map_destroy(m);
        return nullptr;
    }
    d.rec = (const float4*)m->allocations[0];
    d.rcell = (const int32_t*)m->allocations[1];
    d.tri = (const float*)m->allocations[2];
    d.ocell = (const int32_t*)m->allocations[3];
    d.orec = (const float4*)m->allocations[4];
    d.srec = (const float4*)m->allocations[5];
    d.smeta = (const uint32_t*)m->allocations[6];
    d.scell = (const int32_t*)m->allocations[7];
    d.rec_all = (const float4*)m->allocations[8];
    d.rcell_all = (const int32_t*)m->allocations[9];
    // ---------------- offroad distance bound (computed on the device from the offroad grid just uploaded)
    d.bcs = 0.25f;
    d.bx0 = minx - 1.0f;
    d.by0 = miny - 1.0f;
    auto nsub = [&](float lo, float hi) { return (int64_t)std::floor(((double)hi + 1.0 - lo) / d.bcs) + 1; };
    while (nsub(d.bx0, maxx) * nsub(d.by0, maxy) > ((int64_t)16 << 20)) d.bcs *= 2.0f;
    d.binv = 1.0f / d.bcs;
    d.bgx = (int32_t)nsub(d.bx0, maxx);
    d.bgy = (int32_t)nsub(d.by0, maxy);
    const size_t nb = (size_t)d.bgx * d.bgy;
    if (cudaMalloc(&m->allocations[10], nb) != cudaSuccess) {
        fail(TDS_ERR_CUDA, "map_create: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        tds_map_destroy(m);
        return nullptr;
    }
    if (offroad_bound_build(d, (uint8_t*)m->allocations[10]) != TDS_OK) {     // the error is recorded by the builder
        tds_map_destroy(m);
        return nullptr;
    }
    bytes += (int64_t)nb;
    d.obound = (const uint8_t*)m->allocations[10];
    m->info.n_verts = nv; m->info.n_faces = nf;
    m->info.raster_gx = d.rgx; m->info.raster_gy = d.rgy; m->info.raster_records = n_recs; m->info.raster_strips = (int32_t)srecs.size();
    m->info.offroad_gx = d.ogx; m->info.offroad_gy = d.ogy;
    m->info.raster_cell = raster_cell; m->info.offroad_cell = offroad_cell;
    m->info.min_x = minx; m->info.min_y = miny; m->info.max_x = maxx; m->info.max_y = maxy;
    m->info.device_bytes = bytes;
    return m;
}

extern "C" void tds_map_destroy(tds_map_t* map) {
    if (!map) return;
    for (auto& a : map->allocations) if (a) cudaFree(a);
    delete map;
}

extern "C" int tds_map_info(const tds_map_t* map, tds_map_info_t* out) {
    TDS_REQUIRE(map && out, "map_info: null pointer");
    *out = map->info;
    return TDS_OK;
}

extern "C" int tds_map_offroad_bound(const tds_map_t* map, float* h_geom, int32_t* h_dims, uint8_t* h_codes) {
    TDS_REQUIRE(map && h_geom && h_dims, "map_offroad_bound: null pointer");
    const tds::MapDev& d = map->dev;
    h_geom[0] = d.bx0; h_geom[1] = d.by0; h_geom[2] = d.bcs; h_geom[3] = 1.0f / tds::kBoundPerMetre;
    h_dims[0] = d.bgx; h_dims[1] = d.bgy;
    if (h_codes && cudaMemcpy(h_codes, d.obound, (size_t)d.bgx * d.bgy, cudaMemcpyDeviceToHost) != cudaSuccess)
        return tds::fail(TDS_ERR_CUDA, "map_offroad_bound: copy failed: %s", cudaGetErrorString(cudaGetLastError()));
    return TDS_OK;
}
