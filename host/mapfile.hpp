// mapfile.hpp — map checkpoint files (.o3rmap), the same bytes as online_3d_reconstruction_b200/mapfile.py writes and reads.
// Little-endian: a 64-byte header {magic "O3RMAP01", u32 version 1, u32 kind (1 = o3r_cell records of 40 bytes, 2 = o3r_point
// records of 16 bytes), f64 voxel_size, u32 world, u32 rank, u64 n_records, zero up to byte 64}, then the records.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "o3r.h"

namespace host {

enum { MAP_KIND_CELLS = 1, MAP_KIND_POINTS = 2 };

struct MapHeader {
    char magic[8];
    uint32_t version, kind;
    double voxel_size;
    uint32_t world, rank;
    uint64_t n_records;
    uint8_t reserved[24];
};
static_assert(sizeof(MapHeader) == 64, "map file header is 64 bytes");
static_assert(sizeof(o3r_cell) == 40 && sizeof(o3r_point) == 16, "map file records");

inline size_t map_record_bytes(uint32_t kind) { return kind == MAP_KIND_CELLS ? sizeof(o3r_cell) : sizeof(o3r_point); }

// (this host is little-endian, as the format: the structs are written as they are)
inline bool save_map(const std::string& path, uint32_t kind, const void* records, uint64_t n, double voxel_size,
                     uint32_t world = 1, uint32_t rank = 0) {
    MapHeader h;
    memset(&h, 0, sizeof(h));
    memcpy(h.magic, "O3RMAP01", 8);
    h.version = 1; h.kind = kind; h.voxel_size = voxel_size; h.world = world; h.rank = rank; h.n_records = n;
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    bool ok = fwrite(&h, sizeof(h), 1, f) == 1;
    if (ok && n) ok = fwrite(records, map_record_bytes(kind), n, f) == n;
    return fclose(f) == 0 && ok;
}

// Reads a map file for a context that keeps records of `kind` on a grid of `voxel_size`; on refusal returns false with the
// reason in *err.  records receives n_records * record size bytes.
inline bool load_map(const std::string& path, uint32_t kind, double voxel_size, std::vector<uint8_t>& records, uint64_t* n,
                     std::string* err) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) { *err = path + ": cannot open"; return false; }
    auto fail = [&](const std::string& m) { fclose(f); *err = path + ": " + m; return false; };
    fseek(f, 0, SEEK_END);
    const long size = ftell(f);
    fseek(f, 0, SEEK_SET);
    MapHeader h;
    if (size < (long)sizeof(h) || fread(&h, sizeof(h), 1, f) != 1) return fail("shorter than the 64-byte header");
    if (memcmp(h.magic, "O3RMAP01", 8) != 0) return fail("not a map file (bad magic)");
    if (h.version != 1) return fail("map file version " + std::to_string(h.version) + ", this build reads 1");
    if (h.kind != MAP_KIND_CELLS && h.kind != MAP_KIND_POINTS) return fail("unknown record kind " + std::to_string(h.kind));
    const size_t rb = map_record_bytes(h.kind);
    if (h.n_records > ((uint64_t)1 << 48) || (uint64_t)size != sizeof(h) + h.n_records * rb)
        return fail(std::to_string(size) + " bytes, the header announces " + std::to_string(h.n_records) + " records");
    if (h.kind != kind)
        return fail(std::string("holds ") + (h.kind == MAP_KIND_CELLS ? "cells" : "points") + ", this run keeps " +
                    (kind == MAP_KIND_CELLS ? "cells" : "points") + " (--dont_downsample differs)");
    if (memcmp(&h.voxel_size, &voxel_size, sizeof(double)) != 0) {
        char b[160];
        snprintf(b, sizeof(b), "saved at voxel_size %.17g, this run uses %.17g", h.voxel_size, voxel_size);
        return fail(b);
    }
    records.resize(h.n_records * rb);
    if (h.n_records && fread(records.data(), rb, h.n_records, f) != h.n_records) return fail("short read");
    fclose(f);
    *n = h.n_records;
    return true;
}

}  // namespace host
