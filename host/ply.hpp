// ply.hpp — pcl::io::savePLYFileBinary / PLYReader for PointXYZRGB without PCL (pose_functions.cpp:1618-1632).
// The header is byte-identical to what PCL 1.8 writes (see build/cloud.ply): binary little endian, vertex =
// 3 floats + 3 uchars (15 bytes), then "element camera 1" with 21 properties (84 bytes).
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "o3r.h"

namespace host {

inline bool save_ply_binary(const std::string& path, const o3r_point* pts, size_t n) {
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    fprintf(f,
            "ply\nformat binary_little_endian 1.0\ncomment PCL generated\nelement vertex %zu\n"
            "property float x\nproperty float y\nproperty float z\n"
            "property uchar red\nproperty uchar green\nproperty uchar blue\n"
            "element camera 1\n"
            "property float view_px\nproperty float view_py\nproperty float view_pz\n"
            "property float x_axisx\nproperty float x_axisy\nproperty float x_axisz\n"
            "property float y_axisx\nproperty float y_axisy\nproperty float y_axisz\n"
            "property float z_axisx\nproperty float z_axisy\nproperty float z_axisz\n"
            "property float focal\nproperty float scalex\nproperty float scaley\n"
            "property float centerx\nproperty float centery\n"
            "property int viewportx\nproperty int viewporty\n"
            "property float k1\nproperty float k2\nend_header\n",
            n);
    std::vector<uint8_t> rec(n * 15);
    for (size_t i = 0; i < n; ++i) {
        uint8_t* r = &rec[i * 15];
        memcpy(r, &pts[i].x, 12);
        r[12] = (pts[i].rgb >> 16) & 255; r[13] = (pts[i].rgb >> 8) & 255; r[14] = pts[i].rgb & 255;
    }
    bool ok = rec.empty() || fwrite(rec.data(), 1, rec.size(), f) == rec.size();
    // camera: origin (0,0,0), identity axes, focal/scale/center 0, viewport = (width = n, height = 1), k1 = k2 = 0
    float cam[21] = {0};
    cam[3] = cam[7] = cam[11] = 1.0f;
    int32_t vp[2] = {(int32_t)n, 1};
    memcpy(&cam[17], vp, 8);
    ok = ok && fwrite(cam, 4, 21, f) == 21;
    fclose(f);
    return ok;
}

// a triangle mesh (o3r_cloud_mesh): binary little endian, vertex = x y z nx ny nz (floats) + red green blue (uchars),
// 27 bytes; face = a uchar count (3) and three int vertex indices, 13 bytes
inline bool save_mesh_ply(const std::string& path, const o3r_point* pts, const float* normals, size_t n, const uint32_t* tris,
                          size_t m) {
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    fprintf(f,
            "ply\nformat binary_little_endian 1.0\nelement vertex %zu\n"
            "property float x\nproperty float y\nproperty float z\n"
            "property float nx\nproperty float ny\nproperty float nz\n"
            "property uchar red\nproperty uchar green\nproperty uchar blue\n"
            "element face %zu\nproperty list uchar int vertex_indices\nend_header\n",
            n, m);
    std::vector<uint8_t> rec(n * 27);
    for (size_t i = 0; i < n; ++i) {
        uint8_t* r = &rec[i * 27];
        memcpy(r, &pts[i].x, 12);
        memcpy(r + 12, normals + i * 3, 12);
        r[24] = (pts[i].rgb >> 16) & 255; r[25] = (pts[i].rgb >> 8) & 255; r[26] = pts[i].rgb & 255;
    }
    bool ok = rec.empty() || fwrite(rec.data(), 1, rec.size(), f) == rec.size();
    std::vector<uint8_t> face(m * 13);
    for (size_t t = 0; t < m; ++t) {
        uint8_t* r = &face[t * 13];
        r[0] = 3;
        memcpy(r + 1, tris + t * 3, 12);   // indices < 2^31: the int and uint32 bits agree
    }
    ok = ok && (face.empty() || fwrite(face.data(), 1, face.size(), f) == face.size());
    return fclose(f) == 0 && ok;
}

// reads the vertex element of a PLY written by PCL (binary_little_endian, x y z [+ red green blue])
inline bool read_ply(const std::string& path, std::vector<o3r_point>& out) {
    out.clear();
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    char line[512];
    size_t n = 0;
    bool binary = false, in_vertex = false, has_rgb = false;
    int n_props = 0;
    while (fgets(line, sizeof(line), f)) {
        if (!strncmp(line, "format binary_little_endian", 27)) binary = true;
        if (!strncmp(line, "element vertex", 14)) { n = strtoull(line + 14, nullptr, 10); in_vertex = true; continue; }
        if (!strncmp(line, "element", 7)) in_vertex = false;
        if (in_vertex && !strncmp(line, "property", 8)) { ++n_props; if (strstr(line, "red")) has_rgb = true; }
        if (!strncmp(line, "end_header", 10)) break;
    }
    if (!binary || n_props < 3) { fclose(f); return false; }
    const size_t rec = has_rgb ? 15 : 12;
    std::vector<uint8_t> buf(n * rec);
    if (fread(buf.data(), 1, buf.size(), f) != buf.size()) { fclose(f); return false; }
    fclose(f);
    out.resize(n);
    for (size_t i = 0; i < n; ++i) {
        const uint8_t* r = &buf[i * rec];
        memcpy(&out[i].x, r, 12);
        out[i].rgb = has_rgb ? ((uint32_t)r[12] << 16) | ((uint32_t)r[13] << 8) | r[14] : 0u;
    }
    return true;
}

}  // namespace host
