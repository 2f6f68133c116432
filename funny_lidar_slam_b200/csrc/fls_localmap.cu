// fls_localmap.cu — the localization-mode map path around the matcher (SURVEY.md §8f-4):
//   * Localization::LoadLocalMap, the global-map branch (src/slam/localization.cpp:364-410 upstream): the global map stays in HBM;
//     when the pose comes within 50 m of an edge of the current local map (or there is none) a +-100 m pcl::CropBox around the
//     pose is cut on the device (stream compaction, input order kept) and handed to AddCloudToLocalMap without leaving the GPU;
//   * the PCD files behind it (pcl::io::loadPCDFile / savePCDFileBinary as used by include/common/keyframe.h:24-74 and
//     localization.cpp:283-300): a reader / writer for x y z intensity clouds, DATA binary and ascii.
#include <cub/cub.cuh>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "fls_handle.h"

namespace fls {
namespace {

// pcl::CropBox without a transform: keeps min <= p <= max on x, y, z (float compare), drops non-finite points
__global__ void crop_flags_kernel(const float4* __restrict__ p, size_t n, float x0, float y0, float z0, float x1, float y1, float z1,
                                  unsigned char* __restrict__ keep) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 q = p[i];
    const bool fin = isfinite(q.x) && isfinite(q.y) && isfinite(q.z);
    keep[i] = (fin && q.x >= x0 && q.y >= y0 && q.z >= z0 && q.x <= x1 && q.y <= y1 && q.z <= z1) ? 1 : 0;
}

}  // namespace

int Handle::set_global_map(const void* pts, size_t n, size_t stride) {
    const float4* d = upload(pts, n, stride, stage);
    global_map.reserve(n + 1);
    if (n) FLS_CUDA(cudaMemcpyAsync(global_map.p, d, n * sizeof(float4), cudaMemcpyDeviceToDevice, stream));
    global_n = n;
    have_edge = false;  // `first || !has_init_`: local_map_edge_.clear() (:369-373)
    return FLS_OK;
}

int Handle::update_local_map(const double* T, int* updated, size_t* n_local) {
    if (updated) *updated = 0;
    if (global_n == 0) return FLS_ERR_NO_MAP;
    const double pos[3] = {T[12], T[13], T[14]};
    bool need = !have_edge;  // :375-376
    if (have_edge) {
        for (int i = 0; i < 3; ++i) {  // :378-385
            if (std::fabs(pos[i] - local_edge[i]) > 50.0 && std::fabs(pos[i] - local_edge[i + 3]) > 50.0) continue;
            need = true;
            break;
        }
    }
    if (!need) return FLS_OK;
    for (int i = 0; i < 3; ++i) {  // :392-399
        local_edge[i] = pos[i] - 100.0;
        local_edge[i + 3] = pos[i] + 100.0;
    }
    have_edge = true;
    crop_keep.reserve(global_n + 1);
    stage2.reserve(global_n + 1);
    scratch.num_runs.reserve(2);
    crop_flags_kernel<<<(unsigned)((global_n + 255) / 256), 256, 0, stream>>>(global_map.p, global_n, (float)local_edge[0], (float)local_edge[1],
                                                                            (float)local_edge[2], (float)local_edge[3], (float)local_edge[4],
                                                                            (float)local_edge[5], crop_keep.p);  // :401-402 .cast<float>()
    size_t tb = 0;
    cub::DeviceSelect::Flagged(nullptr, tb, global_map.p, crop_keep.p, stage2.p, scratch.num_runs.p, (int)global_n, stream);
    scratch.cub_tmp.reserve(tb + 256);
    tb = scratch.cub_tmp.cap;
    FLS_CUDA(cub::DeviceSelect::Flagged(scratch.cub_tmp.p, tb, global_map.p, crop_keep.p, stage2.p, scratch.num_runs.p, (int)global_n, stream));
    FLS_CUDA(cudaMemcpyAsync(scratch.h_num_runs, scratch.num_runs.p, sizeof(int), cudaMemcpyDeviceToHost, stream));
    FLS_CUDA(cudaStreamSynchronize(stream));
    const size_t m = (size_t)*scratch.h_num_runs;
    launches += 2;
    if (n_local) *n_local = m;
    if (updated) *updated = 1;
    if (m == 0) return FLS_OK;  // `local_map->empty()`: the caller gives up (:129-131); the matcher keeps its map
    // matcher_->AddCloudToLocalMap({*local_map}) (:135, :222) — the cloud is already on the device
    return add_cloud(stage2.p, m);
}

// ---- PCD --------------------------------------------------------------------------------------------------------------------
// Reads FIELDS containing x y z (F 4) and optionally intensity (F 4) from a PCD v0.7 file, DATA ascii or binary.
int pcd_read(const char* path, std::vector<float>& xyzi, std::string& err) {
    std::ifstream f(path, std::ios::binary);
    if (!f) {
        err = std::string("cannot open ") + path;
        return FLS_ERR_INVALID_ARG;
    }
    std::vector<std::string> fields;
    std::vector<int> sizes, counts;
    std::vector<char> types;
    size_t points = 0, width = 0, height = 1;
    std::string data;
    std::string line;
    while (std::getline(f, line)) {
        if (!line.empty() && line.back() == '\r') line.pop_back();
        if (line.empty() || line[0] == '#') continue;
        std::istringstream ss(line);
        std::string key;
        ss >> key;
        if (key == "FIELDS") {
            std::string s;
            while (ss >> s) fields.push_back(s);
        } else if (key == "SIZE") {
            int v;
            while (ss >> v) sizes.push_back(v);
        } else if (key == "TYPE") {
            char c;
            while (ss >> c) types.push_back(c);
        } else if (key == "COUNT") {
            int v;
            while (ss >> v) counts.push_back(v);
        } else if (key == "WIDTH") {
            ss >> width;
        } else if (key == "HEIGHT") {
            ss >> height;
        } else if (key == "POINTS") {
            ss >> points;
        } else if (key == "DATA") {
            ss >> data;
            break;
        }
    }
    if (points == 0) points = width * height;
    if (fields.empty() || sizes.size() != fields.size() || types.size() != fields.size()) {
        err = "malformed PCD header";
        return FLS_ERR_INVALID_ARG;
    }
    if (counts.empty()) counts.assign(fields.size(), 1);
    int off[4] = {-1, -1, -1, -1}, col[4] = {-1, -1, -1, -1};
    int stride = 0, ncol = 0;
    for (size_t k = 0; k < fields.size(); ++k) {
        const char* names[4] = {"x", "y", "z", "intensity"};
        for (int a = 0; a < 4; ++a)
            if (fields[k] == names[a]) {
                if (sizes[k] != 4 || types[k] != 'F') {
                    err = "x / y / z / intensity must be 4-byte floats";
                    return FLS_ERR_UNSUPPORTED;
                }
                off[a] = stride;
                col[a] = ncol;
            }
        stride += sizes[k] * counts[k];
        ncol += counts[k];
    }
    if (off[0] < 0 || off[1] < 0 || off[2] < 0) {
        err = "PCD without x y z";
        return FLS_ERR_INVALID_ARG;
    }
    xyzi.assign(points * 4, 0.f);
    if (data == "binary") {
        std::vector<char> rec(stride);
        for (size_t i = 0; i < points; ++i) {
            if (!f.read(rec.data(), stride)) {
                err = "PCD body shorter than POINTS";
                return FLS_ERR_INVALID_ARG;
            }
            for (int a = 0; a < 4; ++a)
                if (off[a] >= 0) std::memcpy(&xyzi[4 * i + a], rec.data() + off[a], 4);
        }
    } else if (data == "ascii") {
        for (size_t i = 0; i < points; ++i) {
            if (!std::getline(f, line)) {
                err = "PCD body shorter than POINTS";
                return FLS_ERR_INVALID_ARG;
            }
            std::istringstream ss(line);
            for (int c = 0; c < ncol; ++c) {
                double v;
                ss >> v;
                for (int a = 0; a < 4; ++a)
                    if (col[a] == c) xyzi[4 * i + a] = (float)v;
            }
        }
    } else {
        err = "PCD DATA " + data + " not supported (binary_compressed needs LZF)";
        return FLS_ERR_UNSUPPORTED;
    }
    return FLS_OK;
}

// pcl::io::savePCDFileBinary of a PointXYZI cloud: FIELDS x y z intensity, 16-byte records
int pcd_write(const char* path, const float* xyzi, size_t n, std::string& err) {
    std::ofstream f(path, std::ios::binary | std::ios::trunc);
    if (!f) {
        err = std::string("cannot open ") + path;
        return FLS_ERR_INVALID_ARG;
    }
    f << "# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z intensity\nSIZE 4 4 4 4\nTYPE F F F F\nCOUNT 1 1 1 1\nWIDTH " << n
      << "\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS " << n << "\nDATA binary\n";
    f.write(reinterpret_cast<const char*>(xyzi), (std::streamsize)(n * 16));
    return f ? FLS_OK : FLS_ERR_INVALID_ARG;
}

}  // namespace fls
