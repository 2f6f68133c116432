// fls_loam.cu — K5: the kd-tree LOAM plug-ins as one persistent Gauss-Newton kernel.
//
//   LoamPointToPlaneKdtree::Match  (include/registration/loam_point_to_plane_kdtree.h:82-157,204-288 upstream)
//   LoamFull::Match / CornerMatch / PlanarMatch  (include/registration/loam_full_kdtree.h:106-204,211-273,275-345)
//
// Both ask pcl::KdTreeFLANN for the EXACT 5 nearest map points of every transformed feature point — no radius: the
// LoamFull gate `d2[4] > point_search_thres` is applied after the search (:227,:291) and the kd-tree point-to-plane
// variant has no gate at all.  The GPU index is a uniform grid (floor keys, open-addressing table, cell-contiguous
// points) searched by expanding cubes: after the cube of Chebyshev radius R every unseen point is farther than
// (R + distance of the query to the nearest face of its own cell) cells, so the search stops — exactly — as soon as
// the current 5th distance is inside that bound; a finite gate stops it as soon as the bound passes the gate (the
// caller rejects the point either way), and a query that is still not settled after kMaxShell rings scans the whole
// map (far-away / tiny maps; exact by construction).  Ties in distance are broken by visit order (FLANN's order is
// unspecified too).
//
// The loop structure is the shared persistent one (gn_handover, fls_gn.cuh): one thread per feature point, corner
// points first then planar points (the order upstream sums them, :347-372), every class with its own persistent
// {J, residual} record and flag byte for the "flags reset once per Match" rule [quirk 1].
#include "fls_eig.cuh"
#include "fls_gn.cuh"
#include "fls_kernels.h"
#include "fls_plane.cuh"

namespace fls {
namespace {

constexpr int kMaxShell = 6;

__device__ __forceinline__ void scan_cell(const LoamGrid& g, int cx, int cy, int cz, float qx, float qy, float qz, Top5& nn, unsigned& n_cand) {
    unsigned start, count;
    if (!table_find(g.tab, g.mask, pack_key(cx, cy, cz), start, count)) return;
    n_cand += count;
#pragma unroll 2
    for (unsigned j = start; j < start + count; ++j) {
        const float4 p = __ldg(g.pts + j);
        nn.push(dist2_ref(p.x, p.y, p.z, qx, qy, qz), j);
    }
}

// kLoamLanes lanes share one query: lane `sub` visits every kLoamLanes-th cell, keeps a PRIVATE top-5 (the private lists
// of a group are disjoint), and the group's answer is their butterfly merge.
static constexpr int kLoamLanes = 8;
static_assert(kLoamPerBlock * kLoamLanes == kLoamBlock, "fls_kernels.h sizes the sub-grids by kLoamPerBlock");

__device__ __forceinline__ void merge_group(Top5& m, unsigned group_mask) {
#pragma unroll
    for (int o = kLoamLanes / 2; o > 0; o >>= 1) {
        const float e0 = __shfl_xor_sync(group_mask, m.d0, o), e1 = __shfl_xor_sync(group_mask, m.d1, o), e2 = __shfl_xor_sync(group_mask, m.d2, o),
                    e3 = __shfl_xor_sync(group_mask, m.d3, o), e4 = __shfl_xor_sync(group_mask, m.d4, o);
        const unsigned j0 = __shfl_xor_sync(group_mask, m.k0, o), j1 = __shfl_xor_sync(group_mask, m.k1, o), j2 = __shfl_xor_sync(group_mask, m.k2, o),
                       j3 = __shfl_xor_sync(group_mask, m.k3, o), j4 = __shfl_xor_sync(group_mask, m.k4, o);
        m.push(e0, j0);
        m.push(e1, j1);
        m.push(e2, j2);
        m.push(e3, j3);
        m.push(e4, j4);
    }
}

// exact 5-NN; `gate` = squared distance beyond which the caller rejects the point anyway (INFINITY: none).
// Called by all lanes of a group with the same query; every lane returns the group's merged result in `nn`.
__device__ __noinline__ void grid_knn5(const LoamGrid& g, int sub, unsigned group_mask, float qx, float qy, float qz, float gate, Top5& nn,
                                       unsigned& n_cand) {
    nn.init();
    n_cand = 0;
    if (g.n_pts < 5u) return;  // the tree cannot return 5 neighbours
    const float ux = __fmul_rn(qx, g.inv_cell), uy = __fmul_rn(qy, g.inv_cell), uz = __fmul_rn(qz, g.inv_cell);
    const float fx0 = floorf(ux), fy0 = floorf(uy), fz0 = floorf(uz);
    const int kx = (int)fx0, ky = (int)fy0, kz = (int)fz0;
    // distance (in cells) from the query to the nearest face of its own cell
    const float fx = ux - fx0, fy = uy - fy0, fz = uz - fz0;
    const float face = fminf(fminf(fminf(fx, 1.f - fx), fminf(fy, 1.f - fy)), fminf(fz, 1.f - fz));
    Top5 mine;
    mine.init();
#pragma unroll 1
    for (int s = sub; s < 27; s += kLoamLanes) scan_cell(g, kx + c_stencil[s][0], ky + c_stencil[s][1], kz + c_stencil[s][2], qx, qy, qz, mine, n_cand);
#pragma unroll 1
    for (int R = 1;; ++R) {
        nn = mine;
        merge_group(nn, group_mask);
        const float edge = ((float)R + face) * g.cell * 0.9995f;  // conservative: keys are floor(fl(p * inv_cell))
        const float b2 = edge * edge;
        if (nn.full() && nn.d4 <= b2) return;  // settled
        if (b2 > gate) return;                 // everything unseen lies beyond the gate
        if (R >= kMaxShell) break;
        const int S = R + 1;  // ring of Chebyshev radius S
        int cell = 0;
#pragma unroll 1
        for (int dz = -S; dz <= S; ++dz)
#pragma unroll 1
            for (int dy = -S; dy <= S; ++dy) {
                const bool face_row = (dz == -S || dz == S || dy == -S || dy == S);
#pragma unroll 1
                for (int dx = -S; dx <= S; dx += (face_row ? 1 : 2 * S), ++cell)
                    if ((cell & (kLoamLanes - 1)) == sub) scan_cell(g, kx + dx, ky + dy, kz + dz, qx, qy, qz, mine, n_cand);
            }
    }
    // exhaustive scan (far query or very sparse map)
    mine.init();
#pragma unroll 1
    for (unsigned j = (unsigned)sub; j < g.n_pts; j += kLoamLanes) {
        const float4 p = __ldg(g.pts + j);
        mine.push(dist2_ref(p.x, p.y, p.z, qx, qy, qz), j);
    }
    n_cand += g.n_pts / kLoamLanes;
    nn = mine;
    merge_group(nn, group_mask);
}

// LoamFull::CornerMatch per point (:219-270): line through the 5 neighbours by the principal axis of their covariance
__device__ __forceinline__ bool corner_term(const float4* __restrict__ P, const unsigned (&js)[5], const float4 sp, float qx, float qy, float qz,
                                            const double* __restrict__ pose, double line_ratio, double (&J)[6], double& res) {
    double X[5][3], c[3] = {0, 0, 0};
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const float4 a = __ldg(P + js[j]);
        X[j][0] = a.x; X[j][1] = a.y; X[j][2] = a.z;
        c[0] += X[j][0]; c[1] += X[j][1]; c[2] += X[j][2];
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) c[a] /= 5.0;  // rowwise().mean()  (:237)
    double S[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 5; ++j)
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) S[a * 3 + b] += (X[j][a] - c[a]) * (X[j][b] - c[b]);
#pragma unroll
    for (int k = 0; k < 9; ++k) S[k] /= 5.0;  // :239-242
    double lam[3], V[9];
    sym_eig3_dev(S, lam, V);
    if (lam[0] <= line_ratio * lam[1]) return false;  // :249
    const double nx = V[0], ny = V[3], nz = V[6];    // V.col(0); J does not depend on its sign
    const double vx = (double)qx - c[0], vy = (double)qy - c[1], vz = (double)qz - c[2];
    const double wx = vy * nz - vz * ny, wy = vz * nx - vx * nz, wz = vx * ny - vy * nx;  // (q - c) x n
    const double d = sqrt(wx * wx + wy * wy + wz * wz);                                   // :260
    const double ux = wx / d, uy = wy / d, uz = wz / d;
    // J.tail = (-n^)^T u = n x u ; J.head = (n^ (Rp)^)^T u = (Rp) x (n x u)   (:264-265)
    const double tx = ny * uz - nz * uy, ty = nz * ux - nx * uz, tz = nx * uy - ny * ux;
    const double px = sp.x, py = sp.y, pz = sp.z;
    const double rx = pose[0] * px + pose[1] * py + pose[2] * pz;
    const double ry = pose[3] * px + pose[4] * py + pose[5] * pz;
    const double rz = pose[6] * px + pose[7] * py + pose[8] * pz;
    J[0] = ry * tz - rz * ty;
    J[1] = rz * tx - rx * tz;
    J[2] = rx * ty - ry * tx;
    J[3] = tx;
    J[4] = ty;
    J[5] = tz;
    res = d;
    return true;
}

// (cta, ncta): position of this CTA in the (sub-)grid that serves the scan.  `a` by value: as a reference it costs the single-scan
// kernel 32 more bytes of stack frame (grid_knn5 takes the address of a map view).
template <int BLOCK>
__device__ __forceinline__ void loam_gn_loop(const LoamArgs a, const GnLoopCtl& ctl, const int cta, const int ncta) {
    __shared__ double s_pose[12];
    const int n_total = a.n_corner + a.n_planar;
    const int sub = threadIdx.x & (kLoamLanes - 1);
    const unsigned group_mask = ((1u << kLoamLanes) - 1u) << ((threadIdx.x & 31) & ~(kLoamLanes - 1));
    constexpr int kPerBlock = BLOCK / kLoamLanes;
    if (threadIdx.x < 12) s_pose[threadIdx.x] = threadIdx.x < 9 ? __ldcg(&a.state->R[threadIdx.x]) : __ldcg(&a.state->t[threadIdx.x - 9]);
    __syncthreads();
    for (int it = 0; it < ctl.gp.max_iterations; ++it) {  // the hand-over leaves the next pose in s_pose
        double acc[kNumAcc];
#pragma unroll
        for (int k = 0; k < kNumAcc; ++k) acc[k] = 0.0;
        for (int i = cta * kPerBlock + threadIdx.x / kLoamLanes; i < n_total; i += ncta * kPerBlock) {
            const bool is_corner = i < a.n_corner;
            const float4 sp = is_corner ? a.corner[i] : a.planar[i - a.n_corner];
            // pcl::transformPoint with the double transform, stored back as fp32 (:219-220, :284-285, kdtree :211-212)
            const float qx = xform_row_d(s_pose[0], s_pose[1], s_pose[2], s_pose[9], (double)sp.x, (double)sp.y, (double)sp.z);
            const float qy = xform_row_d(s_pose[3], s_pose[4], s_pose[5], s_pose[10], (double)sp.x, (double)sp.y, (double)sp.z);
            const float qz = xform_row_d(s_pose[6], s_pose[7], s_pose[8], s_pose[11], (double)sp.x, (double)sp.y, (double)sp.z);
            const LoamGrid& g = is_corner ? a.corner_map : a.planar_map;
            Top5 nn;
            unsigned n_cand;
            grid_knn5(g, sub, group_mask, qx, qy, qz, a.gate, nn, n_cand);
            acc[kAccCand] += (double)n_cand;
            double J[6], r = 0.0;
            bool use = false;
            if (sub == 0 && nn.full() && !((double)nn.d4 > a.search_thres)) {  // :227 / :291 (search_thres = +inf for the kd-tree point-to-plane plug-in)
                const unsigned js[5] = {nn.k0, nn.k1, nn.k2, nn.k3, nn.k4};
                unsigned fb = 0;
                use = is_corner ? corner_term(g.pts, js, sp, qx, qy, qz, s_pose, a.line_ratio, J, r)
                                : plane_term(g.pts, js, sp, qx, qy, qz, s_pose, a.plane_thres, J, r, fb);
            }
            if (sub != 0) continue;  // lane 0 of the group owns the point's record and sums
            double* rec = a.rec + (size_t)i * 8;
            if (use) {
#pragma unroll
                for (int k = 0; k < 6; ++k) rec[k] = J[k];
                rec[6] = r;
                a.flags[i] = 1;
            } else if (a.flags[i]) {  // stale contribution [quirk 1]
#pragma unroll
                for (int k = 0; k < 6; ++k) J[k] = rec[k];
                r = rec[6];
                use = true;
            }
            if (use) {
#pragma unroll
                for (int p = 0; p < 6; ++p)
#pragma unroll
                    for (int q = p; q < 6; ++q) acc[tri6(p, q)] += J[p] * J[q];
#pragma unroll
                for (int p = 0; p < 6; ++p) acc[21 + p] -= J[p] * r;
                acc[kAccRes] += r;
                if (is_corner) acc[kAccHits] += 1.0;  // number_valid_corner_ (reported, never gates)
                else acc[kAccValid] += 1.0;           // number_valid_planar_ (the < 50 failure test)
            }
        }
        if (gn_handover<BLOCK>(acc, ctl, it, s_pose, cta, ncta)) break;
    }
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) loam_gn_kernel(LoamArgs a, GnLoopCtl ctl) {
    loam_gn_loop<BLOCK>(a, ctl, (int)blockIdx.x, (int)gridDim.x);
}

// A batch of independent LoamPointToPlaneKdtree scans (planar only) against the same (static) map in ONE cooperative launch, a
// sub-grid and a loop per scan (as ndt_gn_batch_kernel); every scan owns its slice of the records and flags.
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) loam_gn_batch_kernel(const LoamBatchItem* __restrict__ items, int n_scans) {
    __shared__ LoamBatchItem s_item;
    gn_batch_item<BLOCK>(items, n_scans, s_item);
    loam_gn_loop<BLOCK>(s_item.a, s_item.ctl, (int)blockIdx.x - s_item.cta0, s_item.ncta);
}

__global__ void loam_clear_flags_kernel(unsigned char* flags, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flags[i] = 0;
}

}  // namespace

int loam_grid_blocks(int n, int device) {
    static int cap[64] = {0};
    if (device >= 0 && device < 64 && !cap[device]) {
        int sms = 0, per_sm = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, loam_gn_kernel<kLoamBlock>, kLoamBlock, 0);
        cap[device] = sms * (per_sm > 0 ? per_sm : 1);
    }
    const int need = (n + kLoamPerBlock - 1) / kLoamPerBlock;
    const int c = (device >= 0 && device < 64) ? cap[device] : 148;
    const int g = need < c ? need : c;
    return g > 0 ? g : 1;
}

void launch_loam_loop(const LoamArgs& a, const GnLoopCtl& ctl, int grid, cudaStream_t st) {
    LoamArgs a_ = a;
    GnLoopCtl c_ = ctl;
    const int n = a.n_corner + a.n_planar;
    if (n > 0) loam_clear_flags_kernel<<<(n + 255) / 256, 256, 0, st>>>(a.flags, n);
    void* params[] = {&a_, &c_};
    FLS_CUDA(cudaLaunchCooperativeKernel((const void*)loam_gn_kernel<kLoamBlock>, dim3(grid), dim3(kLoamBlock), params, 0, st));
}

int loam_max_grid(int device) {
    static int cap[64] = {0};
    if (device >= 0 && device < 64 && !cap[device]) {
        int sms = 0, per_sm = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, loam_gn_batch_kernel<kLoamBlock>, kLoamBlock, 0);
        cap[device] = sms * (per_sm > 0 ? per_sm : 1);
    }
    return (device >= 0 && device < 64) ? cap[device] : 148;
}

void launch_loam_batch(const LoamBatchItem* d_items, int n_scans, int grid, unsigned char* flags, int n_flags, cudaStream_t st) {
    if (n_flags > 0) loam_clear_flags_kernel<<<(n_flags + 255) / 256, 256, 0, st>>>(flags, n_flags);
    void* params[] = {&d_items, &n_scans};
    FLS_CUDA(cudaLaunchCooperativeKernel((const void*)loam_gn_batch_kernel<kLoamBlock>, dim3(grid), dim3(kLoamBlock), params, 0, st));
}

}  // namespace fls
