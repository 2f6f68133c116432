// fls_ndt.cu — K2 (NDT residual + reduction) and K8-NDT (voxel map build / incremental update).
//
// IncrementalNDT (include/registration/incremental_ndt.h upstream) keeps an unordered_map of list nodes holding
// {points_, mu_, sigma_, information_, ndt_estimated_, num_points_}.  Here:
//   * table  : open-addressing slots {packed key (C-truncation of q/voxel, [quirk 5]), voxel index, estimated flag}
//   * hot    : 80-byte records {mu, symmetric information} — the only thing the Match kernel reads
//   * cold   : sigma, counters and a carry buffer of <= min_points_in_voxel pending points per voxel, touched only
//              by AddCloudToLocalMap / UpdateVoxel (:130-227)
// LRU eviction at `capacity` (:203-206) is emulated exactly: stamps per voxel + a host simulation of the sequential insert
// (NdtMap::evict_lru, lru_simulate in fls_map.cu).
#include <cub/cub.cuh>

#include "fls_gn.cuh"
#include "fls_eig.cuh"
#include "fls_kernels.h"
#include "fls_maps.h"

namespace fls {
namespace {

inline unsigned grid_for(size_t n, int block) { return (unsigned)((n + block - 1) / block); }

__device__ __forceinline__ int ndt_coord(double v, double inv) { return (int)__dmul_rn(v, inv); }  // cast<int>() truncates

__global__ void ndt_keys_kernel(const float4* __restrict__ pts, size_t n, double inv, unsigned long long* __restrict__ keys,
                                unsigned* __restrict__ idx) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pts[i];
    keys[i] = pack_key(ndt_coord((double)p.x, inv), ndt_coord((double)p.y, inv), ndt_coord((double)p.z, inv));
    idx[i] = (unsigned)i;
}

__global__ void ndt_table_clear_kernel(HashSlot* tab, size_t slots, int* counter) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i < slots) {
        tab[i].key = kEmptyKey;
        tab[i].start = 0xffffffffu;
        tab[i].count = 0;
    }
    if (i == 0) *counter = 0;
}

__device__ __forceinline__ void inv3_sym_reg(const double* S, double* Ai) {
    // cofactor inverse of a general 3x3 (Eigen's fixed-size inverse, incremental_ndt.h:134,151 upstream)
    const double c00 = S[4] * S[8] - S[5] * S[7], c01 = S[5] * S[6] - S[3] * S[8], c02 = S[3] * S[7] - S[4] * S[6];
    const double det = S[0] * c00 + S[1] * c01 + S[2] * c02;
    const double id = 1.0 / det;
    Ai[0] = c00 * id; Ai[1] = (S[2] * S[7] - S[1] * S[8]) * id; Ai[2] = (S[1] * S[5] - S[2] * S[4]) * id;
    Ai[3] = c01 * id; Ai[4] = (S[0] * S[8] - S[2] * S[6]) * id; Ai[5] = (S[2] * S[3] - S[0] * S[5]) * id;
    Ai[6] = c02 * id; Ai[7] = (S[1] * S[6] - S[0] * S[7]) * id; Ai[8] = (S[0] * S[4] - S[1] * S[3]) * id;
}

struct NdtUpdateArgs {
    const float4* __restrict__ pts;          // filtered cloud, map frame
    const unsigned* __restrict__ idx_sorted;  // point indices grouped by voxel (stable => cloud order inside a voxel)
    const unsigned long long* __restrict__ run_keys;
    const unsigned* __restrict__ starts;
    const unsigned* __restrict__ counts;
    int runs;
    HashSlot* tab;
    unsigned mask;
    NdtHot* hot;
    NdtCold* cold;
    double* carry;
    int* counter;  // [0] high-water mark of voxel indices, [1] overflow flag, [2] free-list cursor
    const int* free_list;
    int n_free;
    unsigned long long call_hi;  // call number << 32
    long long capacity;
    int min_pts, max_pts;
    int first_scan;
};

// sequential mean / covariance over the carried points followed by the run's points (incremental_ndt.h:92-110)
__device__ void mean_cov_seq(const double* carry, int nc, const float4* __restrict__ pts, const unsigned* __restrict__ idx, unsigned s, unsigned c,
                             double* mean, double* cov) {
    const int n = nc + (int)c;
    double sm[3] = {0, 0, 0};
    for (int k = 0; k < nc; ++k)
        for (int a = 0; a < 3; ++a) sm[a] += carry[k * 3 + a];
    for (unsigned k = 0; k < c; ++k) {
        const float4 p = __ldg(pts + idx[s + k]);
        sm[0] += (double)p.x;
        sm[1] += (double)p.y;
        sm[2] += (double)p.z;
    }
    for (int a = 0; a < 3; ++a) mean[a] = sm[a] / (double)n;
    double cc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int k = 0; k < nc; ++k) {
        const double v[3] = {carry[k * 3] - mean[0], carry[k * 3 + 1] - mean[1], carry[k * 3 + 2] - mean[2]};
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) cc[a * 3 + b] += v[a] * v[b];
    }
    for (unsigned k = 0; k < c; ++k) {
        const float4 p = __ldg(pts + idx[s + k]);
        const double v[3] = {(double)p.x - mean[0], (double)p.y - mean[1], (double)p.z - mean[2]};
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) cc[a * 3 + b] += v[a] * v[b];
    }
    for (int a = 0; a < 9; ++a) cov[a] = cc[a] / (double)(n - 1);
}

__device__ __forceinline__ void store_hot(NdtHot* h, const double* mu, const double* info) {
    h->mu[0] = mu[0]; h->mu[1] = mu[1]; h->mu[2] = mu[2];
    h->info[0] = info[0];
    h->info[1] = 0.5 * (info[1] + info[3]);
    h->info[2] = 0.5 * (info[2] + info[6]);
    h->info[3] = info[4];
    h->info[4] = 0.5 * (info[5] + info[7]);
    h->info[5] = info[8];
    h->pad = 0.0;
}

// one thread per touched voxel: find-or-create, then UpdateVoxel (incremental_ndt.h:130-179 upstream)
__global__ void ndt_update_kernel(NdtUpdateArgs a, int* overflow) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.runs) return;
    const unsigned long long key = a.run_keys[r];
    const unsigned s = a.starts[r], c = a.counts[r];
    // find or insert
    unsigned h = hash_key(key) & a.mask;
    unsigned vi;
    bool created = false;
    for (;;) {
        const unsigned long long prev = atomicCAS(&a.tab[h].key, kEmptyKey, key);
        if (prev == kEmptyKey) {
            // indices of evicted voxels first (the LRU tail was evicted before this kernel: NdtMap::evict_lru), then fresh ones
            int id;
            const int k = atomicAdd(a.counter + 2, 1);
            if (k < a.n_free) id = a.free_list[a.n_free - 1 - k];  // the list is a stack
            else id = atomicAdd(a.counter, 1);
            if ((long long)id >= a.capacity) atomicExch(overflow, 1);  // cannot happen once the eviction ran
            vi = (unsigned)id;
            a.tab[h].start = vi;
            created = true;
            break;
        }
        if (prev == key) {
            vi = a.tab[h].start;
            break;
        }
        h = (h + 1) & a.mask;
    }
    if ((long long)vi >= a.capacity) return;
    NdtCold& cd = a.cold[vi];
    double* carry = a.carry + (size_t)vi * a.min_pts * 3;
    if (created) {
        cd.num_points = 0;
        cd.carry_count = 0;
        cd.estimated = 0;
        cd.alive = 1;
        cd.key = key;
        for (int k = 0; k < 9; ++k) cd.sigma[k] = 0;
    }
    cd.stamp = a.call_hi | (unsigned long long)a.idx_sorted[s + c - 1];  // moved to the front by its last point of this call (:208-210)
    if (!cd.estimated) cd.num_points += (int)c;  // VoxelData ctor / AddPoint (:66-76): counted only before the first estimate

    double mu[3], info[9];
    if (a.first_scan) {  // :131-143 — every touched voxel is (re-)estimated from the points of this call only
        if (c > 1u) {
            mean_cov_seq(carry, 0, a.pts, a.idx_sorted, s, c, mu, cd.sigma);
            double S[9];
            for (int k = 0; k < 9; ++k) S[k] = cd.sigma[k] + ((k % 4 == 0) ? 1.0e-3 : 0.0);
            inv3_sym_reg(S, info);
        } else {
            const float4 p = a.pts[a.idx_sorted[s]];
            mu[0] = (double)p.x; mu[1] = (double)p.y; mu[2] = (double)p.z;
            for (int k = 0; k < 9; ++k) info[k] = (k % 4 == 0) ? 1.0e2 : 0.0;
        }
        cd.estimated = 1;
        cd.carry_count = 0;
        store_hot(a.hot + vi, mu, info);
        a.tab[h].count = 1;
        return;
    }
    if (cd.estimated && cd.num_points > a.max_pts) return;  // :145-147 frozen
    const int nc = cd.carry_count;
    const int total = nc + (int)c;
    if (total > a.min_pts) {
        if (!cd.estimated) {  // :149-153
            mean_cov_seq(carry, nc, a.pts, a.idx_sorted, s, c, mu, cd.sigma);
            double S[9];
            for (int k = 0; k < 9; ++k) S[k] = cd.sigma[k] + ((k % 4 == 0) ? 1.0e-3 : 0.0);
            inv3_sym_reg(S, info);
            cd.estimated = 1;
        } else {  // :154-178 running merge + eigen clamp
            double cm[3], cv[9], nm[3], nv[9], om[3];
            mean_cov_seq(carry, nc, a.pts, a.idx_sorted, s, c, cm, cv);
            const NdtHot& oh = a.hot[vi];
            om[0] = oh.mu[0]; om[1] = oh.mu[1]; om[2] = oh.mu[2];
            const double m = (double)cd.num_points, n = (double)total;
            for (int k = 0; k < 3; ++k) nm[k] = (m * om[k] + n * cm[k]) / (m + n);
            for (int x = 0; x < 3; ++x)
                for (int y = 0; y < 3; ++y)
                    nv[x * 3 + y] = (m * (cd.sigma[x * 3 + y] + (om[x] - nm[x]) * (om[y] - nm[y])) + n * (cv[x * 3 + y] + (cm[x] - nm[x]) * (cm[y] - nm[y]))) / (m + n);
            for (int k = 0; k < 3; ++k) mu[k] = nm[k];
            for (int k = 0; k < 9; ++k) cd.sigma[k] = nv[k];
            cd.num_points += total;
            double lam[3], V[9];
            sym_eig3_dev(cd.sigma, lam, V);
            if (lam[1] < lam[0] * 1e-3) lam[1] = lam[0] * 1e-3;
            if (lam[2] < lam[0] * 1e-3) lam[2] = lam[0] * 1e-3;
            for (int x = 0; x < 3; ++x)
                for (int y = 0; y < 3; ++y)
                    info[x * 3 + y] = V[x * 3 + 0] * V[y * 3 + 0] / lam[0] + V[x * 3 + 1] * V[y * 3 + 1] / lam[1] + V[x * 3 + 2] * V[y * 3 + 2] / lam[2];
        }
        cd.carry_count = 0;
        store_hot(a.hot + vi, mu, info);
        a.tab[h].count = 1;
    } else {  // keep the points for a later estimate
        for (unsigned k = 0; k < c; ++k) {
            const float4 p = a.pts[a.idx_sorted[s + k]];
            carry[(nc + k) * 3 + 0] = (double)p.x;
            carry[(nc + k) * 3 + 1] = (double)p.y;
            carry[(nc + k) * 3 + 2] = (double)p.z;
        }
        cd.carry_count = total;
    }
}

// ---- LRU bookkeeping (incremental_ndt.h:193-214) -------------------------------------------------------------------------------
// which touched voxels exist already; counters[3] = to be created, counters[4] = existing and touched
__global__ void ndt_lookup_kernel(int runs, const unsigned long long* __restrict__ run_keys, const HashSlot* __restrict__ tab, unsigned mask,
                                  int* __restrict__ run_vi, int* __restrict__ touch_run, int* counters) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= runs) return;
    unsigned vi, est;
    if (table_find(tab, mask, run_keys[r], vi, est)) {
        run_vi[r] = (int)vi;
        touch_run[vi] = r;
        atomicAdd(counters + 4, 1);
    } else {
        run_vi[r] = -1;
        atomicAdd(counters + 3, 1);
    }
}
__global__ void ndt_live_kernel(const NdtCold* __restrict__ cold, int hi_water, unsigned long long* __restrict__ stamps, unsigned* __restrict__ vis,
                                int* counters) {
    const int vi = blockIdx.x * blockDim.x + threadIdx.x;
    if (vi >= hi_water || !cold[vi].alive) return;
    const int pos = atomicAdd(counters + 5, 1);
    stamps[pos] = cold[vi].stamp;
    vis[pos] = (unsigned)vi;
}
// first point of this call that touches candidate k (0xffffffff: none)
__global__ void ndt_cand_kernel(const unsigned* __restrict__ vis_sorted, int K, const int* __restrict__ touch_run, const unsigned* __restrict__ starts,
                                const unsigned* __restrict__ idx_sorted, unsigned* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const int r = touch_run[vis_sorted[k]];
    out[k] = r >= 0 ? idx_sorted[starts[r]] : 0xffffffffu;
}
__global__ void ndt_create_times_kernel(int runs, const int* __restrict__ run_vi, const unsigned* __restrict__ starts,
                                        const unsigned* __restrict__ idx_sorted, unsigned* __restrict__ out, int* cursor) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= runs || run_vi[r] >= 0) return;
    out[atomicAdd(cursor, 1)] = idx_sorted[starts[r]];
}
__global__ void ndt_evict_kernel(const unsigned* __restrict__ victim_pos, const unsigned char* __restrict__ recreated, int n,
                                 const unsigned* __restrict__ vis_sorted, NdtCold* __restrict__ cold, int* __restrict__ free_list, int free_base,
                                 const int* __restrict__ touch_run, int* __restrict__ run_vi) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned vi = vis_sorted[victim_pos[i]];
    cold[vi].alive = 0;
    free_list[free_base + i] = (int)vi;
    if (recreated[i]) run_vi[touch_run[vi]] = -1;  // touched again later in the call: created anew, empty (:197-201)
}
__global__ void ndt_table_rebuild_kernel(const NdtCold* __restrict__ cold, int hi_water, HashSlot* tab, unsigned mask) {
    const int vi = blockIdx.x * blockDim.x + threadIdx.x;
    if (vi >= hi_water || !cold[vi].alive) return;
    const unsigned long long key = cold[vi].key;
    unsigned h = hash_key(key) & mask;
    for (;;) {
        const unsigned long long prev = atomicCAS(&tab[h].key, kEmptyKey, key);
        if (prev == kEmptyKey) {
            tab[h].start = (unsigned)vi;
            tab[h].count = cold[vi].estimated ? 1u : 0u;
            return;
        }
        h = (h + 1) & mask;
    }
}
__global__ void ndt_table_clear_only_kernel(HashSlot* tab, size_t slots) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i < slots) {
        tab[i].key = kEmptyKey;
        tab[i].start = 0xffffffffu;
        tab[i].count = 0;
    }
}
__global__ void ndt_dump_keys_kernel(const NdtCold* __restrict__ cold, int hi_water, unsigned long long* __restrict__ out, int* cursor) {
    const int vi = blockIdx.x * blockDim.x + threadIdx.x;
    if (vi >= hi_water || !cold[vi].alive) return;
    out[atomicAdd(cursor, 1)] = cold[vi].key;
}

// ---- K2: NDT residual kernel -----------------------------------------------------------------------------------
// One persistent launch runs every Gauss-Newton iteration of a Match (gn_handover, fls_gn.cuh): grid-stride over the
// points, per-thread sums, CTA row, last-CTA fold + solve + release.
template <int BLOCK>
__device__ __forceinline__ void ndt_gn_loop(const NdtArgs& a, const GnLoopCtl& ctl, const int cta, const int ncta) {
    __shared__ double s_pose[12];
    if (threadIdx.x < 9) s_pose[threadIdx.x] = __ldcg(&a.state->R[threadIdx.x]);
    else if (threadIdx.x < 12) s_pose[threadIdx.x] = __ldcg(&a.state->t[threadIdx.x - 9]);
    __syncthreads();
    for (int it = 0; it < ctl.gp.max_iterations; ++it) {  // the hand-over leaves the next pose in s_pose
    double acc[kNumAcc];
#pragma unroll
    for (int k = 0; k < kNumAcc; ++k) acc[k] = 0.0;

    for (int i = cta * BLOCK + threadIdx.x; i < a.n; i += ncta * BLOCK) {
        const float4 sp = a.src[i];
        const double px = sp.x, py = sp.y, pz = sp.z;
        const double* R = s_pose;
        const double qx = xform_row_dd(R[0], R[1], R[2], s_pose[9], px, py, pz);  // incremental_ndt.h:255
        const double qy = xform_row_dd(R[3], R[4], R[5], s_pose[10], px, py, pz);
        const double qz = xform_row_dd(R[6], R[7], R[8], s_pose[11], px, py, pz);
        const int kx = ndt_coord(qx, a.map.inv_voxel), ky = ndt_coord(qy, a.map.inv_voxel), kz = ndt_coord(qz, a.map.inv_voxel);  // :256
        double L0 = 0, L1 = 0, L2 = 0, L3 = 0, L4 = 0, L5 = 0;  // sum of information matrices (sym)
        double w0 = 0, w1 = 0, w2 = 0, chis = 0;
        int cnt = 0, hits = 0;
#pragma unroll 1
        for (int s = 0; s < 7; ++s) {  // stencil order of :122-127 = first 7 entries of c_stencil
            const unsigned long long key = pack_key(kx + c_stencil[s][0], ky + c_stencil[s][1], kz + c_stencil[s][2]);
            unsigned vi, est;
            if (!table_find(a.map.tab, a.map.mask, key, vi, est)) continue;
            ++hits;
            if (!est) continue;  // voxel exists but ndt_estimated_ is false (:263)
            const double2* hp = reinterpret_cast<const double2*>(a.map.hot + vi);
            const double2 h0 = __ldg(hp), h1 = __ldg(hp + 1), h2 = __ldg(hp + 2), h3 = __ldg(hp + 3), h4 = __ldg(hp + 4);
            const double ex = qx - h0.x, ey = qy - h0.y, ez = qz - h1.x;
            const double ixx = h1.y, ixy = h2.x, ixz = h2.y, iyy = h3.x, iyz = h3.y, izz = h4.x;
            const double ux = ixx * ex + ixy * ey + ixz * ez;
            const double uy = ixy * ex + iyy * ey + iyz * ez;
            const double uz = ixz * ex + iyz * ey + izz * ez;
            const double chi = ex * ux + ey * uy + ez * uz;
            if (isnan(chi) || chi > a.outlier_thres) continue;  // :267-271
            L0 += ixx; L1 += ixy; L2 += ixz; L3 += iyy; L4 += iyz; L5 += izz;
            w0 += ux; w1 += uy; w2 += uz;
            chis += chi;
            ++cnt;
        }
        acc[kAccHits] += (double)hits;
        acc[kAccCand] += (double)cnt;
        if (cnt > 0) {
            // B = -R * hat(p)  (3x3), J = [B | I]  (:273-275);  H = [[B^T L B, B^T L],[L B, L]],  err = -[B^T w ; w]
            double B[3][3];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const double r0 = R[r * 3 + 0], r1 = R[r * 3 + 1], r2 = R[r * 3 + 2];
                B[r][0] = -(r1 * pz - r2 * py);
                B[r][1] = -(r2 * px - r0 * pz);
                B[r][2] = -(r0 * py - r1 * px);
            }
            double LB[3][3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                LB[0][c] = L0 * B[0][c] + L1 * B[1][c] + L2 * B[2][c];
                LB[1][c] = L1 * B[0][c] + L3 * B[1][c] + L4 * B[2][c];
                LB[2][c] = L2 * B[0][c] + L4 * B[1][c] + L5 * B[2][c];
            }
            // upper triangle in dx = [dθ(0..2), dt(3..5)] order
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int c = r; c < 3; ++c) acc[tri6(r, c)] += B[0][r] * LB[0][c] + B[1][r] * LB[1][c] + B[2][r] * LB[2][c];
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[tri6(r, 3 + c)] += LB[c][r];  // (B^T L)[r][c] = (L B)[c][r], L symmetric
            acc[tri6(3, 3)] += L0; acc[tri6(3, 4)] += L1; acc[tri6(3, 5)] += L2;
            acc[tri6(4, 4)] += L3; acc[tri6(4, 5)] += L4; acc[tri6(5, 5)] += L5;
#pragma unroll
            for (int r = 0; r < 3; ++r) acc[21 + r] -= (B[0][r] * w0 + B[1][r] * w1 + B[2][r] * w2);
            acc[24] -= w0; acc[25] -= w1; acc[26] -= w2;
            acc[kAccValid] += (double)cnt;
            acc[kAccRes] += chis;
        }
    }
    if (gn_handover<BLOCK>(acc, ctl, it, s_pose, cta, ncta)) break;
    }
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) ndt_gn_kernel(NdtArgs a, GnLoopCtl ctl) {
    ndt_gn_loop<BLOCK>(a, ctl, (int)blockIdx.x, (int)gridDim.x);
}

// A batch of independent scans against the same (static) map in ONE cooperative launch: the grid is cut into one sub-grid
// per scan, each running its own persistent Gauss-Newton loop (own rows, pose record and state) — the ~15 us hand-over of a
// scan overlaps with the residual passes of the others, which is what the single-scan loop cannot hide at these sizes.
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) ndt_gn_batch_kernel(const NdtBatchItem* __restrict__ items, int n_scans) {
    __shared__ NdtBatchItem s_item;
    gn_batch_item<BLOCK>(items, n_scans, s_item);
    ndt_gn_loop<BLOCK>(s_item.a, s_item.ctl, (int)blockIdx.x - s_item.cta0, s_item.ncta);
}

}  // namespace

int ndt_grid(int n, int device) {
    static int cap[64] = {0};
    if (device >= 0 && device < 64 && !cap[device]) {
        int sms = 0, per_sm = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ndt_gn_kernel<kNdtBlock>, kNdtBlock, 0);
        cap[device] = sms * (per_sm > 0 ? per_sm : 1);
    }
    const int need = (n + kNdtBlock - 1) / kNdtBlock;
    const int c = (device >= 0 && device < 64) ? cap[device] : 148;
    const int g = need < c ? need : c;
    return g > 0 ? g : 1;
}
void launch_ndt_loop(const NdtArgs& a, const GnLoopCtl& ctl, int grid, cudaStream_t st) {
    NdtArgs a_ = a;
    GnLoopCtl c_ = ctl;
    void* params[] = {&a_, &c_};
    FLS_CUDA(cudaLaunchCooperativeKernel((const void*)ndt_gn_kernel<kNdtBlock>, dim3(grid), dim3(kNdtBlock), params, 0, st));
}

int ndt_max_grid(int device) {
    ndt_grid(1, device);  // fills the cache
    static int cap[64] = {0};
    if (device >= 0 && device < 64 && !cap[device]) {
        int sms = 0, per_sm = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ndt_gn_batch_kernel<kNdtBlock>, kNdtBlock, 0);
        cap[device] = sms * (per_sm > 0 ? per_sm : 1);
    }
    return (device >= 0 && device < 64) ? cap[device] : 148;
}
void launch_ndt_batch(const NdtBatchItem* d_items, int n_scans, int grid, cudaStream_t st) {
    void* params[] = {&d_items, &n_scans};
    FLS_CUDA(cudaLaunchCooperativeKernel((const void*)ndt_gn_batch_kernel<kNdtBlock>, dim3(grid), dim3(kNdtBlock), params, 0, st));
}

void NdtMap::configure(double voxel_size, int min_points, int max_points, long long cap) {
    voxel = voxel_size;
    inv_voxel = 1.0 / voxel_size;
    min_pts = min_points;
    max_pts = max_points;
    capacity = cap;
}

int NdtMap::add_cloud(const float4* d_cloud, size_t n, float leaf, bool first_scan, cudaStream_t st) {
    if (n == 0) return FLS_OK;
    filtered.reserve(n);
    int l = 0;
    const size_t nf = voxel_grid_device(d_cloud, n, leaf, filtered.p, scratch, st, &l);  // :186
    launches += l;
    if (nf == 0) return FLS_OK;
    if (slots == 0) {  // first use: size everything by the configured capacity
        size_t want = 1024;
        while (want < 2 * (size_t)capacity) want <<= 1;
        slots = want;
        mask = (unsigned)(slots - 1);
        table.reserve(slots);
        hot.reserve((size_t)capacity);
        cold.reserve((size_t)capacity);
        carry.reserve((size_t)capacity * (size_t)(min_pts > 0 ? min_pts : 1) * 3);
        counter.reserve(8);
        ndt_table_clear_kernel<<<grid_for(slots, 256), 256, 0, st>>>(table.p, slots, counter.p);
        launches++;
    }
    BuildScratch& sc = scratch;
    sc.keys.reserve(nf);
    sc.keys_sorted.reserve(nf);
    sc.uniq.reserve(nf);
    sc.idx.reserve(nf);
    sc.idx_sorted.reserve(nf);
    sc.counts.reserve(nf);
    sc.starts.reserve(nf);
    sc.num_runs.reserve(2);
    ndt_keys_kernel<<<grid_for(nf, 256), 256, 0, st>>>(filtered.p, nf, inv_voxel, sc.keys.p, sc.idx.p);
    size_t t1 = 0, t2 = 0, t3 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, sc.keys.p, sc.keys_sorted.p, sc.idx.p, sc.idx_sorted.p, (int)nf, 0, 63, st);
    cub::DeviceRunLengthEncode::Encode(nullptr, t2, sc.keys_sorted.p, sc.uniq.p, sc.counts.p, sc.num_runs.p, (int)nf, st);
    cub::DeviceScan::ExclusiveSum(nullptr, t3, sc.counts.p, sc.starts.p, (int)nf, st);
    size_t tmp = t1 > t2 ? t1 : t2;
    tmp = tmp > t3 ? tmp : t3;
    sc.cub_tmp.reserve(tmp + 256);
    size_t tb = sc.cub_tmp.cap;
    FLS_CUDA(cub::DeviceRadixSort::SortPairs(sc.cub_tmp.p, tb, sc.keys.p, sc.keys_sorted.p, sc.idx.p, sc.idx_sorted.p, (int)nf, 0, 63, st));
    tb = sc.cub_tmp.cap;
    FLS_CUDA(cub::DeviceRunLengthEncode::Encode(sc.cub_tmp.p, tb, sc.keys_sorted.p, sc.uniq.p, sc.counts.p, sc.num_runs.p, (int)nf, st));
    FLS_CUDA(cudaMemcpyAsync(sc.h_num_runs, sc.num_runs.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    FLS_CUDA(cudaStreamSynchronize(st));
    const int runs = *sc.h_num_runs;
    tb = sc.cub_tmp.cap;
    FLS_CUDA(cub::DeviceScan::ExclusiveSum(sc.cub_tmp.p, tb, sc.counts.p, sc.starts.p, runs, st));
    // ---- LRU bookkeeping: which touched voxels exist, how many are created, who has to go first --------------------------------
    const int hi_water0 = hi_water;
    run_vi.reserve((size_t)runs + 1);
    touch_run.reserve((size_t)capacity + 1);
    free_list.reserve((size_t)capacity + 1);
    FLS_CUDA(cudaMemsetAsync(counter.p + 1, 0, 7 * sizeof(int), st));
    if (hi_water0 > 0) FLS_CUDA(cudaMemsetAsync(touch_run.p, 0xff, sizeof(int) * (size_t)hi_water0, st));
    ndt_lookup_kernel<<<grid_for(runs, 256), 256, 0, st>>>(runs, sc.uniq.p, table.p, mask, run_vi.p, touch_run.p, counter.p);
    int hc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    FLS_CUDA(cudaMemcpyAsync(hc, counter.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, st));
    FLS_CUDA(cudaStreamSynchronize(st));
    launches += 1;
    const int n_new = hc[3], n_touched = hc[4];
    ++call_no;
    int n_victims = 0, n_recreated = 0;
    // upstream: after every creation `if (data_.size() >= capacity_) pop_back()` (:203-206) — the list never holds `capacity` voxels
    if ((long long)n_vox + n_new >= capacity) {
        const int rc = evict_lru(runs, n_new, n_touched, st, &n_victims, &n_recreated);
        if (rc != FLS_OK) return rc;
    }
    NdtUpdateArgs ua;
    ua.pts = filtered.p;
    ua.idx_sorted = sc.idx_sorted.p;
    ua.run_keys = sc.uniq.p;
    ua.starts = sc.starts.p;
    ua.counts = sc.counts.p;
    ua.runs = runs;
    ua.tab = table.p;
    ua.mask = mask;
    ua.hot = hot.p;
    ua.cold = cold.p;
    ua.carry = carry.p;
    ua.counter = counter.p;
    ua.free_list = free_list.p;
    ua.n_free = n_free;
    ua.call_hi = call_no << 32;
    ua.capacity = capacity;
    ua.min_pts = min_pts;
    ua.max_pts = max_pts;
    ua.first_scan = first_scan ? 1 : 0;
    int* overflow = counter.p + 1;
    FLS_CUDA(cudaMemsetAsync(counter.p + 1, 0, 2 * sizeof(int), st));  // overflow flag, free-list cursor
    ndt_update_kernel<<<grid_for(runs, 128), 128, 0, st>>>(ua, overflow);
    int h[3] = {0, 0, 0};
    FLS_CUDA(cudaMemcpyAsync(h, counter.p, 3 * sizeof(int), cudaMemcpyDeviceToHost, st));
    FLS_CUDA(cudaStreamSynchronize(st));
    launches += 6;
    hi_water = h[0];
    n_free -= h[2] < n_free ? h[2] : n_free;  // the creations popped that many indices off the free stack
    n_vox = n_vox + (size_t)n_new + (size_t)n_recreated - (size_t)n_victims;
    if (h[1]) return FLS_ERR_CAPACITY;
    return FLS_OK;
}

// Evicts what upstream's sequential insert would evict during this call (exact, including a victim that is touched again later in
// the call): candidates = live voxels by ascending stamp, simulated on the host against the creation times of the new voxels.
int NdtMap::evict_lru(int runs, int n_new, int n_touched, cudaStream_t st, int* n_victims, int* n_recreated) {
    BuildScratch& sc = scratch;
    const int hw = hi_water;
    const size_t n_live = n_vox;
    if (n_live == 0) return FLS_ERR_CAPACITY;  // the first cloud alone overflows the capacity: upstream dereferences an erased voxel (:216-220)
    lru_keys.reserve(n_live + 1);
    lru_keys_sorted.reserve(n_live + 1);
    lru_vals.reserve(n_live + 1);
    lru_vals_sorted.reserve(n_live + 1);
    ndt_live_kernel<<<grid_for(hw, 256), 256, 0, st>>>(cold.p, hw, lru_keys.p, lru_vals.p, counter.p);
    size_t tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, lru_keys.p, lru_keys_sorted.p, lru_vals.p, lru_vals_sorted.p, (int)n_live, 0, 64, st);
    sc.cub_tmp.reserve(tb + 256);
    tb = sc.cub_tmp.cap;
    FLS_CUDA(cub::DeviceRadixSort::SortPairs(sc.cub_tmp.p, tb, lru_keys.p, lru_keys_sorted.p, lru_vals.p, lru_vals_sorted.p, (int)n_live, 0, 64, st));
    // the eviction count without cascades is n_vox + n_new - (capacity - 1); every skipped candidate was touched in this call
    const long long e0 = (long long)n_live + n_new - (capacity - 1);
    size_t K = (size_t)(e0 > 0 ? e0 : 0) + 2 * (size_t)n_touched + 64;
    if (K > n_live) K = n_live;
    sc.k32a.reserve(K + 1);
    sc.k32b.reserve((size_t)n_new + 1);
    ndt_cand_kernel<<<grid_for(K, 256), 256, 0, st>>>(lru_vals_sorted.p, (int)K, touch_run.p, sc.starts.p, sc.idx_sorted.p, sc.k32a.p);
    FLS_CUDA(cudaMemsetAsync(counter.p + 6, 0, sizeof(int), st));
    ndt_create_times_kernel<<<grid_for(runs, 256), 256, 0, st>>>(runs, run_vi.p, sc.starts.p, sc.idx_sorted.p, sc.k32b.p, counter.p + 6);
    std::vector<unsigned> cand(K), creat((size_t)n_new);
    FLS_CUDA(cudaMemcpyAsync(cand.data(), sc.k32a.p, sizeof(unsigned) * K, cudaMemcpyDeviceToHost, st));
    if (n_new) FLS_CUDA(cudaMemcpyAsync(creat.data(), sc.k32b.p, sizeof(unsigned) * (size_t)n_new, cudaMemcpyDeviceToHost, st));
    FLS_CUDA(cudaStreamSynchronize(st));
    launches += 5;
    std::vector<unsigned> victims;
    std::vector<unsigned char> recreated;
    if (!lru_simulate(n_live, (size_t)capacity, cand, creat, victims, recreated)) return FLS_ERR_CAPACITY;
    *n_victims = (int)victims.size();
    *n_recreated = 0;
    for (unsigned char r : recreated) *n_recreated += r ? 1 : 0;
    if (victims.empty()) return FLS_OK;
    // victims -> free list, their keys out of the table (rebuild: open addressing has no cheap delete)
    sc.k32a.reserve(victims.size() + 1);
    sc.minmax.reserve(victims.size() / 4 + 16);
    FLS_CUDA(cudaMemcpyAsync(sc.k32a.p, victims.data(), sizeof(unsigned) * victims.size(), cudaMemcpyHostToDevice, st));
    FLS_CUDA(cudaMemcpyAsync(sc.minmax.p, recreated.data(), victims.size(), cudaMemcpyHostToDevice, st));
    ndt_evict_kernel<<<grid_for(victims.size(), 128), 128, 0, st>>>(sc.k32a.p, reinterpret_cast<const unsigned char*>(sc.minmax.p), (int)victims.size(),
                                                                   lru_vals_sorted.p, cold.p, free_list.p, n_free, touch_run.p, run_vi.p);
    n_free += (int)victims.size();
    ndt_table_clear_only_kernel<<<grid_for(slots, 256), 256, 0, st>>>(table.p, slots);
    ndt_table_rebuild_kernel<<<grid_for(hw, 256), 256, 0, st>>>(cold.p, hw, table.p, mask);
    FLS_CUDA(cudaStreamSynchronize(st));  // the host vectors above are read by the copies
    launches += 3;
    return FLS_OK;
}

size_t NdtMap::dump_keys(unsigned long long* h_out, size_t cap, cudaStream_t st) {
    if (n_vox == 0 || hi_water == 0) return 0;
    lru_keys.reserve(n_vox + 1);
    FLS_CUDA(cudaMemsetAsync(counter.p + 7, 0, sizeof(int), st));
    ndt_dump_keys_kernel<<<grid_for(hi_water, 256), 256, 0, st>>>(cold.p, hi_water, lru_keys.p, counter.p + 7);
    int n = 0;
    FLS_CUDA(cudaMemcpyAsync(&n, counter.p + 7, sizeof(int), cudaMemcpyDeviceToHost, st));
    FLS_CUDA(cudaStreamSynchronize(st));
    const size_t m = (size_t)n < cap ? (size_t)n : cap;
    FLS_CUDA(cudaMemcpy(h_out, lru_keys.p, sizeof(unsigned long long) * m, cudaMemcpyDeviceToHost));
    return m;
}

}  // namespace fls
