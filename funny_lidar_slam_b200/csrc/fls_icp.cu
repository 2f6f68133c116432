// fls_icp.cu — K3: bounded exact 1-NN point-to-point residual + reduction (IcpOptimized), and the
// GetFitnessScore kernel shared by every plug-in.
//
// IcpOptimized::Match (include/registration/icp_optimized.h:54-163 upstream) asks a kd-tree for the exact
// nearest map point and then rejects it when d^2 > max_correspond_distance [quirk 4: squared distance against
// an unsquared threshold].  A correspondence can therefore only survive inside radius sqrt(threshold), so a
// uniform grid with cell >= that radius searched over its 27-cell neighbourhood returns the identical
// correspondence for every accepted point and "nothing" exactly where upstream rejects.
#include "fls_gn.cuh"
#include "fls_kernels.h"

namespace fls {
namespace {

// nearest map point within the 27-cell neighbourhood; returns false when the neighbourhood is empty
__device__ __forceinline__ bool grid_nn1(const IvoxView& g, float qx, float qy, float qz, float& best_d, unsigned& best_j, unsigned& n_cand,
                                         unsigned& n_hits) {
    best_d = INFINITY;
    best_j = 0xffffffffu;
    n_cand = 0;
    n_hits = 0;
    const float ux = __fmul_rn(qx, g.inv_res), uy = __fmul_rn(qy, g.inv_res), uz = __fmul_rn(qz, g.inv_res);
    const int kx = (int)floorf(ux), ky = (int)floorf(uy), kz = (int)floorf(uz);
    const float cell = 1.0f / g.inv_res;
#pragma unroll 1
    for (int s = 0; s < 27; ++s) {
        const int cx = kx + c_stencil[s][0], cy = ky + c_stencil[s][1], cz = kz + c_stencil[s][2];
        // lower bound of the distance from q to the cell box, in metres (conservative by 0.1 %)
        const float ax = fmaxf(0.f, fmaxf((float)cx - ux, ux - (float)(cx + 1)));
        const float ay = fmaxf(0.f, fmaxf((float)cy - uy, uy - (float)(cy + 1)));
        const float az = fmaxf(0.f, fmaxf((float)cz - uz, uz - (float)(cz + 1)));
        const float lb = (ax * ax + ay * ay + az * az) * cell * cell * 0.998f;
        if (lb > best_d) continue;
        unsigned start, count;
        if (!table_find(g.tab, g.mask, pack_key(cx, cy, cz), start, count)) continue;
        n_cand += count;
        n_hits += 1;
#pragma unroll 1
        for (unsigned j = start; j < start + count; ++j) {
            const float4 p = __ldg(g.pts + j);
            const float d = dist2_ref(p.x, p.y, p.z, qx, qy, qz);
            if (d < best_d) {
                best_d = d;
                best_j = j;
            }
        }
    }
    return best_j != 0xffffffffu;
}

// Sub-warp version for the Gauss-Newton loop: kIcpLanes lanes share one query, lane `sub` visits stencil cells
// sub, sub+kIcpLanes, ...; the winner is the lexicographic minimum of (d2, stencil position, point index) — the same
// point the sequential scan above keeps (strict '<' in visit order).  All lanes of the group return the result.
static constexpr int kIcpLanes = 8;
static_assert(kIcpPerBlock * kIcpLanes == kIcpBlock, "fls_kernels.h sizes the sub-grids by kIcpPerBlock");
__device__ __forceinline__ bool grid_nn1_coop(const IvoxView& g, int sub, unsigned group_mask, float qx, float qy, float qz, float& best_d,
                                              unsigned& best_j, unsigned& n_cand, unsigned& n_hits) {
    best_d = INFINITY;
    best_j = 0xffffffffu;
    unsigned best_s = 0xffffu;
    n_cand = 0;
    n_hits = 0;
    const float ux = __fmul_rn(qx, g.inv_res), uy = __fmul_rn(qy, g.inv_res), uz = __fmul_rn(qz, g.inv_res);
    const int kx = (int)floorf(ux), ky = (int)floorf(uy), kz = (int)floorf(uz);
#pragma unroll 1
    for (int s = sub; s < 27; s += kIcpLanes) {
        const int cx = kx + c_stencil[s][0], cy = ky + c_stencil[s][1], cz = kz + c_stencil[s][2];
        unsigned start, count;
        if (!table_find(g.tab, g.mask, pack_key(cx, cy, cz), start, count)) continue;
        n_cand += count;
        n_hits += 1;
#pragma unroll 2
        for (unsigned j = start; j < start + count; ++j) {
            const float4 p = __ldg(g.pts + j);
            const float d = dist2_ref(p.x, p.y, p.z, qx, qy, qz);
            if (d < best_d) {
                best_d = d;
                best_j = j;
                best_s = (unsigned)s;
            }
        }
    }
#pragma unroll
    for (int o = kIcpLanes / 2; o > 0; o >>= 1) {
        const float od = __shfl_xor_sync(group_mask, best_d, o);
        const unsigned oj = __shfl_xor_sync(group_mask, best_j, o);
        const unsigned os = __shfl_xor_sync(group_mask, best_s, o);
        const bool take = (od < best_d) || (od == best_d && (os < best_s || (os == best_s && oj < best_j)));
        if (take) {
            best_d = od;
            best_j = oj;
            best_s = os;
        }
    }
    return best_j != 0xffffffffu;
}

// One persistent launch runs every Gauss-Newton iteration of a Match (gn_handover, fls_gn.cuh).  (cta, ncta): position of this
// CTA in the (sub-)grid that serves the scan.
template <int BLOCK>
__device__ __forceinline__ void icp_gn_loop(const IcpArgs& a, const GnLoopCtl& ctl, const int cta, const int ncta) {
    __shared__ double s_pose[12];
    __shared__ float s_posef[12];
    const int sub = threadIdx.x & (kIcpLanes - 1);
    const unsigned group_mask = ((1u << kIcpLanes) - 1u) << ((threadIdx.x & 31) & ~(kIcpLanes - 1));
    constexpr int kPerBlock = BLOCK / kIcpLanes;
    if (threadIdx.x < 12) s_pose[threadIdx.x] = threadIdx.x < 9 ? __ldcg(&a.state->R[threadIdx.x]) : __ldcg(&a.state->t[threadIdx.x - 9]);
    __syncthreads();
    for (int it = 0; it < ctl.gp.max_iterations; ++it) {  // the hand-over leaves the next pose in s_pose
        if (threadIdx.x < 12) s_posef[threadIdx.x] = (float)s_pose[threadIdx.x];  // R.cast<float>(), t.cast<float>()  (pointcloud_utility.h:145-146)
        __syncthreads();
        double acc[kNumAcc];
#pragma unroll
        for (int k = 0; k < kNumAcc; ++k) acc[k] = 0.0;

        for (int i = cta * kPerBlock + threadIdx.x / kIcpLanes; i < a.n; i += ncta * kPerBlock) {
            const float4 sp = a.src[i];
            const float qx = xform_row_f(s_posef[0], s_posef[1], s_posef[2], s_posef[9], sp.x, sp.y, sp.z);
            const float qy = xform_row_f(s_posef[3], s_posef[4], s_posef[5], s_posef[10], sp.x, sp.y, sp.z);
            const float qz = xform_row_f(s_posef[6], s_posef[7], s_posef[8], s_posef[11], sp.x, sp.y, sp.z);
            float d2;
            unsigned j, nc, nh;
            const bool found = grid_nn1_coop(a.map, sub, group_mask, qx, qy, qz, d2, j, nc, nh);
            acc[kAccCand] += (double)nc;
            acc[kAccHits] += (double)nh;
            if (sub == 0 && found && !((double)d2 > a.max_corr)) {  // icp_optimized.h:87
                const float4 m = __ldg(a.map.pts + j);
                const double e0 = (double)qx - (double)m.x, e1 = (double)qy - (double)m.y, e2 = (double)qz - (double)m.z;
                const double px = sp.x, py = sp.y, pz = sp.z;
                const double* R = s_pose;
                double A[3][3];  // -R * hat(p)   (:100)
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const double r0 = R[r * 3 + 0], r1 = R[r * 3 + 1], r2 = R[r * 3 + 2];
                    A[r][0] = -(r1 * pz - r2 * py);
                    A[r][1] = -(r2 * px - r0 * pz);
                    A[r][2] = -(r0 * py - r1 * px);
                }
                // dx = [dt(0..2), dθ(3..5)]:  H = [[I, A],[A^T, A^T A]],  b = -[e ; A^T e]
                acc[tri6(0, 0)] += 1.0; acc[tri6(1, 1)] += 1.0; acc[tri6(2, 2)] += 1.0;
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int c = 0; c < 3; ++c) acc[tri6(r, 3 + c)] += A[r][c];
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int c = r; c < 3; ++c) acc[tri6(3 + r, 3 + c)] += A[0][r] * A[0][c] + A[1][r] * A[1][c] + A[2][r] * A[2][c];
                acc[21] -= e0; acc[22] -= e1; acc[23] -= e2;
#pragma unroll
                for (int r = 0; r < 3; ++r) acc[24 + r] -= (A[0][r] * e0 + A[1][r] * e1 + A[2][r] * e2);
                acc[kAccValid] += 1.0;
                acc[kAccRes] += sqrt(e0 * e0 + e1 * e1 + e2 * e2);  // total_res += error.norm()  (:126)
            }
        }
        if (gn_handover<BLOCK>(acc, ctl, it, s_pose, cta, ncta)) break;
    }
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) icp_gn_kernel(IcpArgs a, GnLoopCtl ctl) {
    icp_gn_loop<BLOCK>(a, ctl, (int)blockIdx.x, (int)gridDim.x);
}

// A batch of independent scans against the same (static) map in ONE cooperative launch, a sub-grid and a loop per scan (as
// ndt_gn_batch_kernel): the hand-over of one scan overlaps with the residual passes of the others.
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) icp_gn_batch_kernel(const IcpBatchItem* __restrict__ items, int n_scans) {
    __shared__ IcpBatchItem s_item;
    gn_batch_item<BLOCK>(items, n_scans, s_item);
    icp_gn_loop<BLOCK>(s_item.a, s_item.ctl, (int)blockIdx.x - s_item.cta0, s_item.ncta);
}

// GetFitnessScore (icp_optimized.h:191-215 upstream): mean squared 1-NN distance over points with d2 <= max_range
__global__ void fitness_kernel(IvoxView g, const float4* __restrict__ src, int n, float r0, float r1, float r2, float r3, float r4, float r5,
                               float r6, float r7, float r8, float t0, float t1, float t2, float max_range, double* __restrict__ out /*sum, count*/) {
    __shared__ double s_sum[8], s_cnt[8];
    double sum = 0, cnt = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 sp = src[i];
        const float qx = xform_row_f(r0, r1, r2, t0, sp.x, sp.y, sp.z);
        const float qy = xform_row_f(r3, r4, r5, t1, sp.x, sp.y, sp.z);
        const float qz = xform_row_f(r6, r7, r8, t2, sp.x, sp.y, sp.z);
        float d2;
        unsigned j, nc, nh;
        if (grid_nn1(g, qx, qy, qz, d2, j, nc, nh) && d2 <= max_range) {
            sum += (double)d2;
            cnt += 1.0;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        s_sum[warp] = sum;
        s_cnt[warp] = cnt;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, b = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
            a += s_sum[w];
            b += s_cnt[w];
        }
        atomicAdd(out, a);
        atomicAdd(out + 1, b);
    }
}

}  // namespace

int icp_grid_blocks(int n, int device) {
    static int cap[64] = {0};
    if (device >= 0 && device < 64 && !cap[device]) {
        int sms = 0, per_sm = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, icp_gn_kernel<kIcpBlock>, kIcpBlock, 0);
        cap[device] = sms * (per_sm > 0 ? per_sm : 1);
    }
    const int need = (n + kIcpPerBlock - 1) / kIcpPerBlock;
    const int c = (device >= 0 && device < 64) ? cap[device] : 148;
    const int g = need < c ? need : c;
    return g > 0 ? g : 1;
}
void launch_icp_loop(const IcpArgs& a, const GnLoopCtl& ctl, int grid, cudaStream_t st) {
    IcpArgs a_ = a;
    GnLoopCtl c_ = ctl;
    void* params[] = {&a_, &c_};
    FLS_CUDA(cudaLaunchCooperativeKernel((const void*)icp_gn_kernel<kIcpBlock>, dim3(grid), dim3(kIcpBlock), params, 0, st));
}

int icp_max_grid(int device) {
    static int cap[64] = {0};
    if (device >= 0 && device < 64 && !cap[device]) {
        int sms = 0, per_sm = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, icp_gn_batch_kernel<kIcpBlock>, kIcpBlock, 0);
        cap[device] = sms * (per_sm > 0 ? per_sm : 1);
    }
    return (device >= 0 && device < 64) ? cap[device] : 148;
}
void launch_icp_batch(const IcpBatchItem* d_items, int n_scans, int grid, cudaStream_t st) {
    void* params[] = {&d_items, &n_scans};
    FLS_CUDA(cudaLaunchCooperativeKernel((const void*)icp_gn_batch_kernel<kIcpBlock>, dim3(grid), dim3(kIcpBlock), params, 0, st));
}

void launch_fitness(const IvoxView& g, const float4* d_src, int n, const double* T, float max_range, double* d_out2, cudaStream_t st) {
    cudaMemsetAsync(d_out2, 0, 2 * sizeof(double), st);
    if (n <= 0) return;
    int grid = (n + 255) / 256;
    if (grid > 592) grid = 592;
    fitness_kernel<<<grid, 256, 0, st>>>(g, d_src, n, (float)T[0], (float)T[4], (float)T[8], (float)T[1], (float)T[5], (float)T[9], (float)T[2],
                                         (float)T[6], (float)T[10], (float)T[12], (float)T[13], (float)T[14], max_range, d_out2);
}

}  // namespace fls
