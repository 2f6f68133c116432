// fls_gn.cuh — Gauss-Newton plumbing shared by the residual kernels: the per-block reduction of the
// accumulators and the device-side solve / pose update / stop rule (K6).
//
// Conventions per plug-in (SURVEY.md §8a table; all line numbers upstream):
//   LOAM p2plane : dx=[dθ,dt], R <- Exp(dθ)·R, full-pivot solve, stop on thresholds OR |Δ‖dx‖|<1e-4,
//                  fail when n_valid < 50                      (loam_point_to_plane_ivox.h:167-203)
//   NDT          : dx=[dθ,dt], R <- R·Exp(dθ), H^-1·err, stop on thresholds, result forced true,
//                  early-out false when effective < min        (incremental_ndt.h:306-325)
//   ICP          : dx=[dt,dθ], R <- R·Exp(dθ), det==0 -> skip, converged only if thresholds met
//                                                              (icp_optimized.h:129-149)
#pragma once
#include "fls_common.cuh"

namespace fls {

struct GnParams {
    int method;  // fls_method: selects dx layout, update side, solver, stop rule
    int max_iterations;
    int min_effective;  // NDT: min_effective_pts; LOAM: 50 valid planar points
    double rot_thres, pos_thres;
};

// Control block of a persistent (one launch per Match) Gauss-Newton loop
struct GnLoopCtl {
    GnState* state;
    uint4* ll_rows;     // [gridDim.x][32] LL records: per-CTA partial sums
    uint4* ll_pose;     // [kLlPoseLen] LL records: next pose + stop word
    unsigned tag_base;  // Match epoch << 8
    GnParams gp;
    fls_iter_log* log;
    int log_cap;
    double* result;  // optional device buffer of kResultLen doubles, written when the loop stops (fls_set_result_buffer_device)
};
static constexpr int kResultLen = 18;  // column-major 4x4 pose, converged, iterations

// One scan of a batch launch (NDT, ICP, kd-tree point-to-plane): the grid is cut into one sub-grid per scan, scan s is served by
// CTAs [cta0, cta0 + ncta) running its own persistent loop with its own arguments and control block
template <class Args>
struct __align__(16) GnBatchItem {
    Args a;
    GnLoopCtl ctl;
    int cta0, ncta;
    int pad[2];
};

void launch_gn_init(GnState* d_state, const double* T_colmajor, cudaStream_t st);

#ifdef __CUDACC__
// ---- flag-in-data hand-over ("LL" records) ---------------------------------------------------------------------------
// A 16-byte record {lo32, tag, hi32, tag} carries one double together with the tag of the iteration that produced it.
// Each 8-byte half is a single-copy-atomic store, so a reader that sees the expected tag in BOTH halves has the value —
// no fence before the store, no separate flag, no atomic: the latency of a hand-over is one store plus one poll.
// tag = (Match epoch << 8) | (iteration + 1): never 0, unique across the iterations of consecutive Matches.
__device__ __forceinline__ void ll_store(uint4* p, double v, unsigned tag) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    const unsigned lo = (unsigned)b, hi = (unsigned)(b >> 32);
    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(lo), "r"(tag), "r"(hi), "r"(tag) : "memory");
}
__device__ __forceinline__ bool ll_load(const uint4* p, unsigned tag, double& v) {
    unsigned lo, t0, hi, t1;
    asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(t0), "=r"(hi), "=r"(t1) : "l"(p) : "memory");
    v = __longlong_as_double((long long)(((unsigned long long)hi << 32) | lo));
    return t0 == tag && t1 == tag;
}
static constexpr int kLlPoseLen = 16;  // R[9], t[3], done, pad

// Everything gn_step reads from the device state; a caller that has idle time before the totals are ready loads it early
// (one L2 round trip off the critical path).
struct GnPre {
    double R[9], t[3], last_rot, last_pos, cand0, hits0;
    int it;
};
__device__ __forceinline__ void gn_load(const GnState* s, GnPre& q) {
#pragma unroll
    for (int i = 0; i < 9; ++i) q.R[i] = __ldcg(&s->R[i]);
#pragma unroll
    for (int i = 0; i < 3; ++i) q.t[i] = __ldcg(&s->t[i]);
    q.last_rot = __ldcg(&s->last_rot);
    q.last_pos = __ldcg(&s->last_pos);
    q.cand0 = __ldcg(&s->cand_total);
    q.hits0 = __ldcg(&s->hits_total);
    q.it = __ldcg(&s->iter);
}

// One Gauss-Newton step from the reduced totals `tot[kNumAcc]`: fills H/g, solves, updates the pose in `s`,
// applies the plug-in's stop rule.  Executed by a single thread: the arithmetic runs on locals, what the other CTAs wait
// for (pose + stop word, as LL records) goes out first and the bookkeeping follows.
__device__ inline void gn_step_pre(GnState* s, const GnPre& q, const double* tot, const GnParams& p, fls_iter_log* log, int log_cap,
                                   uint4* ll_pose, unsigned ll_tag, double* result = nullptr) {
    double R[9], t[3];
#pragma unroll
    for (int i = 0; i < 9; ++i) R[i] = q.R[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) t[i] = q.t[i];
    const double last_rot = q.last_rot, last_pos = q.last_pos;
    const double cand0 = q.cand0, hits0 = q.hits0;
    const int it = q.it;

    double H[36], g[6], dx[6] = {0, 0, 0, 0, 0, 0};
    for (int r = 0; r < 6; ++r)
        for (int c = r; c < 6; ++c) H[r * 6 + c] = H[c * 6 + r] = tot[tri6(r, c)];
    for (int a = 0; a < 6; ++a) g[a] = tot[21 + a];
    const long long n_valid = (long long)(tot[kAccValid] + 0.5);
    const double sum_res = tot[kAccRes];

    bool stop = false;
    int converged = -1, failed = 0;
    double new_last_rot = last_rot, new_last_pos = last_pos;
    if (p.method == FLS_NDT && n_valid < (long long)p.min_effective) {
        failed = 1;  // incremental_ndt.h:306-309 — T = pose, return false
        converged = 0;
        stop = true;
    } else {
        double Rd[9], Rn[9];
        // H = sum J^T (W) J is symmetric positive definite whenever the problem is well posed: register-resident LDL^T
        // first, the pivoting solver that mirrors the reference's rank behaviour only when that is not safely the case.
        double det_spd = 0.0;
        const bool spd = solve6_spd(H, g, dx, &det_spd);
        if (p.method == FLS_ICP_P2P) {
            const double det = spd ? det_spd : solve6_lu(H, g, dx);
            if (det == 0.0) {
                for (int i = 0; i < 6; ++i) dx[i] = 0;  // icp_optimized.h:129-131 `continue`
            } else {
                for (int a = 0; a < 3; ++a) t[a] += dx[a];
                so3_exp(dx + 3, Rd);
                mat3_mul(R, Rd, Rn);
                for (int i = 0; i < 9; ++i) R[i] = Rn[i];
                if (norm3(dx + 3) < p.rot_thres && norm3(dx) < p.pos_thres) {
                    converged = 1;
                    stop = true;
                }
            }
        } else if (p.method == FLS_NDT) {
            if (!spd) solve6_lu(H, g, dx);
            so3_exp(dx, Rd);
            mat3_mul(R, Rd, Rn);
            for (int i = 0; i < 9; ++i) R[i] = Rn[i];
            for (int a = 0; a < 3; ++a) t[a] += dx[3 + a];
            if (norm3(dx) < p.rot_thres && norm3(dx + 3) < p.pos_thres) stop = true;
            converged = 1;  // forced true after the loop (incremental_ndt.h:325)
        } else {
            if (!spd) solve6_fullpiv(H, g, dx);
            so3_exp(dx, Rd);
            mat3_mul(Rd, R, Rn);
            for (int i = 0; i < 9; ++i) R[i] = Rn[i];
            for (int a = 0; a < 3; ++a) t[a] += dx[3 + a];
            const double rn = norm3(dx), pn = norm3(dx + 3);
            const double drot = fabs(rn - last_rot), dpos = fabs(pn - last_pos);
            new_last_rot = rn;
            new_last_pos = pn;
            if ((rn < p.rot_thres && pn < p.pos_thres) || (drot < 1.0e-4 && dpos < 1.0e-4)) stop = true;
            converged = (n_valid >= (long long)p.min_effective) ? 1 : 0;  // :201-203
        }
        if (it + 1 >= p.max_iterations) stop = true;
    }
    // ---- publish: what the other CTAs wait for goes out first
    if (ll_pose) {
#pragma unroll
        for (int i = 0; i < 9; ++i) ll_store(ll_pose + i, R[i], ll_tag);
#pragma unroll
        for (int i = 0; i < 3; ++i) ll_store(ll_pose + 9 + i, t[i], ll_tag);
        ll_store(ll_pose + 12, stop ? 1.0 : 0.0, ll_tag);
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) s->R[i] = R[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) s->t[i] = t[i];
    if (stop) s->done = 1;
    if (stop && result) {  // packed result for a device-side consumer (the multi-GPU pose all-gather): Eigen Mat4d memory + flags
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            result[c * 4 + 0] = R[c];
            result[c * 4 + 1] = R[3 + c];
            result[c * 4 + 2] = R[6 + c];
            result[c * 4 + 3] = 0.0;
        }
        result[12] = t[0]; result[13] = t[1]; result[14] = t[2]; result[15] = 1.0;
        result[16] = converged > 0 ? 1.0 : 0.0;
        result[17] = (double)(it + 1);
    }
    // pose before the update (LOAM-iVox map insertion rule)
#pragma unroll
    for (int i = 0; i < 9; ++i) s->Rprev[i] = q.R[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) s->tprev[i] = q.t[i];
    s->last_rot = new_last_rot;
    s->last_pos = new_last_pos;
    for (int i = 0; i < 36; ++i) s->H[i] = H[i];
    for (int i = 0; i < 6; ++i) {
        s->g[i] = g[i];
        s->dx[i] = dx[i];
    }
    s->n_valid = n_valid;
    s->sum_res = sum_res;
    s->cand_total = cand0 + tot[kAccCand];
    s->hits_total = hits0 + tot[kAccHits];
    s->iter = it + 1;
    if (converged >= 0) s->converged = converged;
    if (failed) s->failed = 1;
    if (log && it < log_cap) {
        fls_iter_log& L = log[it];
        for (int i = 0; i < 36; ++i) L.H[i] = H[i];
        for (int i = 0; i < 6; ++i) {
            L.g[i] = g[i];
            L.dx[i] = dx[i];
        }
        L.sum_residual = sum_res;
        L.n_valid = n_valid;
    }
}

// Tail of one iteration of a persistent GN loop (all threads of all CTAs call it with their per-thread sums):
// block reduction -> CTA row published as LL records (no fence, no atomic) -> CTA 0 sweeps the rows until every tag matches,
// folds them in a fixed order, runs gn_step and publishes the next pose + stop word as LL records -> everybody polls that
// record.  Needs co-resident CTAs (cooperative launch).  On return s_pose[0..11] (shared memory, row-major R then t) holds
// the pose of the next iteration; returns true when the loop is finished.
template <int BLOCK>
__device__ __forceinline__ bool gn_handover(double (&acc)[kNumAcc], const GnLoopCtl& c, int it, double* s_pose, int cta = -1, int ncta = -1) {
    // (cta, ncta): position of this CTA in the sub-grid that serves the scan (batch launches); default: the whole grid
    if (cta < 0) {
        cta = (int)blockIdx.x;
        ncta = (int)gridDim.x;
    }
    constexpr int W = BLOCK / 32;
    __shared__ double s_red[W][kAccStride];
    __shared__ int s_stop;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned tag = c.tag_base | (unsigned)(it + 1);
#pragma unroll
    for (int k = 0; k < kNumAcc; ++k) {
        double v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) s_red[warp][k] = v;
    }
    if (lane == 0) s_red[warp][kNumAcc] = 0.0;
    __syncthreads();
    if (warp == 0) {
        double v = 0;
#pragma unroll
        for (int w = 0; w < W; ++w) v += s_red[w][lane];
        ll_store(c.ll_rows + (size_t)cta * 32 + lane, v, tag);
    }
    if (cta == 0) {
        GnPre pre;
        if (threadIdx.x == 0) gn_load(c.state, pre);
        __syncthreads();  // s_red is free again
        const int nrows = ncta;
        double sum;
        for (;;) {
            bool ok = true;
            double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
            int r = warp;
            for (; r + 7 * W < nrows; r += 8 * W) {  // 8 independent 16-byte loads in flight per lane
                double v0, v1, v2, v3, v4, v5, v6, v7;
                const bool k0 = ll_load(c.ll_rows + (size_t)r * 32 + lane, tag, v0);
                const bool k1 = ll_load(c.ll_rows + (size_t)(r + W) * 32 + lane, tag, v1);
                const bool k2 = ll_load(c.ll_rows + (size_t)(r + 2 * W) * 32 + lane, tag, v2);
                const bool k3 = ll_load(c.ll_rows + (size_t)(r + 3 * W) * 32 + lane, tag, v3);
                const bool k4 = ll_load(c.ll_rows + (size_t)(r + 4 * W) * 32 + lane, tag, v4);
                const bool k5 = ll_load(c.ll_rows + (size_t)(r + 5 * W) * 32 + lane, tag, v5);
                const bool k6 = ll_load(c.ll_rows + (size_t)(r + 6 * W) * 32 + lane, tag, v6);
                const bool k7 = ll_load(c.ll_rows + (size_t)(r + 7 * W) * 32 + lane, tag, v7);
                ok = ok && k0 && k1 && k2 && k3 && k4 && k5 && k6 && k7;
                a0 += v0; a1 += v1; a2 += v2; a3 += v3;
                a0 += v4; a1 += v5; a2 += v6; a3 += v7;
            }
            for (; r + 3 * W < nrows; r += 4 * W) {
                double v0, v1, v2, v3;
                const bool k0 = ll_load(c.ll_rows + (size_t)r * 32 + lane, tag, v0);
                const bool k1 = ll_load(c.ll_rows + (size_t)(r + W) * 32 + lane, tag, v1);
                const bool k2 = ll_load(c.ll_rows + (size_t)(r + 2 * W) * 32 + lane, tag, v2);
                const bool k3 = ll_load(c.ll_rows + (size_t)(r + 3 * W) * 32 + lane, tag, v3);
                ok = ok && k0 && k1 && k2 && k3;
                a0 += v0; a1 += v1; a2 += v2; a3 += v3;
            }
            for (; r < nrows; r += W) {
                double v0;
                ok = ok && ll_load(c.ll_rows + (size_t)r * 32 + lane, tag, v0);
                a0 += v0;
            }
            sum = (a0 + a1) + (a2 + a3);
            if (__all_sync(0xffffffffu, ok)) break;
            __nanosleep(100);
        }
        s_red[warp][lane] = sum;
        __syncthreads();
        if (warp == 0) {
            double t = 0;
#pragma unroll
            for (int w = 0; w < W; ++w) t += s_red[w][lane];
            __syncwarp();
            s_red[0][lane] = t;
            __syncwarp();
            if (lane == 0) gn_step_pre(c.state, pre, s_red[0], c.gp, c.log, c.log_cap, c.ll_pose, tag, c.result);
        }
    }
    if (threadIdx.x < 13) {
        double v;
        while (!ll_load(c.ll_pose + threadIdx.x, tag, v)) __nanosleep(100);
        if (threadIdx.x < 12) s_pose[threadIdx.x] = v;
        else s_stop = v != 0.0;
    }
    __syncthreads();
    return s_stop != 0;
}

// Prologue of a batch kernel: finds the item whose sub-grid holds this CTA and copies it into shared memory (`s_item`), so the
// loop reads its arguments like kernel parameters.
template <int BLOCK, class Args>
__device__ __forceinline__ void gn_batch_item(const GnBatchItem<Args>* __restrict__ items, int n_scans, GnBatchItem<Args>& s_item) {
    static_assert(sizeof(GnBatchItem<Args>) % 8 == 0, "copied in 8-byte words");
    __shared__ int s_which;
    if (threadIdx.x == 0) {
        int w = 0;
        while (w + 1 < n_scans && (int)blockIdx.x >= items[w + 1].cta0) ++w;
        s_which = w;
    }
    __syncthreads();
    {
        const unsigned long long* src = reinterpret_cast<const unsigned long long*>(items + s_which);
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(&s_item);
        for (int k = threadIdx.x; k < (int)(sizeof(GnBatchItem<Args>) / 8); k += BLOCK) dst[k] = src[k];
    }
    __syncthreads();
}
#endif

}  // namespace fls
