// fls_api.cu — the C ABI of include/fls_b200.h: handle lifetime, host<->device staging and the host side of
// each plug-in's Match / AddCloudToLocalMap / GetFitnessScore.  The Gauss-Newton loop itself runs on the
// device (one persistent kernel per Match or per batch: residuals, 6x6 reduction, solve, pose update and stop rule);
// the host reads the ~1.8 KB state block of every scan back once.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "fls_gn.cuh"
#include "fls_handle.h"

namespace fls {

static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }
const char* last_error_cstr() { return g_last_error.c_str(); }

Handle::Handle(const fls_config& c) : cfg(c) {
    try {
        init();
    } catch (...) {  // a throwing constructor does not run the destructor: give back what was acquired so far
        release();
        throw;
    }
}

void Handle::release() {
    if (h_state) cudaFreeHost(h_state);
    if (h_batch) cudaFreeHost(h_batch);
    h_state = nullptr;
    h_batch = nullptr;
    for (auto& e : prof_ev)
        if (e) cudaEventDestroy(e);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    ev0 = ev1 = nullptr;
    if (stream) cudaStreamDestroy(stream);
    stream = nullptr;
}

void Handle::init() {
    FLS_CUDA(cudaSetDevice(cfg.device));
    FLS_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    FLS_CUDA(cudaEventCreate(&ev0));
    FLS_CUDA(cudaEventCreate(&ev1));
    FLS_CUDA(cudaMallocHost(&h_state, sizeof(GnState) * kMaxBatch + 64));
    h_abort = reinterpret_cast<unsigned*>(h_state + kMaxBatch);  // pinned: a copy into pageable memory would make the enqueue wait for the kernel
    *h_abort = 0;
    state.reserve(kMaxBatch);
    fit_out.reserve(2);
    ivox.set_resolution(cfg.ivox_resolution);
    ivox.key_mode = 0;
    ivox.incremental = cfg.method == FLS_P2PLANE_IVOX && !cfg.localization_mode;  // mapping mode: the map grows by small inserts
    {
        static const int counts[4] = {1, 7, 19, 27};
        ivox.n_stencil = counts[cfg.ivox_nearby];
    }
    ndt.configure(cfg.ndt_voxel_size, cfg.ndt_min_points_in_voxel, cfg.ndt_max_points_in_voxel, cfg.ndt_capacity);
    // search grid of the bounded exact 1-NN: cell >= sqrt(max_correspond_distance)  [quirk 4]
    icp_map.grid.key_mode = 1;
    icp_map.grid.set_resolution((float)(std::sqrt(cfg.icp_max_correspond_distance > 0 ? cfg.icp_max_correspond_distance : 1.0) * 1.001));
    fit_grid.key_mode = 1;
    // exact-search grids of the kd-tree plug-ins: LoamFull only needs neighbours inside sqrt(point_search_thres), so a cell
    // of that size settles every query in the 27-cell pass; the ungated point-to-plane variant uses ~2 map leafs
    kd_planar.grid.key_mode = kd_corner.grid.key_mode = 1;
    if (cfg.method == FLS_LOAM_FULL) {
        const float c = (float)(std::sqrt(cfg.point_search_thres > 0 ? cfg.point_search_thres : 1.0) * 1.001);
        kd_planar.grid.set_resolution(c);
        kd_corner.grid.set_resolution(c);
    } else {
        const float c = 2.0f * (cfg.map_cloud_filter_size > 0.f ? cfg.map_cloud_filter_size : 0.5f);
        kd_planar.grid.set_resolution(c < 0.8f ? 0.8f : c);
        kd_corner.grid.set_resolution(1.0f);
    }
    profile = (cfg.flags & FLS_FLAG_PROFILE) != 0;
    if (profile)
        for (auto& e : prof_ev) FLS_CUDA(cudaEventCreate(&e));
    if (cfg.flags & FLS_FLAG_ITER_LOG) {
        log_cap = cfg.max_iterations > 0 ? cfg.max_iterations : 1;
        log.reserve((size_t)log_cap * kMaxBatch);
        h_log.resize(log_cap);
    }
}

Handle::~Handle() {
    cudaSetDevice(cfg.device);
    if (stream) cudaStreamSynchronize(stream);
    release();
}

// Copy a caller cloud (host memory, `stride` bytes per record) into a packed float4 device buffer.
const float4* Handle::upload(const void* pts, size_t n, size_t stride, DevBuf<float4>& dst) {
    dst.reserve(n);
    if (n == 0) return dst.p;
    if (stride == FLS_LAYOUT_PACKED) {
        FLS_CUDA(cudaMemcpyAsync(dst.p, pts, n * 16, cudaMemcpyHostToDevice, stream));
        h2d_bytes += (long long)(n * 16);
    } else {
        raw.reserve(n * stride);
        FLS_CUDA(cudaMemcpyAsync(raw.p, pts, n * stride, cudaMemcpyHostToDevice, stream));
        h2d_bytes += (long long)(n * stride);
        launch_repack(raw.p, n, stride, dst.p, stream);
        launches++;
    }
    return dst.p;
}

IvoxView Handle::grid_view(const IvoxMap& g) const {
    IvoxView v;
    v.pts = g.pts_sorted.p;
    v.tab = g.table.p;
    v.mask = g.mask;
    v.inv_res = g.inv_res;
    v.max_range2 = cfg.ivox_max_range * cfg.ivox_max_range;
    static const int counts[4] = {1, 7, 19, 27};
    v.n_stencil = counts[cfg.ivox_nearby];
    v.lists = g.lists.p;
    v.ctab = g.ctab.p;
    v.cmask = g.cmask;
    // a query and a candidate of its stencil differ by at most 2*res per axis with a non-zero offset and res otherwise:
    // d^2 <= 12 res^2 for the full 26-neighbourhood
    {
        const char* e = std::getenv("FLS_LIST_PREFETCH");
        v.prefetch = e ? (unsigned)std::atoi(e) : 1u;
    }
    v.fast_knn = (12.0 * 1.01 * (double)g.res * (double)g.res < (double)v.max_range2 && !std::getenv("FLS_EXACT_KNN")) ? 1u : 0u;
    return v;
}
IvoxView Handle::ivox_view() const { return grid_view(ivox); }

void Handle::begin_call() {
    FLS_CUDA(cudaSetDevice(cfg.device));
    launches = 0;
    h2d_bytes = d2h_bytes = 0;
    FLS_CUDA(cudaEventRecord(ev0, stream));
}

void Handle::end_call(fls_match_stats* st) {
    FLS_CUDA(cudaEventRecord(ev1, stream));
    FLS_CUDA(cudaStreamSynchronize(stream));
    float ms = 0;
    FLS_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
    last_gpu_ms = ms;
    if (st) {
        st->gpu_ms = ms;
        st->gpu_launches = launches;
        st->h2d_bytes = h2d_bytes;
        st->d2h_bytes = d2h_bytes;
    }
}

void Handle::set_fit_cloud(const float4* d, size_t n) {
    fit_cloud.reserve(n);
    if (n) FLS_CUDA(cudaMemcpyAsync(fit_cloud.p, d, n * sizeof(float4), cudaMemcpyDeviceToDevice, stream));
    set_fit_view(fit_cloud.p, n);
}

void Handle::set_fit_view(const float4* d, size_t n) {
    fit_src = d;
    fit_n = n;
    fit_version++;
}

// ---- host side of a persistent GN launch (K1 / K2 / K3 / K5) ---------------------------------------------------------
unsigned Handle::next_epoch(size_t ll_records) {
    // LL hand-over records (fls_gn.cuh): never cleared, tags are unique per Match and iteration; zeroed only when (re)allocated,
    // so that uninitialised memory cannot alias a tag
    const size_t cap0 = ll_rows.cap;
    ll_rows.reserve(ll_records);
    if (ll_rows.cap != cap0) FLS_CUDA(cudaMemsetAsync(ll_rows.p, 0, ll_rows.cap * sizeof(uint4), stream));
    match_epoch = (match_epoch + 1) & 0xffffffu;
    if (match_epoch == 0) match_epoch = 1;
    return match_epoch << 8;
}

GnParams Handle::gn_params(int method, int min_effective) const {
    GnParams gp;
    gp.method = method;
    gp.max_iterations = cfg.max_iterations;
    gp.min_effective = min_effective;
    gp.rot_thres = cfg.rotation_converge_thres;
    gp.pos_thres = cfg.position_converge_thres;
    return gp;
}

// control block of scan s of a GN loop: its state, LL rows and pose record, stop rule, iteration log and result slot
GnLoopCtl Handle::gn_ctl(int s, int method, int min_effective, unsigned tag_base, uint4* rows, uint4* pose) const {
    GnLoopCtl c{};
    c.state = state.p + s;
    c.ll_rows = rows;
    c.ll_pose = pose;
    c.tag_base = tag_base;
    c.gp = gn_params(method, min_effective);
    c.log = scan_log(s);
    c.log_cap = log_cap;
    c.result = scan_result(s);
    return c;
}

unsigned char* Handle::table(size_t bytes) {
    if (bytes > h_batch_cap) {
        if (h_batch) cudaFreeHost(h_batch);
        h_batch = nullptr;
        h_batch_cap = 0;
        FLS_CUDA(cudaMallocHost(&h_batch, bytes * 2 + 65536));
        h_batch_cap = bytes * 2 + 65536;
    }
    d_batch.reserve(bytes);
    return h_batch;
}

void Handle::send_table(size_t bytes) {
    FLS_CUDA(cudaMemcpyAsync(d_batch.p, h_batch, bytes, cudaMemcpyHostToDevice, stream));
    h2d_bytes += (long long)bytes;
}

void Handle::read_back(int B) {
    FLS_CUDA(cudaMemcpyAsync(h_state, state.p, sizeof(GnState) * (size_t)B, cudaMemcpyDeviceToHost, stream));
    d2h_bytes += (long long)(sizeof(GnState) * (size_t)B);
    if (log_cap) {
        FLS_CUDA(cudaMemcpyAsync(h_log.data(), log.p, sizeof(fls_iter_log) * log_cap, cudaMemcpyDeviceToHost, stream));
        d2h_bytes += (long long)(sizeof(fls_iter_log) * log_cap);
    }
}

void Handle::unpack(int B, const size_t* n, double* T, int* converged, fls_match_stats* st) {
    float kernel_ms = 0.f;
    if (profile) FLS_CUDA(cudaEventElapsedTime(&kernel_ms, prof_ev[0], prof_ev[1]));
    for (int s = 0; s < B; ++s) {
        const GnState& gs = h_state[s];
        double* Ts = T + 16 * s;
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) Ts[c * 4 + r] = gs.R[r * 3 + c];
            Ts[12 + r] = gs.t[r];
        }
        Ts[3] = Ts[7] = Ts[11] = 0.0;
        Ts[15] = 1.0;
        if (converged) converged[s] = gs.converged;
        if (st) {
            fls_match_stats& o = st[s];
            if (s > 0) std::memset(&o, 0, sizeof(o));  // call-level figures (times, launches, copies) are reported on scan 0
            o.iterations = gs.iter;
            o.converged = gs.converged;
            o.n_source = (long long)n[s];
            o.n_valid = gs.n_valid;
            o.sum_residual = gs.sum_res;
            if (profile) {
                // algorithmic bytes are per scan; the launch and its time are shared by the batch and reported on scan 0
                o.algo_bytes = (long long)gs.iter * (long long)n[s] * per_point_iter_bytes + (long long)(gs.cand_total + 0.5) * per_cand_bytes;
                o.kernel_ms = s == 0 ? kernel_ms : 0.f;
                o.kernel_launches = s == 0 ? 1 : 0;
            }
        }
    }
    std::memcpy(T_final, T, sizeof(T_final));
    log_n = h_state[0].iter < log_cap ? h_state[0].iter : log_cap;
}

// tools/k1_trace.py and the profiles/ summaries parse these lines
void Handle::dump_timing(int B, size_t n0, bool v9) const {
    const GnState& g0 = h_state[0];
    const int iters = g0.iter > 0 ? g0.iter : 1;
    if (cfg.method == FLS_P2PLANE_IVOX)
        std::fprintf(stderr, "[fls timing] batch %d  scan 0: iters %d  candidates/pt-iter %.1f\n", B, g0.iter, g0.cand_total / (double)((long long)n0 * iters));
    else
        std::fprintf(stderr, "[fls timing] iters %d  candidates/pt-iter %.1f  qr-fallback points/iter %.0f of %lld\n", g0.iter,
                     g0.cand_total / (double)((long long)n0 * iters), g0.hits_total / (double)iters, (long long)n0);
    if (v9 && std::getenv("FLS_K1_TRACE")) {
        const unsigned long long* c = &g0.dbg[8][0];
        std::fprintf(stderr, "[fls trace] warp-time us: wait %.0f prefetch %.0f compute %.0f - %.0f | chunks %llu mean compute %.2f us max %.1f us | mixed chunks %llu exact lanes %llu\n",
                     c[0] * 1e-3, c[1] * 1e-3, c[2] * 1e-3, c[3] * 1e-3, c[5], c[5] ? c[2] * 1e-3 / c[5] : 0.0, c[4] * 1e-3, c[6], c[7]);
        for (int it = 0; it < g0.iter && it < 4; ++it)
            std::fprintf(stderr, "[fls trace] it %d: row(cta0)->last row out %.1f us | last row out->folder has all %.1f us | fold trips %llu, first take %.1f us and half %.1f us before the end\n", it,
                         ((double)g0.dbg[10 + it][0] - (double)g0.dbg[it][2]) * 1e-3, ((double)g0.dbg[it][3] - (double)g0.dbg[10 + it][0]) * 1e-3,
                         g0.dbg[10 + it][1], ((double)g0.dbg[it][3] - (double)g0.dbg[10 + it][2]) * 1e-3, ((double)g0.dbg[it][3] - (double)g0.dbg[10 + it][3]) * 1e-3);
    }
    for (int it = 0; it < g0.iter && it < 16; ++it) {
        const unsigned long long* d = g0.dbg[it];
        if (v9)  // [0] item opened on CTA 0, [1] CTA 0 saw the tickets exhausted, [2] CTA 0's row out, [3] folder has all rows
            std::fprintf(stderr, "[fls timing] it %d: open->exhausted %.1f us | exhausted->row(cta0) %.1f us | row(cta0)->all rows %.1f us | all rows->next open %.1f us\n", it,
                         (d[1] - d[0]) * 1e-3, ((double)d[2] - (double)d[1]) * 1e-3, ((double)d[3] - (double)d[2]) * 1e-3,
                         (it + 1 < g0.iter && it + 1 < 16) ? ((double)g0.dbg[it + 1][0] - (double)d[3]) * 1e-3 : 0.0);
        else
            std::fprintf(stderr, "[fls timing] it %d: until all rows in %.1f us | fold %.1f us | solve+publish %.1f us | to next start %.1f us\n", it,
                         (d[1] - d[0]) * 1e-3, (d[2] - d[1]) * 1e-3, (d[3] - d[2]) * 1e-3,
                         (it + 1 < g0.iter && it + 1 < 16) ? (g0.dbg[it + 1][0] - d[3]) * 1e-3 : 0.0);
    }
}

void Handle::finish_match(double* T, int* converged, fls_match_stats* st, size_t n_source) {
    read_back(1);
    end_call(st);
    if (std::getenv("FLS_DEBUG_TIMING")) dump_timing(1, n_source, false);
    unpack(1, &n_source, T, converged, st);
}

// AddCloudToLocalMap of the plug-ins that take one cloud (LoamFull takes {planar, corner}: add_cloud_kd)
int Handle::add_cloud(const float4* d, size_t n) {
    switch (cfg.method) {
        case FLS_P2PLANE_IVOX: return add_cloud_ivox(d, n);
        case FLS_NDT: return add_cloud_ndt(d, n);
        case FLS_ICP_P2P: return add_cloud_icp(d, n);
        case FLS_P2PLANE_KNN: return add_cloud_kd(d, n, nullptr, 0);
        default: return FLS_ERR_UNSUPPORTED;
    }
}

// ---- LoamPointToPlaneIVOX ------------------------------------------------------------------------------------
int Handle::add_cloud_ivox(const float4* d, size_t n) {
    if (cfg.localization_mode) ivox.clear();  // loam_point_to_plane_ivox.h:64-69 upstream: map re-created per call
    else if (ivox.n_pts != 0) return FLS_ERR_UNSUPPORTED;  // external non-first insert relies on Match-internal caches upstream
    const int rc = ivox.append_and_build(d, n, cfg.ivox_capacity, stream);
    launches += ivox.launches;
    ivox.launches = 0;
    if (cfg.localization_mode) set_fit_cloud(d, n);  // :134-138 kd-tree over the raw planar cloud
    return rc;
}

// The whole LoamPointToPlaneIVOX Match of `n_scans` independent scans in one persistent launch (K1, fls_p2plane.cu).
// A single Match is the batch of one.
int Handle::match_ivox_batch(int B, const float4* const* d_scans, const size_t* n, double* T, int* converged, fls_match_stats* st) {
    const int rc = enqueue_ivox_batch(B, d_scans, n, T);
    if (rc != FLS_OK) return rc;
    return finish_ivox_batch(T, converged, st);
}

// everything of a batch up to the asynchronous read-back of the states: nothing here waits for the device
int Handle::enqueue_ivox_batch(int B, const float4* const* d_scans, const size_t* n, const double* T) {
    if (ivox.n_pts == 0) return FLS_ERR_NO_MAP;
    if (B < 1 || B > kMaxBatch) return FLS_ERR_INVALID_ARG;
    int off[kMaxBatch + 1];
    off[0] = 0;
    int grid = 1;
    // K1 generations: the dataflow kernel (v9: TMA-staged runs, work ring, DMMA sums — fls_p2plane_v9.cu) serves batches; a single
    // Match runs on the barrier kernel (v8, fls_p2plane.cu) whose one-chunk-per-warp round has the shorter hand-over (measured on
    // B200, 108 k points: 139 vs 191 us per Match kernel; batch of 8: 683 vs 609 us).  FLS_K1=8 / 9 forces one of them.
    const char* k1 = std::getenv("FLS_K1");
    const int k1v = k1 ? std::atoi(k1) : 0;
    const bool use_v9 = k1v == 9 || (k1v != 8 && B > 1);
    for (int s = 0; s < B; ++s) {
        if (n[s] > 0x3fffffffull || (long long)off[s] + (long long)n[s] > 0x7ffffff0ll) return FLS_ERR_INVALID_ARG;
        off[s + 1] = off[s] + (int)n[s];
        const int g = use_v9 ? p2plane_v9_grid((int)n[s], cfg.device) : p2plane_grid((int)n[s], cfg.device);
        if (g > grid) grid = g;
    }
    const int n_total = off[B];
    const size_t nt = (size_t)n_total;
    rec0.reserve(nt + 1);
    rec1.reserve(nt + 1);
    flags.reserve(nt + 1);
    src_f.reserve(nt + 1);
    state.reserve(kMaxBatch);
    if (log_cap) log.reserve((size_t)log_cap * kMaxBatch);
    // hand-over buffers: one LL row per CTA + one LL pose record per scan
    const unsigned tag_base = next_epoch((size_t)B * grid * 32 + (size_t)B * kLlPoseLen + (size_t)B * 16 * 32);
    // ---- per-batch tables, staged in one pinned block and sent with one copy -------------------------------------------
    const size_t o_pose = 0, o_off = o_pose + sizeof(PoseArg) * kMaxBatch, o_desc = o_off + sizeof(int) * (kMaxBatch + 4),
                 o_ptr = o_desc + sizeof(P2PlaneScan) * kMaxBatch;
    const size_t tbl_bytes = o_ptr + sizeof(void*) * kMaxBatch;
    unsigned char* tbl = table(tbl_bytes);
    PoseArg* hp = reinterpret_cast<PoseArg*>(tbl + o_pose);
    int* ho = reinterpret_cast<int*>(tbl + o_off);
    P2PlaneScan* hd = reinterpret_cast<P2PlaneScan*>(tbl + o_desc);
    const float4** hq = reinterpret_cast<const float4**>(tbl + o_ptr);
    uint4* pose_base = ll_rows.p + (size_t)B * grid * 32;
    for (int s = 0; s < B; ++s) {
        const double* Ts = T + 16 * s;
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) hp[s].R[r * 3 + c] = Ts[c * 4 + r];
            hp[s].t[r] = Ts[12 + r];
        }
        ho[s] = off[s];
        hq[s] = d_scans[s];
        P2PlaneScan& d = hd[s];
        d.src = src_f.p + off[s];
        d.n = (int)n[s];
        d.tag_base = tag_base;
        d.state = state.p + s;
        d.rec0 = rec0.p + off[s];
        d.rec1 = rec1.p + off[s];
        d.flags = flags.p + off[s];
        d.rows = ll_rows.p + (size_t)s * grid * 32;
        d.ll_pose = pose_base + (size_t)s * kLlPoseLen;
        d.log = scan_log(s);
        d.result = scan_result(s);
        d.grows = pose_base + (size_t)B * kLlPoseLen + (size_t)s * 16 * 32;
    }
    ho[B] = off[B];
    send_table(tbl_bytes);
    const PoseArg* d_poses = reinterpret_cast<const PoseArg*>(d_batch.p + o_pose);
    const int* d_off = reinterpret_cast<const int*>(d_batch.p + o_off);
    const P2PlaneScan* d_desc = reinterpret_cast<const P2PlaneScan*>(d_batch.p + o_desc);
    const float4* const* d_ptrs = reinterpret_cast<const float4* const*>(d_batch.p + o_ptr);
    // one prep kernel (state init, flag reset, locality keys) + ONE radix sort + gather for the whole batch: the queries of
    // every scan end up in Morton order of the voxel they fall into at the initial pose (locality only: the sums are
    // order-free up to fp64 rounding, and the persistent per-point records live in the same order for the whole Match)
    prepare_queries(d_ptrs, n_total, d_off, B, d_poses, state.p, ivox_view(), flags.p, src_f.p, scratch, stream, &launches);
    P2PlaneLoopArgs a;
    a.map = ivox_view();
    a.plane_thres = cfg.point_to_planar_thres;
    a.gp = gn_params(FLS_P2PLANE_IVOX, 50);
    a.log_cap = log_cap;
    a.scans = d_desc;
    a.n_scans = B;
    {
        const char* e = std::getenv("FLS_VISIT_GROUP");
        const int v = e ? std::atoi(e) : 8;  // measured at batch 8: group 2 / 3 / 4 / 6 / 8 -> 783 / 734 / 703 / 724 / 687 us per launch
        a.visit_group = v < 1 ? 1 : (v > 8 ? 8 : v);
        if (use_v9) {  // v9 reads the field as tuning knobs of the server's refill policy (fls_p2plane_v9.cu); 0 = defaults
            const char* t = std::getenv("FLS_K1_TGT");
            const char* d = std::getenv("FLS_K1_SEC");
            a.visit_group = ((t ? std::atoi(t) : 0) & 0xff) | (((d ? std::atoi(d) : 0) & 0xff) << 8);
        }
    }
    // roofline accounting (SURVEY.md §8d, K1 — the REFERENCE algorithm's traffic): 16 B source point + n_stencil x 16 B
    // slot probes + 32 B persistent record per point-iteration, 16 B per map record resident in the stencil voxels.
    per_point_iter_bytes = 16 + 16LL * a.map.n_stencil + 32;
    per_cand_bytes = 16;
    a.tickets = nullptr;
    a.ticket_stride = 0;
    a.abort_word = nullptr;
    gn_launch([&] {
        if (use_v9) {  // chunk tickets of the dynamic work distribution: one counter per (scan, iteration)
            a.ticket_stride = cfg.max_iterations + 2;
            tickets.reserve((size_t)B * a.ticket_stride + 4);
            FLS_CUDA(cudaMemsetAsync(tickets.p, 0, sizeof(unsigned) * ((size_t)B * a.ticket_stride + 4), stream));
            a.tickets = tickets.p;
            a.abort_word = tickets.p + (size_t)B * a.ticket_stride;
            launch_p2plane_v9(a, grid, stream);
        } else {
            launch_p2plane_loop(a, grid, stream);
        }
    }, 1, d_scans[0], n[0]);
    read_back(B);
    *h_abort = 0;
    if (use_v9) FLS_CUDA(cudaMemcpyAsync(h_abort, a.abort_word, sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
    pend_n.assign(n, n + B);
    pend_v9 = use_v9;
    return FLS_OK;
}

// waits for the batch enqueued last and unpacks its results
int Handle::finish_ivox_batch(double* T, int* converged, fls_match_stats* st) {
    const int B = (int)pend_n.size();
    if (B < 1) return FLS_ERR_INVALID_ARG;
    end_call(st);
    if (pend_v9 && *h_abort) {
        pend_n.clear();
        set_last_error("p2plane_v9_kernel: watchdog — a wait loop gave up after 4 s (hand-over protocol error)");
        return FLS_ERR_CUDA;
    }
    unpack(B, pend_n.data(), T, converged, st);
    if (std::getenv("FLS_DEBUG_TIMING")) dump_timing(B, pend_n[0], pend_v9);
    pend_n.clear();
    return FLS_OK;
}

int Handle::match_p2plane_ivox(const float4* d_src, size_t n, double* T, int* converged, fls_match_stats* st) {
    const float4* scans[1] = {d_src};
    const size_t ns[1] = {n};
    const int rc = match_ivox_batch(1, scans, ns, T, converged, st);
    if (rc != FLS_OK) return rc;
    const int ni = (int)n;
    if (h_state->converged && !cfg.localization_mode) {
        // :205-206 — the scan enters the map through the cached-5-NN rule (body-frame points, final pose)  [quirk 8]
        stage.reserve(n + 1);
        stage2.reserve(n + 1);
        const GnState& s = *h_state;
        const size_t n_add = select_ivox_inserts(ivox_view(), d_src, ni, s.Rprev, s.tprev, s.R, s.t, 0.5 /* filter_size_map_min_ (:351) */,
                                                 stage2.p, stage.p, scratch, stream, &launches);
        const int rc2 = ivox.append_and_build(stage.p, n_add, cfg.ivox_capacity, stream);
        launches += ivox.launches;
        ivox.launches = 0;
        FLS_CUDA(cudaStreamSynchronize(stream));
        if (st) st->gpu_launches = launches;
        if (rc2 != FLS_OK) return rc2;
    }
    return FLS_OK;
}

// ---- IncrementalNDT ----------------------------------------------------------------------------------------------
int Handle::add_cloud_ndt(const float4* d_cloud, size_t n) {
    const int rc = ndt.add_cloud(d_cloud, n, cfg.source_cloud_filter_size, ndt_first_scan, stream);
    launches += ndt.launches;
    ndt.launches = 0;
    if (cfg.localization_mode && rc == FLS_OK) {
        // kdtree_flann_.setInputCloud(cloud_world) — the voxel-filtered cloud (incremental_ndt.h:188-190)
        const size_t nf = voxel_grid_device(d_cloud, n, cfg.source_cloud_filter_size, ndt.filtered.p, ndt.scratch, stream, &launches);
        set_fit_cloud(ndt.filtered.p, nf);
    }
    ndt_first_scan = cfg.localization_mode != 0;  // :222-226
    return rc;
}

int Handle::match_ndt(const float4* d_in, size_t n_in, double* T, int* converged, fls_match_stats* st) {
    if (ndt.n_vox == 0) return FLS_ERR_NO_MAP;  // CHECK(!grids_.empty())
    src_f.reserve(n_in);
    const size_t n = voxel_grid_device(d_in, n_in, cfg.source_cloud_filter_size, src_f.p, scratch, stream, &launches);  // :232
    const int ni = (int)n;
    const int grid = ndt_grid(ni, cfg.device);
    const unsigned tag_base = next_epoch((size_t)grid * 32 + kLlPoseLen);
    const GnLoopCtl ctl = gn_ctl(0, FLS_NDT, cfg.ndt_min_effective_pts, tag_base, ll_rows.p, ll_rows.p + (size_t)grid * 32);
    double T_in[16];
    std::memcpy(T_in, T, sizeof(T_in));
    launch_gn_init(state.p, T, stream);
    launches++;
    NdtArgs a;
    a.src = src_f.p;
    a.n = ni;
    a.map = ndt.view();
    a.outlier_thres = cfg.ndt_outlier_thres;
    a.state = state.p;
    // roofline accounting (SURVEY.md §8d, K2): 16 B source point + 7 x 16 B slot probes per point-iteration,
    // 80 B voxel record per estimated voxel hit; the 6x6 sums are fused (no per-point output).
    per_point_iter_bytes = 16 + 16LL * 7;
    per_cand_bytes = 80;
    gn_launch([&] { launch_ndt_loop(a, ctl, grid, stream); }, 1, src_f.p, n);
    finish_match(T, converged, st, n);
    if (!h_state->failed && !cfg.localization_mode) {
        // :326-330 — the scan enters the map transformed by the INPUT guess T, not the optimised pose  [quirk 6]
        stage2.reserve(n);
        launch_transform_f(src_f.p, n, T_in, stage2.p, stream);
        launches++;
        const int rc2 = add_cloud_ndt(stage2.p, n);
        FLS_CUDA(cudaStreamSynchronize(stream));
        if (st) st->gpu_launches = launches;
        if (rc2 != FLS_OK) return rc2;
    }
    return FLS_OK;
}

// Match's own VoxelGridCloud of every source of a batch (NDT, ICP), back to back in src_f: scan s at off[s], nf[s] points.  Also
// sizes the per-scan state and logs.  False when a filtered scan is too large for the kernels' int counts.
bool Handle::filter_batch(int B, const float4* const* d_scans, const size_t* n_in, size_t* off, size_t* nf) {
    size_t total_in = 0;
    for (int s = 0; s < B; ++s) total_in += n_in[s];
    src_f.reserve(total_in + 1);
    state.reserve(kMaxBatch);
    if (log_cap) log.reserve((size_t)log_cap * kMaxBatch);
    off[0] = 0;
    for (int s = 0; s < B; ++s) {
        nf[s] = voxel_grid_device(d_scans[s], n_in[s], cfg.source_cloud_filter_size, src_f.p + off[s], scratch, stream, &launches);
        if (nf[s] > 0x3fffffffull) return false;
        off[s + 1] = off[s] + nf[s];
    }
    return true;
}

// Sub-grids of a batch launch (NDT, ICP, kd-tree point-to-plane): every scan gets the CTAs its points need, scaled down together
// when the device cannot hold them all.  A scan of a batch that fits runs on the CTAs of its single Match, hence gives its result
// bit for bit.  Returns the grid, 0 when the device cannot give every scan a CTA.
static int split_subgrids(int B, const int* need, int cap, int* ncta) {
    if (B > cap) return 0;
    int tot_need = 0;
    for (int s = 0; s < B; ++s) tot_need += need[s];
    int grid = 0;
    for (int s = 0; s < B; ++s) {
        ncta[s] = tot_need <= cap ? need[s] : (int)((long long)need[s] * (cap - B) / tot_need) + 1;
        grid += ncta[s];
    }
    return grid;
}

// n_scans independent IncrementalNDT::Match calls against the same (static) map in ONE cooperative launch (fls_ndt.cu:
// ndt_gn_batch_kernel — one sub-grid and one persistent Gauss-Newton loop per scan).  Localization semantics only: the map is
// not modified (incremental_ndt.h:222-226, flag_first_scan_ stays set).
int Handle::match_ndt_batch(int B, const float4* const* d_scans, const size_t* n_in, double* T, int* converged, fls_match_stats* st) {
    if (ndt.n_vox == 0) return FLS_ERR_NO_MAP;
    if (B < 1 || B > kMaxBatch) return FLS_ERR_INVALID_ARG;
    size_t off[kMaxBatch + 1], nf[kMaxBatch];
    if (!filter_batch(B, d_scans, n_in, off, nf)) return FLS_ERR_INVALID_ARG;  // incremental_ndt.h:232
    int need[kMaxBatch], ncta[kMaxBatch];
    for (int s = 0; s < B; ++s) need[s] = std::max(1, (int)((nf[s] + kNdtBlock - 1) / kNdtBlock));
    const int grid = split_subgrids(B, need, ndt_max_grid(cfg.device), ncta);
    if (grid == 0) return FLS_ERR_INVALID_ARG;
    const unsigned tag_base = next_epoch((size_t)grid * 32 + (size_t)B * kLlPoseLen);
    const size_t tbl_bytes = sizeof(NdtBatchItem) * (size_t)B;
    NdtBatchItem* items = reinterpret_cast<NdtBatchItem*>(table(tbl_bytes));
    uint4* pose_base = ll_rows.p + (size_t)grid * 32;
    int cta0 = 0;
    for (int s = 0; s < B; ++s) {
        launch_gn_init(state.p + s, T + 16 * s, stream);
        launches++;
        NdtBatchItem& it = items[s];
        std::memset(&it, 0, sizeof(it));
        it.a.src = src_f.p + off[s];
        it.a.n = (int)nf[s];
        it.a.map = ndt.view();
        it.a.outlier_thres = cfg.ndt_outlier_thres;
        it.a.state = state.p + s;
        it.ctl = gn_ctl(s, FLS_NDT, cfg.ndt_min_effective_pts, tag_base, ll_rows.p + (size_t)cta0 * 32, pose_base + (size_t)s * kLlPoseLen);
        it.cta0 = cta0;
        it.ncta = ncta[s];
        cta0 += ncta[s];
    }
    send_table(tbl_bytes);
    per_point_iter_bytes = 16 + 16LL * 7;
    per_cand_bytes = 80;
    gn_launch([&] { launch_ndt_batch(reinterpret_cast<const NdtBatchItem*>(d_batch.p), B, grid, stream); }, 1, src_f.p, nf[0]);
    read_back(B);
    end_call(st);
    unpack(B, nf, T, converged, st);
    return FLS_OK;
}

// ---- IcpOptimized ------------------------------------------------------------------------------------------------
int Handle::add_cloud_icp(const float4* d_cloud, size_t n) {
    // icp_optimized.h:173-187: sliding window of the last local_map_size clouds (the map is replaced in localization mode),
    // then local_map_ptr_ = VoxelGridCloud(local_map_ptr_, map_cloud_filter_size_); GetFitnessScore searches the same tree
    const int rc = window_add(icp_map, d_cloud, n, (size_t)cfg.local_map_size, cfg.map_cloud_filter_size, 0, cfg.localization_mode != 0);
    set_fit_view(icp_map.cloud.p, icp_map.n);
    return rc;
}

static void mat3_from_T(const double* T, double* R) {
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[r * 3 + c] = T[c * 4 + r];
}

// IsNeedAddCloud (icp_optimized.h:218-236, loam_point_to_plane_kdtree.h:186-202, loam_full_kdtree.h:356-371): key-frame
// gating on translation / RPY deltas against a persistent last_T that starts at the first pose it sees  [quirk 7]
bool Handle::need_add_cloud(const double* T, double* last_T, bool* have_last) const {
    if (!*have_last) {
        std::memcpy(last_T, T, 16 * sizeof(double));
        *have_last = true;
    }
    double Rl[9], Rc[9], Rli[9], Rd[9];
    mat3_from_T(last_T, Rl);
    mat3_from_T(T, Rc);
    {  // 3x3 inverse by cofactors
        const double c00 = Rl[4] * Rl[8] - Rl[5] * Rl[7], c01 = Rl[5] * Rl[6] - Rl[3] * Rl[8], c02 = Rl[3] * Rl[7] - Rl[4] * Rl[6];
        const double id = 1.0 / (Rl[0] * c00 + Rl[1] * c01 + Rl[2] * c02);
        Rli[0] = c00 * id; Rli[1] = (Rl[2] * Rl[7] - Rl[1] * Rl[8]) * id; Rli[2] = (Rl[1] * Rl[5] - Rl[2] * Rl[4]) * id;
        Rli[3] = c01 * id; Rli[4] = (Rl[0] * Rl[8] - Rl[2] * Rl[6]) * id; Rli[5] = (Rl[2] * Rl[3] - Rl[0] * Rl[5]) * id;
        Rli[6] = c02 * id; Rli[7] = (Rl[1] * Rl[6] - Rl[0] * Rl[7]) * id; Rli[8] = (Rl[0] * Rl[4] - Rl[1] * Rl[3]) * id;
    }
    mat3_mul(Rli, Rc, Rd);
    const double roll = std::atan2(Rd[7], Rd[8]), pitch = std::asin(-Rd[6]), yaw = std::atan2(Rd[3], Rd[0]);
    const double dt[3] = {T[12] - last_T[12], T[13] - last_T[13], T[14] - last_T[14]};
    if (norm3(dt) > cfg.dist_thre_add_cloud || std::fabs(roll) > cfg.rot_thre_add_cloud || std::fabs(pitch) > cfg.rot_thre_add_cloud ||
        std::fabs(yaw) > cfg.rot_thre_add_cloud) {
        std::memcpy(last_T, T, 16 * sizeof(double));
        return true;
    }
    return false;
}

int Handle::match_icp(const float4* d_in, size_t n_in, double* T, int* converged, fls_match_stats* st) {
    if (n_in <= 10) return FLS_ERR_TOO_FEW_POINTS;  // CHECK_GT(ordered_cloud_.size(), 10u)  (:55)
    if (icp_map.grid.n_pts == 0) return FLS_ERR_NO_MAP;
    src_f.reserve(n_in);
    const size_t n = voxel_grid_device(d_in, n_in, cfg.source_cloud_filter_size, src_f.p, scratch, stream, &launches);  // :57
    const int ni = (int)n;
    const int grid = icp_grid_blocks(ni, cfg.device);
    const unsigned tag_base = next_epoch((size_t)grid * 32 + kLlPoseLen);
    const GnLoopCtl ctl = gn_ctl(0, FLS_ICP_P2P, 0, tag_base, ll_rows.p, ll_rows.p + (size_t)grid * 32);
    launch_gn_init(state.p, T, stream);
    launches++;
    IcpArgs a;
    a.src = src_f.p;
    a.n = ni;
    a.map = grid_view(icp_map.grid);
    a.max_corr = cfg.icp_max_correspond_distance;
    a.state = state.p;
    // roofline accounting (SURVEY.md §8d, K3): 16 B source point + 27 x 16 B slot probes, 16 B per scanned map record
    per_point_iter_bytes = 16 + 16LL * 27;
    per_cand_bytes = 16;
    gn_launch([&] { launch_icp_loop(a, ctl, grid, stream); }, 1, src_f.p, n);
    finish_match(T, converged, st, n);
    if (h_state->converged && !cfg.localization_mode) {
        // IsNeedAddCloud (:218-236): key-frame gating on translation / RPY deltas against a persistent last_T
        if (need_add_cloud(T, icp_last_T, &icp_have_last)) {
            stage.reserve(n);
            launch_transform_f(src_f.p, n, T, stage.p, stream);  // :156 TransformPointCloud(source, final) in float
            launches++;
            const int rc2 = add_cloud_icp(stage.p, n);
            FLS_CUDA(cudaStreamSynchronize(stream));
            if (st) st->gpu_launches = launches;
            if (rc2 != FLS_OK) return rc2;
        }
    }
    return FLS_OK;
}

// n_scans independent IcpOptimized::Match calls against the same (static) map in ONE cooperative launch (fls_icp.cu:
// icp_gn_batch_kernel — one sub-grid and one persistent Gauss-Newton loop per scan).  Localization mode: the map is not modified.
int Handle::match_icp_batch(int B, const float4* const* d_scans, const size_t* n_in, double* T, int* converged, fls_match_stats* st) {
    if (B < 1 || B > kMaxBatch) return FLS_ERR_INVALID_ARG;
    for (int s = 0; s < B; ++s)
        if (n_in[s] <= 10) return FLS_ERR_TOO_FEW_POINTS;  // CHECK_GT(ordered_cloud_.size(), 10u)  (:55), for the whole call
    if (icp_map.grid.n_pts == 0) return FLS_ERR_NO_MAP;
    size_t off[kMaxBatch + 1], nf[kMaxBatch];
    if (!filter_batch(B, d_scans, n_in, off, nf)) return FLS_ERR_INVALID_ARG;  // :57
    int need[kMaxBatch], ncta[kMaxBatch];
    for (int s = 0; s < B; ++s) need[s] = std::max(1, (int)((nf[s] + kIcpPerBlock - 1) / kIcpPerBlock));
    const int grid = split_subgrids(B, need, icp_max_grid(cfg.device), ncta);
    if (grid == 0) return FLS_ERR_INVALID_ARG;
    const unsigned tag_base = next_epoch((size_t)grid * 32 + (size_t)B * kLlPoseLen);
    const size_t tbl_bytes = sizeof(IcpBatchItem) * (size_t)B;
    IcpBatchItem* items = reinterpret_cast<IcpBatchItem*>(table(tbl_bytes));
    uint4* pose_base = ll_rows.p + (size_t)grid * 32;
    const IvoxView map = grid_view(icp_map.grid);
    int cta0 = 0;
    for (int s = 0; s < B; ++s) {
        launch_gn_init(state.p + s, T + 16 * s, stream);
        launches++;
        IcpBatchItem& it = items[s];
        std::memset(&it, 0, sizeof(it));
        it.a.src = src_f.p + off[s];
        it.a.n = (int)nf[s];
        it.a.map = map;
        it.a.max_corr = cfg.icp_max_correspond_distance;
        it.a.state = state.p + s;
        it.ctl = gn_ctl(s, FLS_ICP_P2P, 0, tag_base, ll_rows.p + (size_t)cta0 * 32, pose_base + (size_t)s * kLlPoseLen);
        it.cta0 = cta0;
        it.ncta = ncta[s];
        cta0 += ncta[s];
    }
    send_table(tbl_bytes);
    per_point_iter_bytes = 16 + 16LL * 27;
    per_cand_bytes = 16;
    // GetFitnessScore after a batch scores scan 0 at its final pose
    gn_launch([&] { launch_icp_batch(reinterpret_cast<const IcpBatchItem*>(d_batch.p), B, grid, stream); }, 1, src_f.p, nf[0]);
    read_back(B);
    end_call(st);
    unpack(B, nf, T, converged, st);
    return FLS_OK;
}

// ---- LoamPointToPlaneKdtree / LoamFull -------------------------------------------------------------------------------
static LoamGrid loam_grid_of(const Handle::WindowMap& w) {
    LoamGrid g;
    g.pts = w.grid.pts_sorted.p;
    g.tab = w.grid.table.p;
    g.mask = w.grid.mask;
    g.inv_cell = w.grid.inv_res;
    g.cell = w.grid.res;
    g.n_pts = (unsigned)w.grid.n_pts;
    return g;
}

int Handle::window_add(WindowMap& w, const float4* d_cloud, size_t n, size_t window, float leaf, int filter_mode, bool replace) {
    const float4* merged = d_cloud;
    size_t n_merged = n;
    size_t depth = 1;
    if (!replace) {
        std::unique_ptr<Cloud> c(new Cloud());
        c->buf.reserve(n);
        if (n) FLS_CUDA(cudaMemcpyAsync(c->buf.p, d_cloud, n * sizeof(float4), cudaMemcpyDeviceToDevice, stream));
        c->n = n;
        w.deque.push_back(std::move(c));
        if (w.deque.size() > window) {
            FLS_CUDA(cudaStreamSynchronize(stream));  // the evicted buffer may still feed a copy in flight
            w.deque.pop_front();
        }
        n_merged = 0;
        for (auto& q : w.deque) n_merged += q->n;
        w.merged.reserve(n_merged);
        size_t off = 0;
        for (auto& q : w.deque) {
            if (q->n) FLS_CUDA(cudaMemcpyAsync(w.merged.p + off, q->buf.p, q->n * sizeof(float4), cudaMemcpyDeviceToDevice, stream));
            off += q->n;
        }
        merged = w.merged.p;
        depth = w.deque.size();
    }
    w.cloud.reserve(n_merged);
    if (filter_mode == 0 || depth > 5) {
        w.n = voxel_grid_device(merged, n_merged, leaf, w.cloud.p, scratch, stream, &launches);
    } else {
        if (n_merged) FLS_CUDA(cudaMemcpyAsync(w.cloud.p, merged, n_merged * sizeof(float4), cudaMemcpyDeviceToDevice, stream));
        w.n = n_merged;
    }
    w.grid.clear();
    const int rc = w.grid.append_and_build(w.cloud.p, w.n, 0, stream);
    launches += w.grid.launches;
    w.grid.launches = 0;
    return rc;
}

int Handle::add_cloud_kd(const float4* d_planar, size_t n_planar, const float4* d_corner, size_t n_corner) {
    if (cfg.method == FLS_P2PLANE_KNN) {
        // loam_point_to_plane_kdtree.h:56-80: localization mode replaces the map, mapping mode slides a window; both
        // end in VoxelGridCloud(local_map, map_cloud_filter_size) + kd-tree
        const int rc = window_add(kd_planar, d_planar, n_planar, (size_t)cfg.local_map_size, cfg.map_cloud_filter_size, 0,
                                  cfg.localization_mode != 0);
        if (rc == FLS_OK) set_fit_cloud(kd_planar.cloud.p, kd_planar.n);  // GetFitnessScore searches the same tree (:159-183)
        return rc;
    }
    // loam_full_kdtree.h:66-104: {planar, corner}, both windows slide, filters only beyond 5 clouds
    int rc = window_add(kd_planar, d_planar, n_planar, (size_t)cfg.local_map_size, cfg.map_cloud_filter_size, 1, false);
    if (rc != FLS_OK) return rc;
    return window_add(kd_corner, d_corner, n_corner, (size_t)cfg.corner_local_map_size, cfg.corner_map_filter_size, 1, false);
}

int Handle::match_kd(const float4* d_planar, size_t n_planar, const float4* d_corner, size_t n_corner, double* T, int* converged,
                     fls_match_stats* st) {
    const bool full = cfg.method == FLS_LOAM_FULL;
    if (kd_planar.n == 0) return FLS_ERR_NO_MAP;
    if (!full) n_corner = 0;
    const size_t n = n_planar + n_corner;
    const int ni = (int)n;
    const int grid = loam_grid_blocks(ni, cfg.device);
    const unsigned tag_base = next_epoch((size_t)grid * 32 + kLlPoseLen);
    const GnLoopCtl ctl = gn_ctl(0, cfg.method, 50, tag_base, ll_rows.p, ll_rows.p + (size_t)grid * 32);
    launch_gn_init(state.p, T, stream);
    launches++;
    rec_d.reserve(n * 8 + 8);
    flags.reserve(n + 1);
    LoamArgs a;
    a.corner = d_corner;
    a.n_corner = (int)n_corner;
    a.planar = d_planar;
    a.n_planar = (int)n_planar;
    a.planar_map = loam_grid_of(kd_planar);
    a.corner_map = full ? loam_grid_of(kd_corner) : a.planar_map;
    a.plane_thres = cfg.point_to_planar_thres;
    a.search_thres = full ? cfg.point_search_thres : INFINITY;
    a.line_ratio = cfg.line_ratio_thres;
    a.gate = full ? (float)cfg.point_search_thres * 1.0001f : INFINITY;
    a.state = state.p;
    a.rec = rec_d.p;
    a.flags = flags.p;
    // roofline accounting (K5): 16 B source point + 27 x 16 B slot probes + 56 B persistent record, 16 B per scanned map record
    per_point_iter_bytes = 16 + 16LL * 27 + 56;
    per_cand_bytes = 16;
    gn_launch([&] { launch_loam_loop(a, ctl, grid, stream); }, 2, d_planar, n_planar);
    finish_match(T, converged, st, n);
    // key-frame insertion: loam_point_to_plane_kdtree.h:146-150 (gate evaluated before the mode test), loam_full_kdtree.h:178-186
    if (h_state->converged && need_add_cloud(T, kd_last_T, &kd_have_last) && (full || !cfg.localization_mode)) {
        int rc2;
        if (full) {
            stage.reserve(n_planar);
            stage2.reserve(n_corner);
            launch_transform_d(d_planar, n_planar, T, stage.p, stream);  // pcl::transformPointCloud(cloud, out, T_) with the double matrix
            launch_transform_d(d_corner, n_corner, T, stage2.p, stream);
            launches += 2;
            rc2 = add_cloud_kd(stage.p, n_planar, stage2.p, n_corner);
        } else {
            stage.reserve(n_planar);
            launch_transform_f(d_planar, n_planar, T, stage.p, stream);  // TransformPointCloud(source, final): fp32 with R, t cast to float
            launches++;
            rc2 = add_cloud_kd(stage.p, n_planar, nullptr, 0);
        }
        FLS_CUDA(cudaStreamSynchronize(stream));
        if (st) st->gpu_launches = launches;
        if (rc2 != FLS_OK) return rc2;
    }
    return FLS_OK;
}

// n_scans independent LoamPointToPlaneKdtree::Match calls (planar clouds) against the same (static) map in ONE cooperative launch
// (fls_loam.cu: loam_gn_batch_kernel).  Localization mode: no key frame is inserted, so the scans are independent; the key-frame
// gate's last_T, which match_kd updates even there, is read only by insertions and is left alone.
int Handle::match_kd_batch(int B, const float4* const* d_scans, const size_t* n, double* T, int* converged, fls_match_stats* st) {
    if (B < 1 || B > kMaxBatch) return FLS_ERR_INVALID_ARG;
    if (kd_planar.n == 0) return FLS_ERR_NO_MAP;
    size_t off[kMaxBatch + 1];
    off[0] = 0;
    for (int s = 0; s < B; ++s) {
        if (n[s] > 0x3fffffffull) return FLS_ERR_INVALID_ARG;
        off[s + 1] = off[s] + n[s];
    }
    if (off[B] > 0x7ffffff0ull) return FLS_ERR_INVALID_ARG;
    int need[kMaxBatch], ncta[kMaxBatch];
    for (int s = 0; s < B; ++s) need[s] = std::max(1, (int)((n[s] + kLoamPerBlock - 1) / kLoamPerBlock));
    const int grid = split_subgrids(B, need, loam_max_grid(cfg.device), ncta);
    if (grid == 0) return FLS_ERR_INVALID_ARG;
    state.reserve(kMaxBatch);
    if (log_cap) log.reserve((size_t)log_cap * kMaxBatch);
    rec_d.reserve(off[B] * 8 + 8);
    flags.reserve(off[B] + 1);
    const unsigned tag_base = next_epoch((size_t)grid * 32 + (size_t)B * kLlPoseLen);
    const size_t tbl_bytes = sizeof(LoamBatchItem) * (size_t)B;
    LoamBatchItem* items = reinterpret_cast<LoamBatchItem*>(table(tbl_bytes));
    uint4* pose_base = ll_rows.p + (size_t)grid * 32;
    const LoamGrid planar_map = loam_grid_of(kd_planar);
    int cta0 = 0;
    for (int s = 0; s < B; ++s) {
        launch_gn_init(state.p + s, T + 16 * s, stream);
        launches++;
        LoamBatchItem& it = items[s];
        std::memset(&it, 0, sizeof(it));
        it.a.corner = d_scans[s];
        it.a.n_corner = 0;
        it.a.planar = d_scans[s];
        it.a.n_planar = (int)n[s];
        it.a.planar_map = planar_map;
        it.a.corner_map = planar_map;
        it.a.plane_thres = cfg.point_to_planar_thres;
        it.a.search_thres = INFINITY;
        it.a.line_ratio = cfg.line_ratio_thres;
        it.a.gate = INFINITY;
        it.a.state = state.p + s;
        it.a.rec = rec_d.p + off[s] * 8;
        it.a.flags = flags.p + off[s];
        it.ctl = gn_ctl(s, FLS_P2PLANE_KNN, 50, tag_base, ll_rows.p + (size_t)cta0 * 32, pose_base + (size_t)s * kLlPoseLen);
        it.cta0 = cta0;
        it.ncta = ncta[s];
        cta0 += ncta[s];
    }
    send_table(tbl_bytes);
    per_point_iter_bytes = 16 + 16LL * 27 + 56;
    per_cand_bytes = 16;
    // GetFitnessScore after a batch scores scan 0 at its final pose
    gn_launch([&] { launch_loam_batch(reinterpret_cast<const LoamBatchItem*>(d_batch.p), B, grid, flags.p, (int)off[B], stream); }, 2, d_scans[0],
              n[0]);
    read_back(B);
    end_call(st);
    unpack(B, n, T, converged, st);
    return FLS_OK;
}

// ---- GetFitnessScore -------------------------------------------------------------------------------------------------
int Handle::fitness(float max_range, float* score) {
    *score = 3.402823466e+38f;  // FloatNaN / "no inliers" upstream
    if (cfg.method == FLS_LOAM_FULL) return FLS_OK;  // loam_full_kdtree.h:206-208 FloatNaN
    // ICP and the kd-tree point-to-plane plug-in always search their tree; NDT / iVox return FloatNaN outside localization mode
    if (cfg.method != FLS_ICP_P2P && cfg.method != FLS_P2PLANE_KNN && !cfg.localization_mode) return FLS_OK;
    if (fit_n == 0 || last_src == nullptr || last_src_n == 0 || !(max_range > 0.f)) return FLS_OK;
    begin_call();
    if (fit_grid_version != fit_version || fit_grid_range != max_range) {
        fit_grid.set_resolution(std::sqrt(max_range) * 1.001f);
        fit_grid.clear();
        const int rc = fit_grid.append_and_build(fit_src, fit_n, 0, stream);
        launches += fit_grid.launches;
        fit_grid.launches = 0;
        if (rc != FLS_OK) return rc;
        fit_grid_version = fit_version;
        fit_grid_range = max_range;
    }
    launch_fitness(grid_view(fit_grid), last_src, (int)last_src_n, T_final, max_range, fit_out.p, stream);
    launches++;
    double h[2] = {0, 0};
    FLS_CUDA(cudaMemcpyAsync(h, fit_out.p, sizeof(h), cudaMemcpyDeviceToHost, stream));
    end_call(nullptr);
    if (h[1] > 0) *score = (float)(h[0] / h[1]);
    return FLS_OK;
}

}  // namespace fls

// =====================================================================================================================
using fls::Handle;

#define FLS_TRY try {
#define FLS_CATCH                                              \
    }                                                          \
    catch (const fls::CudaError& e) { return e.status; }       \
    catch (const std::bad_alloc&) {                            \
        fls::set_last_error("host allocation failed");         \
        return FLS_ERR_CUDA;                                   \
    }

static bool stride_ok(size_t stride) { return stride == 16 || (stride >= 20 && stride % 4 == 0); }

extern "C" {

int fls_abi_version(void) { return FLS_ABI_VERSION; }

int fls_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char* fls_last_error(void) { return fls::last_error_cstr(); }

int fls_project(int device, const void* raw, const int32_t* ring, size_t n, size_t stride, int32_t n_rows, int32_t n_cols, float horizontal_resolution,
                float min_distance, float max_distance, float* ordered, float* depth, int32_t* col, int32_t* row_start, int32_t* row_end,
                size_t* n_ordered) {
    if ((!raw && n) || (!ring && n) || !ordered || !depth || !col || !row_start || !row_end || !n_ordered || !stride_ok(stride))
        return FLS_ERR_INVALID_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return FLS_ERR_NO_DEVICE;
    return fls::project_device(device, raw, ring, nullptr, nullptr, n, stride, n_rows, n_cols, horizontal_resolution, min_distance, max_distance, ordered,
                               depth, col, row_start, row_end, n_ordered);
}

int fls_project_imu(int device, const void* raw, const int32_t* ring, const float* time, size_t n, size_t stride, const fls_imu_buffer* imu,
                    int32_t n_rows, int32_t n_cols, float horizontal_resolution, float min_distance, float max_distance, float* ordered, float* depth,
                    int32_t* col, int32_t* row_start, int32_t* row_end, size_t* n_ordered) {
    if ((!raw && n) || (!ring && n) || !ordered || !depth || !col || !row_start || !row_end || !n_ordered || !stride_ok(stride))
        return FLS_ERR_INVALID_ARG;
    if (imu && imu->n_imu && !time && n) return FLS_ERR_INVALID_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return FLS_ERR_NO_DEVICE;
    return fls::project_device(device, raw, ring, time, imu, n, stride, n_rows, n_cols, horizontal_resolution, min_distance, max_distance, ordered,
                               depth, col, row_start, row_end, n_ordered);
}

int fls_preprocess(int device, const float* raw_xyzit, size_t n, const fls_imu_buffer* imu, float min_distance, float max_distance, int32_t jump_span,
                   float planar_leaf, float* ordered, size_t* n_ordered, float* planar, size_t* n_planar) {
    if ((!raw_xyzit && n) || !ordered || !planar || !n_ordered || !n_planar || jump_span < 1 || !(planar_leaf > 0.f)) return FLS_ERR_INVALID_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return FLS_ERR_NO_DEVICE;
    return fls::preprocess_device(device, raw_xyzit, n, imu, min_distance, max_distance, jump_span, planar_leaf, ordered, n_ordered, planar, n_planar);
}

const char* fls_strerror(int status) {
    switch (status) {
        case FLS_OK: return "ok";
        case FLS_ERR_INVALID_ARG: return "invalid argument";
        case FLS_ERR_CUDA: return "CUDA runtime error (see fls_last_error)";
        case FLS_ERR_NO_DEVICE: return "no sm_100 CUDA device (this library has no CPU fallback)";
        case FLS_ERR_UNSUPPORTED: return "method or mode not supported by this build";
        case FLS_ERR_NO_MAP: return "Match called before AddCloudToLocalMap";
        case FLS_ERR_CAPACITY: return "voxel capacity reached (LRU eviction is not emulated on the device)";
        case FLS_ERR_TOO_FEW_POINTS: return "too few points";
        default: return "unknown status";
    }
}

int fls_config_default(fls_config* c, int method) {
    if (!c || method < 0 || method > FLS_LOAM_FULL) return FLS_ERR_INVALID_ARG;
    std::memset(c, 0, sizeof(*c));
    c->method = method;
    c->device = 0;
    c->localization_mode = 1;
    c->max_iterations = 10;               // config/localization/config_turing.yaml:49
    c->position_converge_thres = 0.01;    // :51
    c->rotation_converge_thres = 0.01;    // :52
    c->point_to_planar_thres = 0.1;       // :50
    c->ivox_resolution = 0.5f;            // loam_point_to_plane_ivox.h:55
    c->ivox_nearby = FLS_NEARBY18;        // :56
    c->ivox_capacity = 1000000;           // ivox_map.h:35
    c->ivox_max_range = 5.0f;             // ivox_map.h:58
    c->ivox_k = 5;                        // ivox_map.h:57
    c->ndt_voxel_size = 1.0;              // config/mapping/config_nclt_ndt.yaml:42-51
    c->ndt_outlier_thres = 5.0;
    c->ndt_min_points_in_voxel = 5;
    c->ndt_max_points_in_voxel = 50;
    c->ndt_min_effective_pts = 50;
    c->ndt_capacity = 100000;
    c->icp_max_correspond_distance = 1.0;  // config/localization/config_nclt_icp.yaml:42-48
    c->rot_thre_add_cloud = 0.2;
    c->dist_thre_add_cloud = 1.0;
    c->local_map_size = 50;
    c->source_cloud_filter_size = 0.2f;
    c->map_cloud_filter_size = 0.4f;
    c->point_search_thres = 1.0;
    c->line_ratio_thres = 3.0;
    c->corner_map_filter_size = 0.2f;
    c->corner_local_map_size = 50;
    if (method == FLS_NDT) {
        c->max_iterations = 30;
        c->position_converge_thres = 0.005;
        c->rotation_converge_thres = 0.005;
    } else if (method == FLS_ICP_P2P) {
        c->max_iterations = 30;
        c->position_converge_thres = 0.005;
        c->rotation_converge_thres = 0.005;
        c->source_cloud_filter_size = 0.4f;
    } else if (method == FLS_P2PLANE_KNN) {
        c->max_iterations = 8;  // config/localization/config_nclt.yaml:45
        c->position_converge_thres = 0.005;
        c->rotation_converge_thres = 0.005;
        c->map_cloud_filter_size = 0.5f;
    } else if (method == FLS_LOAM_FULL) {
        c->max_iterations = 30;  // config/mapping/config_nclt_loam_full.yaml:40-58
        c->rotation_converge_thres = 0.05;
        c->point_to_planar_thres = 0.2;
    }
    return FLS_OK;
}

static int validate(const fls_config* c) {
    if (!c) return FLS_ERR_INVALID_ARG;
    if (c->method < 0 || c->method > FLS_LOAM_FULL) return FLS_ERR_INVALID_ARG;
    // the reference CHECK_NE()s every threshold against its "NaN" sentinel = numeric_limits::max (constant_variable.h:10-15)
    if (c->max_iterations <= 0 || c->max_iterations == 2147483647) return FLS_ERR_INVALID_ARG;
    if (c->max_iterations > 254) return FLS_ERR_UNSUPPORTED;  // 8-bit iteration field of the hand-over tags (fls_gn.cuh); upstream configs use 8-30
    if (!(c->position_converge_thres < 1e300) || !(c->rotation_converge_thres < 1e300)) return FLS_ERR_INVALID_ARG;
    if (c->ivox_nearby < 0 || c->ivox_nearby > 3) return FLS_ERR_INVALID_ARG;
    if (c->method == FLS_P2PLANE_IVOX) {
        if (!(c->point_to_planar_thres < 1e300) || !(c->ivox_resolution > 0.f)) return FLS_ERR_INVALID_ARG;
        if (c->ivox_k != 5) return FLS_ERR_UNSUPPORTED;  // upstream always asks for 5 (loam_point_to_plane_ivox.h:269)
    } else if (c->method == FLS_NDT) {
        if (!(c->ndt_voxel_size > 0) || !(c->ndt_voxel_size < 1e300) || !(c->ndt_outlier_thres < 1e300) || !(c->source_cloud_filter_size > 0.f) ||
            c->ndt_capacity <= 0 || c->ndt_capacity == 2147483647 || c->ndt_min_points_in_voxel < 0 || c->ndt_min_points_in_voxel > 64)
            return FLS_ERR_INVALID_ARG;
    } else if (c->method == FLS_ICP_P2P) {
        if (!(c->icp_max_correspond_distance > 0) || !(c->icp_max_correspond_distance < 1e300) || !(c->source_cloud_filter_size > 0.f) ||
            !(c->map_cloud_filter_size > 0.f) || c->local_map_size <= 0)
            return FLS_ERR_INVALID_ARG;
    } else if (c->method == FLS_P2PLANE_KNN) {
        if (!(c->point_to_planar_thres < 1e300) || !(c->rot_thre_add_cloud < 1e300) || !(c->dist_thre_add_cloud < 1e300) ||
            !(c->map_cloud_filter_size > 0.f) || c->local_map_size <= 0)
            return FLS_ERR_INVALID_ARG;  // loam_point_to_plane_kdtree.h:43-50
    } else {
        if (!(c->point_to_planar_thres < 1e300) || !(c->point_search_thres < 1e300) || !(c->point_search_thres > 0) ||
            !(c->line_ratio_thres < 1e300) || !(c->rot_thre_add_cloud < 1e300) || !(c->dist_thre_add_cloud < 1e300) ||
            !(c->map_cloud_filter_size > 0.f) || !(c->corner_map_filter_size > 0.f) || c->local_map_size <= 0 || c->corner_local_map_size <= 0)
            return FLS_ERR_INVALID_ARG;  // loam_full_kdtree.h:41-53
    }
    return FLS_OK;
}

int fls_create(const fls_config* cfg, fls_handle** out) {
    if (!out) return FLS_ERR_INVALID_ARG;
    *out = nullptr;
    const int v = validate(cfg);
    if (v != FLS_OK) return v;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || cfg->device < 0 || cfg->device >= ndev) {
        fls::set_last_error("no usable CUDA device");
        return FLS_ERR_NO_DEVICE;
    }
    FLS_TRY
    Handle* h = new Handle(*cfg);
    *out = reinterpret_cast<fls_handle*>(h);
    return FLS_OK;
    FLS_CATCH
}

void fls_destroy(fls_handle* h) { delete reinterpret_cast<Handle*>(h); }

int fls_add_cloud(fls_handle* hh, int n_clouds, const void* const* pts, const size_t* n, size_t stride) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !pts || !n || n_clouds < 1 || !stride_ok(stride)) return FLS_ERR_INVALID_ARG;
    // CHECK_EQ(cloud_list.size(), 1) everywhere except LoamFull, which takes {planar, corner} (loam_full_kdtree.h:66-68)
    const int want = h->cfg.method == FLS_LOAM_FULL ? 2 : 1;
    if (n_clouds != want) return FLS_ERR_INVALID_ARG;
    for (int k = 0; k < n_clouds; ++k)
        if (!pts[k] && n[k]) return FLS_ERR_INVALID_ARG;
    FLS_TRY
    h->begin_call();
    const float4* d = h->upload(pts[0], n[0], stride, h->stage);
    int rc;
    if (h->cfg.method == FLS_LOAM_FULL) rc = h->add_cloud_kd(d, n[0], h->upload(pts[1], n[1], stride, h->stage2), n[1]);
    else rc = h->add_cloud(d, n[0]);
    h->end_call(nullptr);
    return rc;
    FLS_CATCH
}

static int match_dispatch(Handle* h, const float4* d_ordered, size_t n_ordered, const float4* d_planar, size_t n_planar, const float4* d_corner,
                          size_t n_corner, double* T, int* converged, fls_match_stats* st) {
    switch (h->cfg.method) {
        case FLS_P2PLANE_IVOX: return h->match_p2plane_ivox(d_planar, n_planar, T, converged, st);
        case FLS_NDT: return h->match_ndt(d_ordered, n_ordered, T, converged, st);
        case FLS_ICP_P2P: return h->match_icp(d_ordered, n_ordered, T, converged, st);
        case FLS_P2PLANE_KNN:
        case FLS_LOAM_FULL: return h->match_kd(d_planar, n_planar, d_corner, n_corner, T, converged, st);
        default: return FLS_ERR_UNSUPPORTED;
    }
}

int fls_match(fls_handle* hh, const void* ordered, size_t n_ordered, const void* planar, size_t n_planar, const void* corner, size_t n_corner,
              size_t stride, double T[16], int* converged, fls_match_stats* st) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !T || !stride_ok(stride)) return FLS_ERR_INVALID_ARG;
    FLS_TRY
    if (st) std::memset(st, 0, sizeof(*st));
    h->begin_call();
    const float4* d_ord = nullptr;
    const float4* d_pla = nullptr;
    const float4* d_cor = nullptr;
    const bool uses_planar = h->cfg.method >= FLS_P2PLANE_IVOX;
    if (uses_planar) {
        if (!planar && n_planar) return FLS_ERR_INVALID_ARG;
        d_pla = h->upload(planar, n_planar, stride, h->src);
        if (h->cfg.method == FLS_LOAM_FULL) {
            if (!corner && n_corner) return FLS_ERR_INVALID_ARG;
            d_cor = h->upload(corner, n_corner, stride, h->src2);
        } else {
            n_corner = 0;
        }
    } else {
        if (!ordered && n_ordered) return FLS_ERR_INVALID_ARG;
        d_ord = h->upload(ordered, n_ordered, stride, h->src);
    }
    return match_dispatch(h, d_ord, n_ordered, d_pla, n_planar, d_cor, n_corner, T, converged, st);
    FLS_CATCH
}

int fls_match_device(fls_handle* hh, const void* d_points, size_t n, double T[16], int* converged, fls_match_stats* st) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !T || (!d_points && n)) return FLS_ERR_INVALID_ARG;
    FLS_TRY
    if (st) std::memset(st, 0, sizeof(*st));
    h->begin_call();
    const float4* d = static_cast<const float4*>(d_points);
    if (h->cfg.method == FLS_LOAM_FULL) return FLS_ERR_UNSUPPORTED;  // two feature clouds: use fls_match
    return match_dispatch(h, d, n, d, n, nullptr, 0, T, converged, st);
    FLS_CATCH
}

// Uploads B host scans back to back into h->src (packed copy, or copy + repack); ptrs receives their device addresses.
static int stage_scans(Handle* h, int B, const void* const* scans, const size_t* n, size_t stride, const float4** ptrs) {
    size_t total = 0;
    for (int s = 0; s < B; ++s) {
        if (!scans[s] && n[s]) return FLS_ERR_INVALID_ARG;
        total += n[s];
    }
    h->src.reserve(total + 1);
    if (stride != FLS_LAYOUT_PACKED) h->raw.reserve(total * stride);
    size_t off = 0;
    for (int s = 0; s < B; ++s) {
        ptrs[s] = h->src.p + off;
        if (n[s]) {
            if (stride == FLS_LAYOUT_PACKED) {
                FLS_CUDA(cudaMemcpyAsync(h->src.p + off, scans[s], n[s] * 16, cudaMemcpyHostToDevice, h->stream));
            } else {
                FLS_CUDA(cudaMemcpyAsync(h->raw.p + off * stride, scans[s], n[s] * stride, cudaMemcpyHostToDevice, h->stream));
                fls::launch_repack(h->raw.p + off * stride, n[s], stride, h->src.p + off, h->stream);
                h->launches++;
            }
            h->h2d_bytes += (long long)(n[s] * stride);
        }
        off += n[s];
    }
    return FLS_OK;
}

static int device_scans(int B, const void* const* d_scans, const size_t* n, const float4** ptrs) {
    for (int s = 0; s < B; ++s) {
        if (!d_scans[s] && n[s]) return FLS_ERR_INVALID_ARG;
        ptrs[s] = static_cast<const float4*>(d_scans[s]);
    }
    return FLS_OK;
}

// the plug-ins fls_match_batch serves: a batch of one is the single Match (so mapping mode keeps working), more go to the batch kernels
static bool batch_method(int method) { return method != FLS_LOAM_FULL; }

static int match_batch_dispatch(Handle* h, int B, const float4* const* ptrs, const size_t* n, double* T, int* converged, fls_match_stats* st) {
    switch (h->cfg.method) {
        case FLS_P2PLANE_IVOX:
            return B == 1 ? h->match_p2plane_ivox(ptrs[0], n[0], T, converged, st) : h->match_ivox_batch(B, ptrs, n, T, converged, st);
        case FLS_NDT: return B == 1 ? h->match_ndt(ptrs[0], n[0], T, converged, st) : h->match_ndt_batch(B, ptrs, n, T, converged, st);
        case FLS_ICP_P2P: return B == 1 ? h->match_icp(ptrs[0], n[0], T, converged, st) : h->match_icp_batch(B, ptrs, n, T, converged, st);
        case FLS_P2PLANE_KNN:
            return B == 1 ? h->match_kd(ptrs[0], n[0], nullptr, 0, T, converged, st) : h->match_kd_batch(B, ptrs, n, T, converged, st);
        default: return FLS_ERR_UNSUPPORTED;
    }
}

int fls_match_batch(fls_handle* hh, int n_scans, const void* const* planar, const size_t* n, size_t stride, double* T, int* converged,
                    fls_match_stats* st) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !planar || !n || !T || n_scans < 1 || n_scans > fls::kMaxBatch || !stride_ok(stride)) return FLS_ERR_INVALID_ARG;
    if (!batch_method(h->cfg.method)) return FLS_ERR_UNSUPPORTED;
    // scans of one batch are matched against the same map state: only meaningful when Match does not modify the map
    if (n_scans > 1 && !h->cfg.localization_mode) return FLS_ERR_UNSUPPORTED;
    FLS_TRY
    if (st) std::memset(st, 0, sizeof(*st) * (size_t)n_scans);
    h->begin_call();
    const float4* ptrs[fls::kMaxBatch];
    const int rc = stage_scans(h, n_scans, planar, n, stride, ptrs);
    return rc != FLS_OK ? rc : match_batch_dispatch(h, n_scans, ptrs, n, T, converged, st);
    FLS_CATCH
}

int fls_match_batch_begin(fls_handle* hh, int n_scans, const void* const* planar, const size_t* n, size_t stride, const double* T) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !planar || !n || !T || n_scans < 1 || n_scans > fls::kMaxBatch || !stride_ok(stride)) return FLS_ERR_INVALID_ARG;
    if (h->cfg.method != FLS_P2PLANE_IVOX) return FLS_ERR_UNSUPPORTED;
    if (!h->cfg.localization_mode) return FLS_ERR_UNSUPPORTED;  // the map must not change between begin and end
    if (!h->pend_n.empty()) return FLS_ERR_INVALID_ARG;         // one batch in flight per handle
    FLS_TRY
    h->begin_call();
    const float4* ptrs[fls::kMaxBatch];
    const int rc = stage_scans(h, n_scans, planar, n, stride, ptrs);
    return rc != FLS_OK ? rc : h->enqueue_ivox_batch(n_scans, ptrs, n, T);
    FLS_CATCH
}

int fls_match_batch_begin_device(fls_handle* hh, int n_scans, const void* const* d_planar, const size_t* n, const double* T) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !d_planar || !n || !T || n_scans < 1 || n_scans > fls::kMaxBatch) return FLS_ERR_INVALID_ARG;
    if (h->cfg.method != FLS_P2PLANE_IVOX) return FLS_ERR_UNSUPPORTED;
    if (!h->cfg.localization_mode) return FLS_ERR_UNSUPPORTED;
    if (!h->pend_n.empty()) return FLS_ERR_INVALID_ARG;
    FLS_TRY
    h->begin_call();
    const float4* ptrs[fls::kMaxBatch];
    const int rc = device_scans(n_scans, d_planar, n, ptrs);
    return rc != FLS_OK ? rc : h->enqueue_ivox_batch(n_scans, ptrs, n, T);
    FLS_CATCH
}

int fls_match_batch_end(fls_handle* hh, double* T, int* converged, fls_match_stats* st) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !T) return FLS_ERR_INVALID_ARG;
    if (h->pend_n.empty()) return FLS_ERR_INVALID_ARG;
    FLS_TRY
    if (st) std::memset(st, 0, sizeof(*st) * h->pend_n.size());
    return h->finish_ivox_batch(T, converged, st);
    FLS_CATCH
}

int fls_match_batch_device(fls_handle* hh, int n_scans, const void* const* d_planar, const size_t* n, double* T, int* converged,
                           fls_match_stats* st) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !d_planar || !n || !T || n_scans < 1 || n_scans > fls::kMaxBatch) return FLS_ERR_INVALID_ARG;
    if (!batch_method(h->cfg.method)) return FLS_ERR_UNSUPPORTED;
    if (n_scans > 1 && !h->cfg.localization_mode) return FLS_ERR_UNSUPPORTED;
    FLS_TRY
    if (st) std::memset(st, 0, sizeof(*st) * (size_t)n_scans);
    h->begin_call();
    const float4* ptrs[fls::kMaxBatch];
    const int rc = device_scans(n_scans, d_planar, n, ptrs);
    return rc != FLS_OK ? rc : match_batch_dispatch(h, n_scans, ptrs, n, T, converged, st);
    FLS_CATCH
}

int fls_fitness(fls_handle* hh, float max_range, float* score) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !score) return FLS_ERR_INVALID_ARG;
    FLS_TRY
    return h->fitness(max_range, score);
    FLS_CATCH
}

int fls_set_result_buffer_device(fls_handle* hh, double* d_results, size_t capacity_scans) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || (d_results && capacity_scans == 0)) return FLS_ERR_INVALID_ARG;
    h->result_buf = d_results;
    h->result_cap = d_results ? capacity_scans : 0;
    return FLS_OK;
}

int fls_get_iter_log(const fls_handle* hh, fls_iter_log* out, int capacity) {
    const Handle* h = reinterpret_cast<const Handle*>(hh);
    if (!h || !out || capacity < 0) return FLS_ERR_INVALID_ARG;
    const int n = h->log_n < capacity ? h->log_n : capacity;
    for (int i = 0; i < n; ++i) out[i] = h->h_log[i];
    return n;
}

int fls_set_global_map(fls_handle* hh, const void* pts, size_t n, size_t stride) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || (!pts && n) || !stride_ok(stride)) return FLS_ERR_INVALID_ARG;
    FLS_TRY
    h->begin_call();
    const int rc = h->set_global_map(pts, n, stride);
    h->end_call(nullptr);
    return rc;
    FLS_CATCH
}

int fls_update_local_map(fls_handle* hh, const double* T, int* updated, size_t* n_local) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !T) return FLS_ERR_INVALID_ARG;
    FLS_TRY
    h->begin_call();
    const int rc = h->update_local_map(T, updated, n_local);
    h->end_call(nullptr);
    return rc;
    FLS_CATCH
}

int fls_pcd_read(const char* path, float* xyzi, size_t capacity, size_t* n) {
    if (!path || !n || (capacity && !xyzi)) return FLS_ERR_INVALID_ARG;
    std::vector<float> v;
    std::string err;
    const int rc = fls::pcd_read(path, v, err);
    if (rc != FLS_OK) {
        fls::set_last_error(err);
        return rc;
    }
    *n = v.size() / 4;
    const size_t m = *n < capacity ? *n : capacity;
    if (m) std::memcpy(xyzi, v.data(), m * 16);
    return FLS_OK;
}

int fls_pcd_write(const char* path, const float* xyzi, size_t n) {
    if (!path || (!xyzi && n)) return FLS_ERR_INVALID_ARG;
    std::string err;
    const int rc = fls::pcd_write(path, xyzi, n, err);
    if (rc != FLS_OK) fls::set_last_error(err);
    return rc;
}

int fls_get_voxel_keys(fls_handle* hh, int32_t* keys_xyz, size_t capacity, size_t* n) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !n || (capacity && !keys_xyz)) return FLS_ERR_INVALID_ARG;
    if (h->cfg.method != FLS_NDT && h->cfg.method != FLS_P2PLANE_IVOX) return FLS_ERR_UNSUPPORTED;
    FLS_TRY
    FLS_CUDA(cudaSetDevice(h->cfg.device));
    std::vector<unsigned long long> packed(capacity + 1);
    const size_t m = h->cfg.method == FLS_NDT ? h->ndt.dump_keys(packed.data(), capacity, h->stream) : h->ivox.dump_keys(packed.data(), capacity, h->stream);
    for (size_t i = 0; i < m; ++i) {
        const unsigned long long k = packed[i];
        const int c[3] = {(int)((k >> 42) & 0x1fffffu), (int)((k >> 21) & 0x1fffffu), (int)(k & 0x1fffffu)};
        for (int a = 0; a < 3; ++a) keys_xyz[3 * i + a] = (c[a] & 0x100000) ? c[a] - 0x200000 : c[a];  // 21-bit two's complement
    }
    *n = h->cfg.method == FLS_NDT ? h->ndt.n_vox : h->ivox.n_vox;
    return FLS_OK;
    FLS_CATCH
}

int fls_get_map_points(fls_handle* hh, float* xyzi, size_t capacity, size_t* n) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !n || (capacity && !xyzi)) return FLS_ERR_INVALID_ARG;
    if (h->cfg.method != FLS_P2PLANE_IVOX) return FLS_ERR_UNSUPPORTED;
    FLS_TRY
    FLS_CUDA(cudaSetDevice(h->cfg.device));
    FLS_CUDA(cudaStreamSynchronize(h->stream));
    const size_t m = h->ivox.n_pts < capacity ? h->ivox.n_pts : capacity;
    if (m) FLS_CUDA(cudaMemcpy(xyzi, h->ivox.pts_all.p, m * sizeof(float4), cudaMemcpyDeviceToHost));
    *n = h->ivox.n_pts;
    return FLS_OK;
    FLS_CATCH
}

int fls_get_map_info(const fls_handle* hh, fls_map_info* out) {
    const Handle* h = reinterpret_cast<const Handle*>(hh);
    if (!h || !out) return FLS_ERR_INVALID_ARG;
    std::memset(out, 0, sizeof(*out));
    if (h->cfg.method == FLS_P2PLANE_IVOX) {
        out->n_points = (long long)h->ivox.n_pts;
        out->n_voxels = (long long)h->ivox.n_vox;
        out->table_slots = h->ivox.n_pts ? (long long)h->ivox.mask + 1 : 0;
        out->bytes = (long long)h->ivox.bytes();
        out->incremental_inserts = (long long)h->ivox.n_incremental;
        out->full_builds = (long long)h->ivox.n_full;
    } else if (h->cfg.method == FLS_NDT) {
        out->n_voxels = (long long)h->ndt.n_vox;
        out->table_slots = (long long)h->ndt.slots;
        out->bytes = (long long)h->ndt.bytes();
    } else if (h->cfg.method == FLS_ICP_P2P) {
        const fls::IvoxMap& g = h->icp_map.grid;
        out->n_points = (long long)g.n_pts;
        out->n_voxels = (long long)g.n_vox;
        out->table_slots = g.n_pts ? (long long)g.mask + 1 : 0;
        out->bytes = (long long)g.bytes();
    } else {  // kd-tree plug-ins: planar map (+ corner map for LoamFull)
        const bool full = h->cfg.method == FLS_LOAM_FULL;
        out->n_points = (long long)(h->kd_planar.n + (full ? h->kd_corner.n : 0));
        out->n_voxels = (long long)(h->kd_planar.grid.n_vox + (full ? h->kd_corner.grid.n_vox : 0));
        out->table_slots = (h->kd_planar.n ? (long long)h->kd_planar.grid.mask + 1 : 0) + (full && h->kd_corner.n ? (long long)h->kd_corner.grid.mask + 1 : 0);
        out->bytes = (long long)(h->kd_planar.grid.bytes() + h->kd_planar.cloud.bytes() + (full ? h->kd_corner.grid.bytes() + h->kd_corner.cloud.bytes() : 0));
    }
    return FLS_OK;
}

int fls_ivox_add_points(fls_handle* hh, const void* pts, size_t n, size_t stride) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || (!pts && n) || !stride_ok(stride)) return FLS_ERR_INVALID_ARG;
    if (h->cfg.method != FLS_P2PLANE_IVOX) return FLS_ERR_UNSUPPORTED;
    FLS_TRY
    h->begin_call();
    const float4* d = h->upload(pts, n, stride, h->stage);
    const int rc = h->ivox.append_and_build(d, n, h->cfg.ivox_capacity, h->stream);
    h->launches += h->ivox.launches;
    h->ivox.launches = 0;
    h->end_call(nullptr);
    return rc;
    FLS_CATCH
}

int fls_ivox_knn(fls_handle* hh, const void* queries, size_t n, size_t stride, int k, float* out_pts, int32_t* out_count) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !queries || !out_pts || !out_count || k != 5 || !stride_ok(stride)) return FLS_ERR_INVALID_ARG;
    if (h->cfg.method != FLS_P2PLANE_IVOX) return FLS_ERR_UNSUPPORTED;
    if (h->ivox.n_pts == 0) return FLS_ERR_NO_MAP;
    FLS_TRY
    h->begin_call();
    const float4* dq = h->upload(queries, n, stride, h->src);
    fls::DevBuf<float4> d_out;
    fls::DevBuf<int> d_found;
    d_out.reserve(n * 5);
    d_found.reserve(n);
    fls::launch_ivox_knn_test(h->ivox_view(), dq, (int)n, d_out.p, d_found.p, h->stream);
    FLS_CUDA(cudaMemcpyAsync(out_pts, d_out.p, n * 5 * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    FLS_CUDA(cudaMemcpyAsync(out_count, d_found.p, n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    h->end_call(nullptr);
    return FLS_OK;
    FLS_CATCH
}

int fls_voxel_grid(int device, const void* pts, size_t n, size_t stride, float leaf, float* out, size_t* n_out) {
    if ((!pts && n) || !out || !n_out || !stride_ok(stride) || !(leaf > 0.f)) return FLS_ERR_INVALID_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return FLS_ERR_NO_DEVICE;
    FLS_TRY
    FLS_CUDA(cudaSetDevice(device));
    *n_out = 0;
    if (n == 0) return FLS_OK;
    cudaStream_t st;
    FLS_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    int rc = FLS_OK;
    try {
        fls::DevBuf<unsigned char> raw;
        fls::DevBuf<float4> in, outb;
        fls::BuildScratch sc;
        in.reserve(n);
        outb.reserve(n);
        if (stride == 16) {
            FLS_CUDA(cudaMemcpyAsync(in.p, pts, n * 16, cudaMemcpyHostToDevice, st));
        } else {
            raw.reserve(n * stride);
            FLS_CUDA(cudaMemcpyAsync(raw.p, pts, n * stride, cudaMemcpyHostToDevice, st));
            fls::launch_repack(raw.p, n, stride, in.p, st);
        }
        int l = 0;
        const size_t m = fls::voxel_grid_device(in.p, n, leaf, outb.p, sc, st, &l);
        FLS_CUDA(cudaMemcpyAsync(out, outb.p, m * 16, cudaMemcpyDeviceToHost, st));
        FLS_CUDA(cudaStreamSynchronize(st));
        *n_out = m;
    } catch (const fls::CudaError& e) {
        rc = e.status;
    }
    cudaStreamDestroy(st);
    return rc;
    FLS_CATCH
}

int fls_extract_features(const fls_feature_cfg* cfg, const float* depth, const int32_t* col, size_t n, const int32_t* row_start,
                         const int32_t* row_end, int32_t n_rows, int32_t* corner_idx, size_t* n_corner, int32_t* planar_idx, size_t* n_planar,
                         fls_match_stats* stats) {
    if (!cfg || !depth || !col || !row_start || !row_end || !corner_idx || !n_corner || !planar_idx || !n_planar || n_rows < 0)
        return FLS_ERR_INVALID_ARG;
    // the reference CHECK_NE()s both thresholds against FloatNaN (feature_extractor.cpp:19-20)
    if (!(cfg->corner_threshold < 3.0e38f) || !(cfg->planar_threshold < 3.0e38f)) return FLS_ERR_INVALID_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev) return FLS_ERR_NO_DEVICE;
    FLS_TRY
    return fls::extract_features_device(cfg->device, depth, col, n, row_start, row_end, n_rows, cfg->corner_threshold, cfg->planar_threshold,
                                        corner_idx, n_corner, planar_idx, n_planar, stats);
    FLS_CATCH
}

}  // extern "C"
