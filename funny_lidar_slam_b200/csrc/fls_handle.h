// fls_handle.h — the object behind `fls_handle*`: configuration, stream, device-resident map and scan state.
#pragma once
#include <deque>
#include <memory>
#include <vector>

#include "fls_common.cuh"
#include "fls_kernels.h"
#include "fls_maps.h"

namespace fls {

struct Handle {
    fls_config cfg;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;

    // per-call accounting (fls_match_stats)
    int launches = 0;
    long long h2d_bytes = 0, d2h_bytes = 0;
    float last_gpu_ms = 0.f;

    // scan-side buffers
    DevBuf<unsigned char> raw;  // strided caller records before repacking
    DevBuf<float4> src;         // uploaded scan (packed float4)
    DevBuf<float4> src_f;       // scan after Match's own VoxelGridCloud (ICP / NDT)
    DevBuf<float4> stage;       // clouds handed to AddCloudToLocalMap
    DevBuf<float4> stage2;      // transformed / filtered intermediates
    DevBuf<float4> rec0, rec1;  // persistent per-point {J, |d|} records (LOAM plug-ins)
    DevBuf<unsigned char> flags;
    DevBuf<unsigned> tickets;   // chunk ticket counters of the LOAM-iVox kernel (dynamic work distribution)
    DevBuf<uint4> ll_rows;      // LL hand-over records of the persistent LOAM-iVox kernel: [grid][32] rows + pose record
    unsigned match_epoch = 0;   // tag prefix of those records
    unsigned char* h_batch = nullptr;  // pinned staging of the per-batch tables (poses, offsets, scan descriptors, CTA map, pointers)
    size_t h_batch_cap = 0;
    DevBuf<unsigned char> d_batch;
    DevBuf<GnState> state;
    GnState* h_state = nullptr;  // pinned
    DevBuf<fls_iter_log> log;
    std::vector<fls_iter_log> h_log;
    int log_cap = 0, log_n = 0;
    double T_final[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    cudaEvent_t prof_ev[2] = {nullptr, nullptr};  // FLS_FLAG_PROFILE: around the GN launch of a Match (kernel_ms)
    bool profile = false;
    long long per_point_iter_bytes = 0;  // fixed part of the algorithmic bytes per point-iteration (set by match_*)
    long long per_cand_bytes = 0;        // bytes per scanned map record
    BuildScratch scratch;                // voxel-grid passes of Match

    // optional caller-owned device buffer that receives {pose, converged, iterations} per scan (fls_set_result_buffer_device)
    double* result_buf = nullptr;
    size_t result_cap = 0;

    // source cloud of the last Match (for GetFitnessScore): device pointer + count
    const float4* last_src = nullptr;
    size_t last_src_n = 0;

    // maps
    IvoxMap ivox;      // LoamPointToPlaneIVOX
    NdtMap ndt;        // IncrementalNDT
    bool ndt_first_scan = true;  // flag_first_scan_ (incremental_ndt.h:394)
    // ICP and the kd-tree LOAM plug-ins (LoamPointToPlaneKdtree, LoamFull): sliding window of clouds -> VoxelGrid -> exact search grid
    struct Cloud {
        DevBuf<float4> buf;
        size_t n = 0;
    };
    struct WindowMap {
        std::deque<std::unique_ptr<Cloud>> deque;  // cloud_deque_ (icp_optimized.h:246) / planar_cloud_deque_ / corner_cloud_deque_
        DevBuf<float4> merged;                     // concatenation of the window
        DevBuf<float4> cloud;                      // what upstream builds the kd-tree on
        size_t n = 0;
        IvoxMap grid;                              // floor-keyed uniform grid over `cloud`
    };
    WindowMap icp_map;          // IcpOptimized: local_map_ptr_
    bool icp_have_last = false;  // `static last_T` of IsNeedAddCloud (icp_optimized.h:219)  [quirk 7]
    double icp_last_T[16];
    WindowMap kd_planar, kd_corner;
    bool kd_have_last = false;  // `static last_T` of IsNeedAddCloud  [quirk 7]
    double kd_last_T[16];
    DevBuf<double> rec_d;       // persistent {J[6], residual} records of the kd-tree plug-ins
    DevBuf<float4> src2;        // uploaded corner features (LoamFull)

    // GetFitnessScore support: cloud the upstream kd-tree is built on (a view of fit_cloud or of a map's own cloud) + a search grid
    // sized for max_range
    DevBuf<float4> fit_cloud;
    const float4* fit_src = nullptr;
    size_t fit_n = 0;
    unsigned long long fit_version = 0, fit_grid_version = ~0ull;
    float fit_grid_range = -1.f;
    IvoxMap fit_grid;
    DevBuf<double> fit_out;

    explicit Handle(const fls_config& c);
    ~Handle();
    void init();     // body of the constructor
    void release();  // streams, events, pinned memory
    Handle(const Handle&) = delete;
    Handle& operator=(const Handle&) = delete;

    void begin_call();
    void end_call(fls_match_stats* st);
    const float4* upload(const void* pts, size_t n, size_t stride, DevBuf<float4>& dst);
    IvoxView ivox_view() const;
    IvoxView grid_view(const IvoxMap& g) const;
    void set_fit_cloud(const float4* d, size_t n);  // copies the cloud
    void set_fit_view(const float4* d, size_t n);   // the cloud must stay in place until the next set_fit_*

    // host side of a GN launch, shared by every Match path
    unsigned next_epoch(size_t ll_records);  // reserves the LL records and returns the tag base of a new Match
    GnParams gn_params(int method, int min_effective) const;
    fls_iter_log* scan_log(int s) const { return log_cap ? log.p + (size_t)s * log_cap : nullptr; }
    double* scan_result(int s) const { return result_buf && (size_t)s < result_cap ? result_buf + (size_t)s * kResultLen : nullptr; }
    GnLoopCtl gn_ctl(int s, int method, int min_effective, unsigned tag_base, uint4* rows, uint4* pose) const;
    unsigned char* table(size_t bytes);  // pinned staging of a per-launch table of `bytes` (device copy: d_batch)
    void send_table(size_t bytes);
    // the GN launch: `launch` enqueues `n_launches` kernels, timed for kernel_ms; GetFitnessScore scores `src`
    template <class Launch>
    void gn_launch(Launch&& launch, int n_launches, const float4* src, size_t n) {
        if (profile) FLS_CUDA(cudaEventRecord(prof_ev[0], stream));
        launch();
        if (profile) FLS_CUDA(cudaEventRecord(prof_ev[1], stream));
        launches += n_launches;
        last_src = src;
        last_src_n = n;
    }
    void read_back(int B);  // enqueues the copies of the B scan states and of scan 0's iteration log
    // after end_call: poses (column-major) into T, flags into converged, per-scan stats (call-level figures on scan 0)
    void unpack(int B, const size_t* n_source, double* T, int* converged, fls_match_stats* st);
    void dump_timing(int B, size_t n0, bool v9) const;  // FLS_DEBUG_TIMING / FLS_K1_TRACE: device timeline of scan 0
    void finish_match(double* T, int* converged, fls_match_stats* st, size_t n_source);  // the single-scan GN paths

    int add_cloud(const float4* d_cloud, size_t n);
    int add_cloud_ivox(const float4* d_cloud, size_t n);
    int match_p2plane_ivox(const float4* d_src, size_t n, double* T, int* converged, fls_match_stats* st);
    // n_scans independent scans against the (static) map in ONE persistent launch; d_scans: host array of device pointers
    int match_ivox_batch(int n_scans, const float4* const* d_scans, const size_t* n, double* T, int* converged, fls_match_stats* st);
    // the same in two halves (fls_match_batch_begin / _end): enqueue without waiting, then wait + unpack
    int enqueue_ivox_batch(int n_scans, const float4* const* d_scans, const size_t* n, const double* T);
    int finish_ivox_batch(double* T, int* converged, fls_match_stats* st);
    std::vector<size_t> pend_n;  // scans of the batch in flight (empty: none)
    bool pend_v9 = false;
    unsigned* h_abort = nullptr;  // watchdog word of the last v9 launch (pinned, behind h_state; read back with the states)

    int add_cloud_ndt(const float4* d_cloud, size_t n);
    int match_ndt(const float4* d_src, size_t n, double* T, int* converged, fls_match_stats* st);
    bool filter_batch(int n_scans, const float4* const* d_scans, const size_t* n_in, size_t* off, size_t* nf);  // ICP / NDT sources
    int match_ndt_batch(int n_scans, const float4* const* d_scans, const size_t* n, double* T, int* converged, fls_match_stats* st);

    int add_cloud_icp(const float4* d_cloud, size_t n);
    int match_icp(const float4* d_src, size_t n, double* T, int* converged, fls_match_stats* st);
    int match_icp_batch(int n_scans, const float4* const* d_scans, const size_t* n, double* T, int* converged, fls_match_stats* st);

    // filter_mode 0: always VoxelGrid(leaf); 1: only once the window holds more than 5 clouds (loam_full_kdtree.h:91-99)
    int window_add(WindowMap& w, const float4* d_cloud, size_t n, size_t window, float leaf, int filter_mode, bool replace);
    int add_cloud_kd(const float4* d_planar, size_t n_planar, const float4* d_corner, size_t n_corner);
    int match_kd(const float4* d_planar, size_t n_planar, const float4* d_corner, size_t n_corner, double* T, int* converged, fls_match_stats* st);
    int match_kd_batch(int n_scans, const float4* const* d_planar, const size_t* n, double* T, int* converged, fls_match_stats* st);  // FLS_P2PLANE_KNN
    bool need_add_cloud(const double* T, double* last_T, bool* have_last) const;

    int fitness(float max_range, float* score);

    // localization-mode map path (fls_localmap.cu): resident global map, +-100 m crop around the pose when needed
    DevBuf<float4> global_map;
    size_t global_n = 0;
    DevBuf<unsigned char> crop_keep;
    double local_edge[6] = {0, 0, 0, 0, 0, 0};
    bool have_edge = false;
    int set_global_map(const void* pts, size_t n, size_t stride);
    int update_local_map(const double* T_colmajor, int* updated, size_t* n_local);
};

}  // namespace fls
