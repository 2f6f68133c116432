// fls_kernels.h — launch interfaces of the residual kernels (K1 p2plane/iVox, K2 NDT, K3 ICP, K5 kd-tree LOAM) and GetFitnessScore.
#pragma once
#include "fls_common.cuh"
#include "fls_gn.cuh"
#include "fls_ivox.cuh"
#include "fls_maps.h"

namespace fls {

static constexpr int kP2PlaneBlock = 768;  // default shape of the persistent LOAM-iVox kernel: one 24-warp CTA per SM (fls_p2plane.cu)
static constexpr int kNdtBlock = 512;  // few CTA rows for the folder: a dense scan fills the device with ~150-300 CTAs instead of > 1000
static constexpr int kIcpBlock = 512;   // 64 queries x 8 lanes per CTA: few rows for the folder
static constexpr int kLoamBlock = 256;

static constexpr int kMaxBatch = 64;  // scans per fls_match_batch call

struct PoseArg {
    double R[9];  // row-major
    double t[3];
};

// One scan of a batch (device-resident descriptor read by the persistent LoamPointToPlaneIVOX kernel)
struct P2PlaneScan {
    const float4* src;  // body-frame scan in Morton order of the query voxel, packed float4
    int n;
    unsigned tag_base;         // Match epoch << 8 (hand-over tags, fls_gn.cuh)
    GnState* state;
    float4* rec0;  // persistent per-point record: J0..J3
    float4* rec1;  //                              J4, J5, |d|, 1
    unsigned char* flags;
    uint4* rows;     // [grid][32] LL records {lo, tag, hi, tag}: one per CTA and sum
    uint4* ll_pose;  // [kLlPoseLen] LL records: next pose + stop word, published by the folding CTA
    fls_iter_log* log;
    double* result;  // optional packed result (kResultLen doubles), written by the folder when the scan stops
    uint4* grows;    // v9: [16][32] LL records: group rows of the two-level fold
};

// whole-loop arguments of the persistent LoamPointToPlaneIVOX kernel (K1 + fused K6); one launch = a batch of scans
struct P2PlaneLoopArgs {
    IvoxView map;
    double plane_thres;
    GnParams gp;
    int log_cap;
    const P2PlaneScan* scans;  // [n_scans]; every CTA serves every scan, CTA (s mod grid) folds and solves scan s
    int n_scans;
    int visit_group;  // scans per visit (1..8): a warp works through its chunk of each of them between two CTA barriers
    unsigned* tickets;  // v9: chunk ticket counters [n_scans][ticket_stride], zeroed before the launch
    int ticket_stride;  // >= max_iterations + 2
    unsigned* abort_word;  // v9 watchdog: zeroed before the launch, non-zero when a wait loop gave up (protocol error)
};
int p2plane_block();                   // threads per CTA of the selected kernel shape
int p2plane_max_grid(int device);      // co-resident CTAs
int p2plane_chunks(int n);             // warp-sized (32-point) work chunks
int p2plane_grid(int n, int device);    // CTAs that serve a scan of n points: its chunks / warps per CTA, + the folder, <= co-resident
void launch_p2plane_loop(const P2PlaneLoopArgs& a, int grid, cudaStream_t st);
// generation 9 of the same loop (fls_p2plane_v9.cu): barrier-free dataflow, TMA-staged candidate runs, DMMA sums
int p2plane_v9_grid(int n_max, int device);
void launch_p2plane_v9(const P2PlaneLoopArgs& a, int grid, cudaStream_t st);
// d_scan_ptrs[n_scans]: device pointers of the scans; d_offsets[n_scans + 1]: their positions in the batch; d_poses / d_states[n_scans]
void prepare_queries(const float4* const* d_scan_ptrs, int n_total, const int* d_offsets, int n_scans, const PoseArg* d_poses, GnState* d_states,
                     const IvoxView& map, unsigned char* d_flags, float4* d_sorted, BuildScratch& sc, cudaStream_t st, int* launches);
// LOAM-iVox Match-internal AddCloudToLocalMap: classify + compact the points that enter the map (d_world, d_out: n records)
size_t select_ivox_inserts(const IvoxView& map, const float4* d_src, int n, const double* R_prev, const double* t_prev, const double* R_fin,
                           const double* t_fin, double filter, float4* d_world, float4* d_out, BuildScratch& sc, cudaStream_t st, int* launches);
void launch_ivox_knn_test(const IvoxView& map, const float4* d_q, int n, float4* d_out, int* d_found, cudaStream_t st);

struct NdtArgs {
    const float4* __restrict__ src;  // voxel-filtered scan, body frame
    int n;
    NdtView map;
    double outlier_thres;
    GnState* state;
};
int ndt_grid(int n, int device);  // co-resident grid of the persistent kernel
void launch_ndt_loop(const NdtArgs& a, const GnLoopCtl& ctl, int grid, cudaStream_t st);
// batch of scans in one launch: scan s is served by CTAs [cta0, cta0 + ncta) of the grid (its own persistent loop)
using NdtBatchItem = GnBatchItem<NdtArgs>;
int ndt_max_grid(int device);  // co-resident CTAs of the batch kernel
void launch_ndt_batch(const NdtBatchItem* d_items, int n_scans, int grid, cudaStream_t st);

struct IcpArgs {
    const float4* __restrict__ src;  // voxel-filtered scan, body frame
    int n;
    IvoxView map;  // floor-keyed search grid over the voxel-filtered local map
    double max_corr;
    GnState* state;
};
int icp_grid_blocks(int n, int device);
void launch_icp_loop(const IcpArgs& a, const GnLoopCtl& ctl, int grid, cudaStream_t st);
static constexpr int kIcpPerBlock = kIcpBlock / 8;  // queries per CTA (8 lanes share one)
using IcpBatchItem = GnBatchItem<IcpArgs>;
int icp_max_grid(int device);  // co-resident CTAs of the batch kernel
void launch_icp_batch(const IcpBatchItem* d_items, int n_scans, int grid, cudaStream_t st);

// K5 — kd-tree LOAM plug-ins (LoamPointToPlaneKdtree, LoamFull): exact unbounded 5-NN over a uniform grid
struct LoamGrid {
    const float4* __restrict__ pts;    // cell-contiguous map points
    const HashSlot* __restrict__ tab;  // floor-keyed occupied-cell table
    unsigned mask;
    float inv_cell, cell;
    unsigned n_pts;
};
struct LoamArgs {
    const float4* __restrict__ corner;  // body-frame corner features (LoamFull only)
    int n_corner;
    const float4* __restrict__ planar;  // body-frame planar features
    int n_planar;
    LoamGrid corner_map, planar_map;
    double plane_thres;    // point_to_planar_thres
    double search_thres;   // point_search_thres on the 5th squared distance (+inf: none)
    double line_ratio;     // line_ratio_thres
    float gate;            // search_thres as the search's stop bound
    GnState* state;
    double* __restrict__ rec;  // [n_corner + n_planar][8] persistent {J[6], residual, -}
    unsigned char* __restrict__ flags;
};
int loam_grid_blocks(int n, int device);
void launch_loam_loop(const LoamArgs& a, const GnLoopCtl& ctl, int grid, cudaStream_t st);
static constexpr int kLoamPerBlock = kLoamBlock / 8;  // queries per CTA (8 lanes share one)
using LoamBatchItem = GnBatchItem<LoamArgs>;
int loam_max_grid(int device);  // co-resident CTAs of the batch kernel
// clears the flags of all `n_flags` points of the batch (once per Match [quirk 1]), then runs the batch in one launch
void launch_loam_batch(const LoamBatchItem* d_items, int n_scans, int grid, unsigned char* flags, int n_flags, cudaStream_t st);

// d_out2[0] = sum of squared NN distances <= max_range, d_out2[1] = how many; T column-major (cast to float inside)
void launch_fitness(const IvoxView& g, const float4* d_src, int n, const double* T_colmajor, float max_range, double* d_out2, cudaStream_t st);

}  // namespace fls
