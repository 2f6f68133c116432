/*
 * fls_b200.h — C ABI of the B200-native (sm_100a) scan-matching frontend.
 *
 * Drop-in boundary for funny_lidar_slam's registration plug-in interface.  Every entry point is what
 * a thin `RegistrationInterface` adapter (funny_lidar_slam_b200/shim/b200_registration.h, see
 * INTEGRATION.md) binds; citations are relative to the reference tree (zm0612/funny_lidar_slam):
 *
 *   fls_create / fls_destroy   <- plug-in constructors selected by mode string in
 *                                 FrontEnd::InitMatcher (src/slam/frontend.cpp:30-88) and
 *                                 Localization::InitMatcher (src/slam/localization.cpp:43-92)
 *   fls_add_cloud              <- RegistrationInterface::AddCloudToLocalMap
 *                                 (include/registration/registration_interface.h:17)
 *   fls_match                  <- RegistrationInterface::Match (registration_interface.h:13)
 *   fls_fitness                <- RegistrationInterface::GetFitnessScore (registration_interface.h:19)
 *   fls_extract_features       <- loam::FeatureExtractor::ExtractFeatures
 *                                 (include/loam/feature_extractor.h:22, src/loam/feature_extractor.cpp:35-44)
 *   fls_project / _imu         <- loam::PointcloudProjector::Project (src/loam/pointcloud_projector.cpp:32-133)
 *   fls_preprocess             <- PreProcessing::Run range gate + LidarDistortionCorrector::ProcessPoint + jump span + VoxelGrid
 *                                 (src/slam/preprocessing.cpp:181-225, src/lidar/lidar_distortion_corrector.cpp:37-64)
 *   fls_voxel_grid             <- VoxelGridCloud (include/common/pointcloud_utility.h:216-224,263-271)
 *
 * Conventions
 *   * Points are read from caller memory as {float x, y, z, <pad>, intensity ...} records `stride_bytes`
 *     apart: stride 32 with intensity at byte offset 16 is pcl::PointXYZI (the reference's cloud type,
 *     include/common/data_type.h:29-30); stride 16 is packed {x, y, z, intensity}.  Use FLS_LAYOUT_*.
 *   * Poses are Eigen `Mat4d` memory: 16 doubles, COLUMN-major (include/common/data_type.h:55).
 *   * All functions return 0 on success or a negative fls_status; nothing aborts, nothing throws
 *     (the reference's only runtime failure signal is `Match` returning false, frontend.cpp:208-210).
 *   * A handle is used from one thread at a time (the reference calls every plug-in method from the
 *     single frontend / localization thread: src/slam/system.cpp:52-53,68-69).  Each handle owns one CUDA
 *     stream; fls_match is synchronous with respect to the caller.
 */
#ifndef FLS_B200_H
#define FLS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FLS_ABI_VERSION 1

typedef struct fls_handle fls_handle;

typedef enum {
    FLS_OK = 0,
    FLS_ERR_INVALID_ARG = -1,   /* null pointer, bad stride, sentinel ("NaN") parameter left unset */
    FLS_ERR_CUDA = -2,          /* a CUDA runtime call failed; fls_last_error() has the text */
    FLS_ERR_NO_DEVICE = -3,     /* no sm_100 device visible — the product has NO CPU fallback */
    FLS_ERR_UNSUPPORTED = -4,   /* method / mode not implemented by this build */
    FLS_ERR_NO_MAP = -5,        /* Match before AddCloudToLocalMap (reference: CHECK(!grids_.empty())) */
    FLS_ERR_CAPACITY = -6,      /* voxel count would exceed the LRU capacity (eviction not emulated on device) */
    FLS_ERR_TOO_FEW_POINTS = -7 /* reference: CHECK_GT(ordered_cloud_.size(), 10u) icp_optimized.h:55 */
} fls_status;

/* Mode strings of include/common/constant_variable.h:21-25, in the same order as SURVEY.md §8b. */
typedef enum {
    FLS_ICP_P2P = 0,      /* kIcpOptimized       -> IcpOptimized<double>          */
    FLS_NDT = 1,          /* kIncrementalNDT     -> IncrementalNDT                */
    FLS_P2PLANE_IVOX = 2, /* kPointToPlane_IVOX  -> LoamPointToPlaneIVOX<double>  */
    FLS_P2PLANE_KNN = 3,  /* kPointToPlane_KdTree-> LoamPointToPlaneKdtree<double>*/
    FLS_LOAM_FULL = 4     /* kLoamFull_KdTree    -> LoamFull<double>              */
} fls_method;

/* IVoxMap::NearbyType (include/ivox_map/ivox_map.h:24-29) */
typedef enum { FLS_NEARBY_CENTER = 0, FLS_NEARBY6 = 1, FLS_NEARBY18 = 2, FLS_NEARBY26 = 3 } fls_nearby;

/* point record layouts accepted by every `stride_bytes` argument */
#define FLS_LAYOUT_PCL_XYZI 32u /* pcl::PointXYZI: x,y,z,pad | intensity,pad,pad,pad */
#define FLS_LAYOUT_PACKED 16u   /* x,y,z,intensity */

/* All constructor arguments of the five plug-ins (same names as the reference's ctor parameters). */
typedef struct {
    int32_t method;            /* fls_method */
    int32_t device;            /* CUDA device ordinal */
    int32_t localization_mode; /* is_localization_mode: Match never modifies the map */
    int32_t max_iterations;    /* opti_iter_num / max_iterations / max_iteration */
    double position_converge_thres;
    double rotation_converge_thres;

    /* LoamPointToPlaneIVOX / LoamPointToPlaneKdtree / LoamFull (loam_point_to_plane_ivox.h:36-58) */
    double point_to_planar_thres;
    float ivox_resolution;    /* 0.5  (loam_point_to_plane_ivox.h:55) */
    int32_t ivox_nearby;      /* FLS_NEARBY18 (:56) */
    int64_t ivox_capacity;    /* 1000000 voxels (ivox_map.h:35) */
    float ivox_max_range;     /* 5.0 (ivox_map.h:58) */
    int32_t ivox_k;           /* 5 (ivox_map.h:57) */

    /* IncrementalNDT (incremental_ndt.h:22-26) */
    double ndt_voxel_size;
    double ndt_outlier_thres;
    int32_t ndt_min_points_in_voxel;
    int32_t ndt_max_points_in_voxel;
    int32_t ndt_min_effective_pts;
    int32_t ndt_capacity;

    /* IcpOptimized (icp_optimized.h:24-27) */
    double icp_max_correspond_distance;
    double rot_thre_add_cloud;
    double dist_thre_add_cloud;
    int32_t local_map_size;

    /* shared down-sampling leafs */
    float source_cloud_filter_size; /* ICP / NDT: VoxelGridCloud at the top of Match */
    float map_cloud_filter_size;    /* ICP / kd-tree maps */

    /* LoamFull (loam_full_kdtree.h:33-44) */
    double point_search_thres;
    double line_ratio_thres;
    float corner_map_filter_size;
    int32_t corner_local_map_size;

    uint32_t flags; /* FLS_FLAG_* */
    uint32_t reserved[7];
} fls_config;

#define FLS_FLAG_ITER_LOG 1u /* keep per-iteration H, g, dx, n_valid, sum_res for fls_get_iter_log */
#define FLS_FLAG_PROFILE 2u  /* bracket every residual-kernel launch with CUDA events (fills kernel_ms / kernel_launches) */

typedef struct {
    int32_t iterations;   /* GN iterations executed */
    int32_t converged;    /* the bool Match returns */
    int64_t n_source;     /* points entering the GN loop (after Match's own VoxelGridCloud where the plug-in has one) */
    int64_t n_valid;      /* number_valid_planar_ / effective_num of the last executed iteration */
    double sum_residual;  /* overall_res_planar_ / total_res of the last executed iteration */
    float gpu_ms;         /* device time of this call's kernels (CUDA events on the handle's stream) */
    int32_t gpu_launches; /* kernels of this library launched by the call */
    int64_t h2d_bytes;    /* bytes copied host->device by the call */
    int64_t d2h_bytes;    /* bytes copied device->host by the call */
    float kernel_ms;      /* FLS_FLAG_PROFILE: summed device time of the residual kernel over the executed iterations */
    int32_t kernel_launches; /* FLS_FLAG_PROFILE: how many launches kernel_ms covers (= iterations) */
    int64_t algo_bytes;   /* FLS_FLAG_PROFILE: algorithmic bytes those launches moved (DESIGN.md "roofline accounting") */
} fls_match_stats;  /* valid only when the call returned FLS_OK */

typedef struct {
    double H[36]; /* row-major 6x6 (symmetric) */
    double g[6];
    double dx[6];
    double sum_residual;
    int64_t n_valid;
} fls_iter_log;

typedef struct {
    int64_t n_points;    /* map points resident on the device */
    int64_t n_voxels;    /* occupied voxels (iVox / NDT) or grid cells (ICP) */
    int64_t table_slots; /* open-addressing table size */
    int64_t bytes;       /* device bytes held by the map */
    int64_t incremental_inserts; /* LOAM-iVox mapping mode: inserts that only rewrote the touched voxels and the centres around them */
    int64_t full_builds;         /* ... and inserts (incl. the first) that rebuilt table + stencil lists from all points */
} fls_map_info;

/* Fill `cfg` with the parameter set the reference ships for `method` (config YAMLs; SURVEY.md App. B). */
int fls_config_default(fls_config* cfg, int method);

int fls_create(const fls_config* cfg, fls_handle** out);
void fls_destroy(fls_handle* h);

/* AddCloudToLocalMap.  `n_clouds` is the initializer_list arity (1, or 2 = {planar, corner} for LoamFull).
 * Clouds are in the map frame. */
int fls_add_cloud(fls_handle* h, int n_clouds, const void* const* pts, const size_t* n, size_t stride_bytes);

/* Match.  Pass the PointcloudCluster members the plug-in reads (include/lidar/pointcloud_cluster.h:13-26):
 * ordered_cloud_ (ICP, NDT), planar_cloud_ (P2PLANE_*), corner_cloud_ + planar_cloud_ (LOAM_FULL); unused
 * ones may be NULL/0.  T is in-out and written even when *converged == 0 (icp_optimized.h:152,
 * incremental_ndt.h:307,334, loam_point_to_plane_ivox.h:198). */
int fls_match(fls_handle* h, const void* ordered, size_t n_ordered, const void* planar, size_t n_planar, const void* corner, size_t n_corner,
              size_t stride_bytes, double T_colmajor[16], int* converged, fls_match_stats* stats);

/* Same as fls_match but the scan is already resident in device memory as packed float4 {x,y,z,i}
 * (the `value` leg of bench.py).  `d_points` is a device pointer on the handle's device.  The LOAM plug-ins keep the pointer for a
 * later fls_fitness (the source cloud of the last Match, as upstream keeps source_cloud_ptr_): the buffer must stay valid and
 * unchanged until the next Match on the handle, or fls_fitness must not be called.  `stats` (here and in every Match entry) is
 * meaningful only when the call returns FLS_OK. */
int fls_match_device(fls_handle* h, const void* d_points, size_t n, double T_colmajor[16], int* converged, fls_match_stats* stats);

/* GetFitnessScore(max_range): FLT_MAX when unsupported / no inliers, as upstream.  After a batch (fls_match_batch*) it scores scan 0
 * of the batch at its final pose, with the same cloud its single Match would leave. */
int fls_fitness(fls_handle* h, float max_range, float* score);

/* Batched Match for throughput (the benchmark entry SURVEY.md §8b names): `n_scans` (<= 64) independent scans, each with its
 * own in-out pose T[s*16 .. s*16+15], converged[s] and stats[s], matched against the same map in ONE persistent launch.
 * Implemented for FLS_P2PLANE_IVOX (one persistent work-queue kernel for the batch), and for FLS_NDT, FLS_ICP_P2P and
 * FLS_P2PLANE_KNN (one cooperative launch, a sub-grid and a Gauss-Newton loop per scan); FLS_LOAM_FULL returns
 * FLS_ERR_UNSUPPORTED (its Match inserts key frames even in localization mode, and it needs corner clouds).  More than one scan
 * requires localization_mode (Match must not modify the map); a batch of one is exactly fls_match, in either mode.
 * The entry reads the planar clouds for FLS_P2PLANE_IVOX and FLS_P2PLANE_KNN, the ordered clouds for FLS_NDT and FLS_ICP_P2P.
 * An FLS_ICP_P2P batch with a scan of <= 10 points is refused as a whole (FLS_ERR_TOO_FEW_POINTS) before anything runs.
 * Call-level figures (gpu_ms, gpu_launches, byte counts, kernel_ms) are reported in stats[0]; per-scan fields everywhere.
 * Results are identical to n_scans separate fls_match calls.  The _device variant takes device pointers to packed float4 scans. */
int fls_match_batch(fls_handle* h, int n_scans, const void* const* planar, const size_t* n, size_t stride_bytes, double* T_colmajor,
                    int* converged, fls_match_stats* stats);
/* fls_match_batch in two halves, so that a caller with two handles overlaps the host->device copy of one batch with the kernels of
 * the other: _begin enqueues the copies, the matching and the read-back on the handle's stream and returns without waiting (the
 * host buffers — pinned, to be asynchronous — and `n` must stay valid until _end); _end waits and fills T / converged / stats like
 * fls_match_batch.  FLS_P2PLANE_IVOX in localization mode; one batch in flight per handle. */
int fls_match_batch_begin(fls_handle* h, int n_scans, const void* const* planar, const size_t* n, size_t stride_bytes, const double* T_colmajor);
int fls_match_batch_begin_device(fls_handle* h, int n_scans, const void* const* d_planar, const size_t* n, const double* T_colmajor);
int fls_match_batch_end(fls_handle* h, double* T_colmajor, int* converged, fls_match_stats* stats);
int fls_match_batch_device(fls_handle* h, int n_scans, const void* const* d_planar, const size_t* n, double* T_colmajor, int* converged,
                           fls_match_stats* stats);

/* Device-side results for a consumer that lives on the GPU (the per-batch NCCL all-gather of poses, SURVEY.md §8e): once set,
 * every Match additionally writes, for scan s of the call, 18 doubles at d_results + 18*s — the column-major Mat4d pose
 * (what T receives), converged (0/1), iterations — from inside the Gauss-Newton kernel when the scan stops; the buffer is
 * complete when the Match call returns.  `capacity_scans` bounds s; NULL unsets.  The buffer is owned by the caller and must
 * stay valid until unset or the handle is destroyed. */
int fls_set_result_buffer_device(fls_handle* h, double* d_results, size_t capacity_scans);

/* per-iteration log of the last fls_match (needs FLS_FLAG_ITER_LOG; batch: scan 0); returns the number of entries written */
int fls_get_iter_log(const fls_handle* h, fls_iter_log* out, int capacity);

int fls_get_map_info(const fls_handle* h, fls_map_info* out);
/* Keys (x, y, z voxel coordinates, int32 triples) of the voxels the map currently holds, in no particular order: FLS_NDT
 * (IncrementalNDT::grids_, incremental_ndt.h:393) and FLS_P2PLANE_IVOX (IVoxMap::grids_map_, ivox_map.h:70).  Introspection for the
 * LRU parity tests; writes at most `capacity` triples and returns the voxel count in *n. */
int fls_get_voxel_keys(fls_handle* h, int32_t* keys_xyz, size_t capacity, size_t* n);
/* The points the FLS_P2PLANE_IVOX map holds (packed x, y, z, intensity), in insertion order; at most `capacity` points are written, the
 * count is returned in *n.  Introspection for the map parity tests. */
int fls_get_map_points(fls_handle* h, float* xyzi, size_t capacity, size_t* n);

/* Test hook: IVoxMap::GetClosestPoint for a batch of map-frame queries (packed float4 host arrays).
 * out_pts receives n*k packed points (unused slots zero), out_count the number found per query. */
/* IVoxMap::AddPoints (include/ivox_map/ivox_map.h:44, src/ivox_map/ivox_map.cpp:122-143): the points enter the FLS_P2PLANE_IVOX map as
 * they are (map frame, no insertion rule), in order, with upstream's LRU policy at `ivox_capacity`.  The map of a handle in
 * localization mode is otherwise replaced by fls_add_cloud; this entry appends. */
int fls_ivox_add_points(fls_handle* h, const void* pts, size_t n, size_t stride_bytes);
int fls_ivox_knn(fls_handle* h, const void* queries, size_t n, size_t stride_bytes, int k, float* out_pts, int32_t* out_count);

/* VoxelGridCloud on the device: `out` must hold n packed float4 records; *n_out receives the count. */
int fls_voxel_grid(int device, const void* pts, size_t n, size_t stride_bytes, float leaf, float* out, size_t* n_out);

/* LOAM feature extraction on the projector's arrays (PointcloudCluster::point_depth_vec_, point_col_index_vec_,
 * row_start_index_vec_, row_end_index_vec_).  corner_idx / planar_idx receive indices into the ordered cloud in
 * the reference's emission order; capacities: corner >= 120*V, planar >= n + 6*V. */
typedef struct {
    float corner_threshold;
    float planar_threshold;
    int32_t device;
    int32_t reserved;
} fls_feature_cfg;
int fls_extract_features(const fls_feature_cfg* cfg, const float* depth, const int32_t* col, size_t n, const int32_t* row_start,
                         const int32_t* row_end, int32_t n_rows, int32_t* corner_idx, size_t* n_corner, int32_t* planar_idx, size_t* n_planar,
                         fls_match_stats* stats);

/* PointcloudProjector::Project (src/loam/pointcloud_projector.cpp:32-133): raw cloud + ring per point (firing order) ->
 * ordered_cloud_ (packed float4, capacity n_rows*n_cols), point_depth_vec_ / point_col_index_vec_ (n_rows*n_cols entries, the
 * first *n_ordered meaningful), row_start_index_vec_ / row_end_index_vec_ (n_rows).  Without an IMU buffer the de-skew of :100-103
 * is the identity; fls_project_imu below applies it. */
int fls_project(int device, const void* raw, const int32_t* ring, size_t n, size_t stride_bytes, int32_t n_rows, int32_t n_cols,
                float horizontal_resolution, float min_distance, float max_distance, float* ordered, float* depth, int32_t* col,
                int32_t* row_start, int32_t* row_end, size_t* n_ordered);

/* Localization mode, the map side (Localization::LoadLocalMap, src/slam/localization.cpp:364-410, and its callers :127-135, :216-224):
 * fls_set_global_map keeps the global map resident in device memory; fls_update_local_map(T) re-cuts the local map — a +-100 m
 * pcl::CropBox around the translation of T, input order kept — when there is none yet or the pose is within 50 m of one of its
 * edges, and hands it to AddCloudToLocalMap of the handle's plug-in without a host round trip.  *updated = 1 when a new local map
 * was cut (need_update_local_map_), *n_local its size (0: LoadLocalMap returned an empty cloud; the matcher's map is untouched). */
int fls_set_global_map(fls_handle* h, const void* pts, size_t n, size_t stride_bytes);
int fls_update_local_map(fls_handle* h, const double T_colmajor[16], int* updated, size_t* n_local);

/* PCD v0.7 files as pcl::io::loadPCDFile / savePCDFileBinary read and write them for x y z intensity clouds
 * (include/common/keyframe.h:24-74, src/slam/localization.cpp:283-300): fls_pcd_read fills at most `capacity` packed
 * x, y, z, intensity records (DATA ascii or binary; extra fields are skipped, a missing intensity reads 0) and returns the point
 * count of the file in *n; fls_pcd_write writes DATA binary. */
int fls_pcd_read(const char* path, float* xyzi, size_t capacity, size_t* n);
int fls_pcd_write(const char* path, const float* xyzi, size_t n);

/* IMU orientation samples around a scan — what LidarDistortionCorrector reads through its DataSearcher<IMUData>
 * (include/lidar/lidar_distortion_corrector.h:11-48, src/lidar/lidar_distortion_corrector.cpp:19-64): time stamps in microseconds
 * (ascending), unit quaternions in Eigen coefficient order x, y, z, w, the reference time of the scan (SetRefTime) and the
 * lidar -> imu extrinsic (column-major 4x4).  n_imu == 0 (or a NULL pointer to the struct): no de-skew, points pass unchanged. */
typedef struct {
    const uint64_t* imu_time_us;
    const double* imu_quat_xyzw;
    size_t n_imu;
    uint64_t ref_time_us;
    double T_lidar_to_imu[16];
} fls_imu_buffer;

/* PreProcessing::Run, the branch of the plug-ins that take no features (src/slam/preprocessing.cpp:181-225): per raw point
 * {x, y, z, intensity, time-relative-to-ref [s]} (5 floats, firing order): range gate [min_distance, max_distance], IMU de-skew
 * (a point whose time is outside the IMU buffer is dropped), ordered_cloud_ = every kept point, planar_cloud_ = the kept points
 * whose RAW index is a multiple of jump_span, then pcl::VoxelGrid(planar_leaf).  Outputs: packed x, y, z, intensity records,
 * each buffer with room for n points.  When ref_time_us is outside the IMU buffer upstream skips the scan: both counts are 0. */
int fls_preprocess(int device, const float* raw_xyzit, size_t n, const fls_imu_buffer* imu, float min_distance, float max_distance,
                   int32_t jump_span, float planar_leaf, float* ordered, size_t* n_ordered, float* planar, size_t* n_planar);

/* fls_project with the per-point de-skew of pointcloud_projector.cpp:100-103: `time` holds the time of every raw point relative to
 * ref_time_us [s].  A point whose time is outside the IMU buffer does not claim its cell; the depth of a cell stays the range of
 * the raw point (:57, :105). */
int fls_project_imu(int device, const void* raw, const int32_t* ring, const float* time, size_t n, size_t stride_bytes, const fls_imu_buffer* imu,
                    int32_t n_rows, int32_t n_cols, float horizontal_resolution, float min_distance, float max_distance, float* ordered,
                    float* depth, int32_t* col, int32_t* row_start, int32_t* row_end, size_t* n_ordered);

const char* fls_strerror(int status);
const char* fls_last_error(void); /* thread-local text of the last CUDA failure */
int fls_abi_version(void);
int fls_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* FLS_B200_H */
