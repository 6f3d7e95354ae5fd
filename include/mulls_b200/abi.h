/*
 * mulls_b200 C-ABI — the drop-in boundary of the MULLS registration hot path on B200.
 *
 * Every entry point below is what a reference-side binding for this path would call. The
 * reference interface each one replaces is cited as file:line relative to the MULLS tree
 * (YuePanEdward/MULLS @ b275607):
 *
 *   mulls_icp_run            <- lo::CRegistration<PointT>::mm_lls_icp
 *                               include/common/cregistration.hpp:1114-1440
 *                               (determine_corres :1701-1835, multi_metrics_lls_tran_estimation
 *                                :1869-1967, pt2pl/pt2li/pt2pt_lls_summation :1976-2275,
 *                                get_multi_metrics_lls_residual :2518-2677, the per-class PCL kd-tree
 *                                build :1209-1232, intersection_filter :2894-2922)
 *   mulls_icp_run_batch      <- the same call made for N independent scan pairs (BASELINE config 4)
 *   mulls_create_pipelined   <- (no reference counterpart: the scheduler that overlaps PCIe copies and kernels)
 *   mulls_batch_upload /
 *   mulls_batch_run_resident <- same, split so that inputs can stay resident in HBM between runs
 *   mulls_icp_run_sharded    <- the same call with the source clouds sharded over ranks
 *                               (BASELINE config 5); the per-iteration exchange is delegated to a
 *                               caller-supplied all-reduce; mulls_icp_run_sharded_nccl: the same over NCCL inside the
 *                               library (mulls_nccl_unique_id, mulls_nccl_init)
 *   mulls_nn_query           <- block1->tree_*->nearestKSearch(pt, 1, ...): the kd-trees mm_lls_icp leaves behind
 *                               (cregistration.hpp:1213-1232), read at src/map_manager.cpp:197-205
 *   mulls_scan_read / _probe <- DataIo::read_pc_cloud_block, include/common/dataio.hpp:1732-1756 (read_pcd_file :279-287,
 *                               read_bin_file :357-377); mulls_pose_write <- write_lo_pose_overwrite / _append :1896-1926
 *   mulls_pca_features       <- lo::PrincipleComponentAnalysis<PointT>::get_pc_pca_feature
 *                               include/common/pca.hpp:294-354 (+ get_pca_feature :390-434)
 *   mulls_map_update         <- lo::MapManager::update_local_map, src/map_manager.cpp:17-145
 *   mulls_classify_nground   <- lo::CFilter<PointT>::classify_nground_pts, include/common/cfilter.hpp:2058-2290
 *   mulls_icp_run_to_map     <- mm_lls_icp with block1 = the device-resident local map
 *   mulls_fast_ground_filter <- lo::CFilter<PointT>::fast_ground_filter, include/common/cfilter.hpp:1658-2036
 *   mulls_voxel_downsample   <- lo::CFilter<PointT>::voxel_downsample, include/common/cfilter.hpp:83-165
 *   mulls_extract_semantic_pts <- lo::CFilter<PointT>::extract_semantic_pts, include/common/cfilter.hpp:2295-2413
 *                               (mulls_voxel_downsample, mulls_fast_ground_filter and mulls_classify_nground also accept
 *                                device pointers for their input rows and output buffers)
 *
 * Plain C, plain pointers and sizes. No torch / Eigen / PCL types cross this boundary; the C++ shim
 * in include/common/cregistration.hpp converts Eigen/PCL objects to these PODs.
 *
 * Return convention: every function returns 0 on success or a negative MULLS_E_* code for
 * *infrastructure* errors (CUDA failure, bad argument, unsupported option). The *algorithmic* status
 * of a registration (1, -1, -2, -3 exactly as cregistration.hpp:1131-1136) is in mulls_icp_result.code.
 * There is no CPU fallback: without a CUDA device mulls_create fails with MULLS_E_CUDA.
 */
#ifndef MULLS_B200_ABI_H
#define MULLS_B200_ABI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MULLS_NUM_CLASSES 6
/* Order of the feature classes everywhere in this ABI == the index order of `used_feature_type`
 * inside mm_lls_icp (cregistration.hpp:1196-1232): ground, pillar, facade, beam, roof, vertex. */
enum {
    MULLS_GROUND = 0,
    MULLS_PILLAR = 1,
    MULLS_FACADE = 2,
    MULLS_BEAM = 3,
    MULLS_ROOF = 4,
    MULLS_VERTEX = 5
};

/* infrastructure error codes */
enum {
    MULLS_OK = 0,
    MULLS_E_CUDA = -100,        /* CUDA runtime error, see mulls_last_error */
    MULLS_E_ARG = -101,         /* invalid argument */
    MULLS_E_CAPACITY = -102,    /* more points / pairs than the context was created for */
    MULLS_E_UNSUPPORTED = -103, /* option of mm_lls_icp that this build does not implement */
    MULLS_E_COMM = -104,        /* the caller's all-reduce callback failed */
    MULLS_E_IO = -105           /* a scan / pose file could not be opened or parsed */
};

#define MULLS_MAX_TRACE_ITERS 64

/* Zero-copy view of pcl::PointCloud<pcl::PointXYZINormal>::points (utility.hpp:40):
 * 12 floats (48 bytes) per point: x y z _ | normal_x normal_y normal_z _ | intensity curvature _ _ .
 * For pillar/beam clouds normal_* holds the principal direction (pca.hpp:437-454). Host pointer. */
typedef struct mulls_cloud_view {
    const float *aos48;
    size_t n;
} mulls_cloud_view;

/* The 21 scalar/string arguments of mm_lls_icp (cregistration.hpp:1114-1123), same names, same
 * defaults (see mulls_icp_default_params), plus the target block's bounding box that the function
 * reads from registration_cons.block1->local_bound (cregistration.hpp:2916). */
typedef struct mulls_icp_params {
    int32_t max_iter_num;
    float dis_thre_unit;
    float converge_translation;
    float converge_rotation_d;
    float dis_thre_min;
    float dis_thre_update_rate;
    char used_feature_type[8]; /* "111110" + NUL; order ground,pillar,facade,beam,roof,vertex */
    char weight_strategy[8];   /* "1101" + NUL; balance,residual,distance,intensity */
    float z_xy_balanced_ratio;
    float pt2pt_residual_window;
    float pt2pl_residual_window;
    float pt2li_residual_window;
    int32_t apply_intersection_filter;
    int32_t apply_motion_undistortion_while_registration; /* sources carry the timestamp ratio in `curvature` */
    int32_t normal_shooting_on;                           /* k = 10 normal-shooting candidates for ground/facade/roof */
    float normal_bearing;
    int32_t use_more_points; /* informational: the caller already chose pc_* vs pc_*_down */
    int32_t keep_less_source_points; /* random down-sampling of :2866-2892, deterministic in random_seed */
    float sigma_thre;
    float min_neccessary_corr_ratio;
    float max_bearable_rotation_d;
    double target_bound[6]; /* block1->local_bound: min_x min_y min_z max_x max_y max_z */
    /* Seed of the random down-sampling used by keep_less_source_points. The reference seeds pcl::RandomSample
     * with time(NULL) (cfilter.hpp:620, SURVEY Q11), i.e. its result is not reproducible; here the kept subset is
     * a deterministic uniform sample: the k points with the smallest splitmix64(seed, cloud, index) keys. */
    uint32_t random_seed;
    uint32_t _pad;
} mulls_icp_params;

/* Outputs of mm_lls_icp: constraint_t::Trans1_2 / information_matrix / sigma / confidence
 * (cregistration.hpp:1405, :1418-1420) and the return code (:1439). Matrices are ROW-major. */
typedef struct mulls_icp_result {
    double T[16];
    double info[36];
    float sigma;
    float confidence;
    int32_t code;  /* 1 ok, -1 step too large, -2 too few correspondences, -3 sigma too large, 0 no iteration */
    int32_t iters; /* number of loop bodies entered (the failing / converging one included) */
    uint32_t n_corr[MULLS_NUM_CLASSES]; /* |Corr_f| per class in the last executed iteration */
    uint32_t n_src[MULLS_NUM_CLASSES];  /* source points per class left after the last executed iteration */
} mulls_icp_result;

/* Optional per-iteration trace (parity tests): what the reference would LOG(INFO) per iteration. */
typedef struct mulls_icp_trace {
    int32_t n_iter;
    int32_t _pad;
    double atpa[MULLS_MAX_TRACE_ITERS][36]; /* row-major, symmetrised as at cregistration.hpp:1924-1938 */
    double atpb[MULLS_MAX_TRACE_ITERS][6];
    double x[MULLS_MAX_TRACE_ITERS][6];
    uint32_t n_corr[MULLS_MAX_TRACE_ITERS][MULLS_NUM_CLASSES];
    uint32_t n_src[MULLS_MAX_TRACE_ITERS][MULLS_NUM_CLASSES]; /* source sizes after determine_corres */
} mulls_icp_trace;

typedef struct mulls_ctx mulls_ctx;

/* Create a context on CUDA device `device` able to hold `max_pairs` scan pairs of at most
 * `max_src_pts` source and `max_tgt_pts` target points each (sum over the six classes). */
mulls_ctx *mulls_create(int device, size_t max_pairs, size_t max_src_pts, size_t max_tgt_pts);
/* Same, with `n_lanes` independent lanes (own CUDA stream, buffers and host thread each): batch calls split their
 * pairs over the lanes, so that the H2D copy of one slice overlaps the registration of another and small kernels
 * fill each other's tails. Results are identical to a single-lane context (pairs are independent). */
mulls_ctx *mulls_create_pipelined(int device, size_t max_pairs, size_t max_src_pts, size_t max_tgt_pts, int n_lanes);
void mulls_destroy(mulls_ctx *ctx);
const char *mulls_last_error(const mulls_ctx *ctx); /* ctx may be NULL: error of the failed create */

/* Fill `p` with the default arguments of mm_lls_icp (cregistration.hpp:1115-1123). */
void mulls_icp_default_params(mulls_icp_params *p);

/* One registration: host clouds in, host result out (H2D + all iterations + D2H inside). */
int mulls_icp_run(mulls_ctx *ctx, const mulls_cloud_view tgt[MULLS_NUM_CLASSES],
                  const mulls_cloud_view src[MULLS_NUM_CLASSES], const mulls_icp_params *params,
                  const double init_guess[16] /* row-major 4x4 */, mulls_icp_result *out,
                  mulls_icp_trace *trace /* may be NULL */);

/* n_pairs independent registrations in one call. tgt/src are [n_pairs][6]. */
int mulls_icp_run_batch(mulls_ctx *ctx, size_t n_pairs, const mulls_cloud_view *tgt,
                        const mulls_cloud_view *src, const mulls_icp_params *params /* [n_pairs] */,
                        const double *init_guess /* [n_pairs][16] */, mulls_icp_result *out /* [n_pairs] */,
                        mulls_icp_trace *trace /* [n_pairs] or NULL */);

/* Split form: copy the inputs to HBM once, then run the whole path (ingest: filter, spatial sort,
 * grid build; all iterations; posterior) any number of times from the resident copies. */
int mulls_batch_upload(mulls_ctx *ctx, size_t n_pairs, const mulls_cloud_view *tgt,
                       const mulls_cloud_view *src, const mulls_icp_params *params,
                       const double *init_guess);
int mulls_batch_run_resident(mulls_ctx *ctx, mulls_icp_result *out /* [n_pairs] or NULL */,
                             mulls_icp_trace *trace /* [n_pairs] or NULL */);

/* Statistics of the last run on this context (for bench.py). */
typedef struct mulls_run_stats {
    uint64_t kernel_launches;   /* kernels of this library launched by the last run */
    uint64_t algorithmic_bytes; /* sum over pairs and executed iterations of 28*(N_s,active + N_t) */
    uint64_t iterations;        /* sum over pairs of executed iterations */
    uint64_t search_launches;   /* launches of the search kernel (one per ICP iteration of the batch) */
    float ms_ingest;            /* device time of the ingest phase (CUDA events) */
    float ms_iterate;           /* device time of the iteration kernels */
    float ms_search;            /* device time of the fused transform+NN+claim kernel only */
    float ms_total;
    float ms_search_iter[MULLS_MAX_TRACE_ITERS]; /* per-iteration device time of the search kernel */
    /* one-shot calls with host buffers (mulls_icp_run_batch): where the call's wall time went */
    float ms_host_pack; /* host: repacking the clouds into the pinned staging (0 when they are shipped as rows) */
    float ms_h2d;       /* device: first cloud copy enqueued -> last cloud copy done */
    float ms_host_call; /* host: wall time of the whole call */
    float ms_host_upload; /* host: wall time of the upload part (tables, packing, enqueueing the copies) */
} mulls_run_stats;
int mulls_get_stats(const mulls_ctx *ctx, mulls_run_stats *out);

/* Source-sharded single registration (BASELINE config 5): every rank holds the full target and a
 * contiguous slice of every source class starting at global index src_index_base[c]. The caller
 * supplies the all-reduce used once (sum, doubles) or twice (+ min, int32 claim table) per
 * iteration on device buffers; with NCCL: ncclAllReduce(buf, buf, count, type, op, comm, stream). */
typedef int (*mulls_allreduce_fn)(void *user, void *device_buf, size_t count,
                                  int dtype /* 0 = float64, 1 = int32 */, int op /* 0 = sum, 1 = min */,
                                  void *cuda_stream);
int mulls_icp_run_sharded(mulls_ctx *ctx, const mulls_cloud_view tgt[MULLS_NUM_CLASSES],
                          const mulls_cloud_view src_shard[MULLS_NUM_CLASSES],
                          const uint32_t src_index_base[MULLS_NUM_CLASSES],
                          const uint32_t src_global_n[MULLS_NUM_CLASSES],
                          const mulls_icp_params *params, const double init_guess[16],
                          mulls_allreduce_fn allreduce, void *user, mulls_icp_result *out,
                          mulls_icp_trace *trace);

/* The same over NCCL, entirely inside the library (no callback, nothing interpreted in the loop): the three
 * exchanges of an iteration are ncclAllReduce calls enqueued on the context's stream between its kernels.
 * libnccl.so.2 is resolved at run time with dlopen (inside a PyTorch process: the NCCL PyTorch has loaded), so the
 * library has no link-time dependency on NCCL.
 *   mulls_nccl_unique_id   rank 0 creates an id (ncclGetUniqueId) and ships the 128 bytes to the other ranks by any
 *                          means (MPI, a file, torch.distributed.broadcast)
 *   mulls_nccl_init        collective: ncclCommInitRank on the context's device; the communicator belongs to the
 *                          context and is destroyed with it
 *   mulls_icp_run_sharded_nccl   `comm` = an ncclComm_t of the SAME libnccl (e.g. one the application already has
 *                          for these ranks), or NULL for the context's own (mulls_nccl_init) */
#define MULLS_NCCL_ID_BYTES 128
int mulls_nccl_unique_id(char id[MULLS_NCCL_ID_BYTES]);
int mulls_nccl_init(mulls_ctx *ctx, int rank, int world, const char id[MULLS_NCCL_ID_BYTES]);
int mulls_icp_run_sharded_nccl(mulls_ctx *ctx, void *comm /* ncclComm_t or NULL */,
                               const mulls_cloud_view tgt[MULLS_NUM_CLASSES],
                               const mulls_cloud_view src_shard[MULLS_NUM_CLASSES],
                               const uint32_t src_index_base[MULLS_NUM_CLASSES],
                               const uint32_t src_global_n[MULLS_NUM_CLASSES], const mulls_icp_params *params,
                               const double init_guess[16], mulls_icp_result *out, mulls_icp_trace *trace);

/* Stand-in for block1->tree_* (cregistration.hpp:1213-1232): mm_lls_icp leaves a kd-tree per target class in
 * registration_cons.block1, and MapManager::map_scan_feature_pts_distance_removal (src/map_manager.cpp:221-258, called
 * from :197-205) runs nearestKSearch(point, 1, ...) on them. Here the last mulls_icp_run / mulls_icp_run_batch (pair 0)
 * on `ctx` leaves its sorted target slices and their grid in HBM, and this call answers the same query on them:
 * for every query point the exact nearest target of class `cls` (FLANN float distance, ties to the lower index)
 * within the radius the registration searched (2.5 * dis_thre_unit, which covers dynamic_dist_thre_max of
 * map_manager.h:28). idx[i] = index of that target in the caller's ORIGINAL class cloud (the reference's index is
 * into its bbox-filtered private clone), d2[i] = squared distance; nothing within the radius: idx -1, d2 +inf.
 * Targets removed by the intersection filter are not candidates (as in the reference: the trees are built after
 * the filter, :1186-1232). Returns MULLS_E_ARG if no registration has run on the context since its last upload. */
int mulls_nn_query(mulls_ctx *ctx, int cls, const float *xyz /* [n][3], host */, size_t n, int32_t *idx /* [n] */,
                   float *d2 /* [n] */);

/* PCA neighbourhood features (pca.hpp:294-354): for every `stride`-th point of `cloud` take the
 * at most `k` nearest neighbours within `radius` (the point itself included), and return
 * eigenvalues (descending), principal direction, normal direction, and the neighbour count.
 * k <= 0 or k > 1024 is treated as 1024 (the reference uses 25..50). */
typedef struct mulls_pca_out {
    float *eigenvalues; /* [n][3] lambda1 >= lambda2 >= lambda3 (pcl::PCA convention) */
    float *principal;   /* [n][3] unit principal direction (eigenvector of lambda1) */
    float *normal;      /* [n][3] unit normal direction (col0 x col1, pcl::PCA convention) */
    int32_t *pt_num;    /* [n] neighbours used (0 for points skipped by the stride) */
} mulls_pca_out;
int mulls_pca_features(mulls_ctx *ctx, mulls_cloud_view cloud, float radius, int k, int stride,
                       mulls_pca_out *out);

/* ---- Device-resident local map (SURVEY §8(f) rank 1) -------------------------------------------------------
 * lo::MapManager::update_local_map, src/map_manager.cpp:17-145 (+ map_based_dynamic_close_removal :149-217,
 * map_scan_feature_pts_distance_removal :221-258; cloudblock_t::append_feature / transform_feature
 * utility.hpp:438-470, :495-516; CFilter::dist_filter cfilter.hpp:838-873; random_downsample_pcl :606-628;
 * get_cloud_bbx utility.hpp:817-847). The six target clouds of the scan-to-map registration stay in HBM between
 * frames: per frame only the new scan's down-sampled feature clouds cross PCIe, and mulls_icp_run_to_map reads the
 * target straight from the map. */
typedef struct mulls_map mulls_map;

/* Arguments of update_local_map (include/pgo/map_manager.h:22-32), same names and defaults. */
typedef struct mulls_map_params {
    float local_map_radius;              /* 80 */
    int32_t max_num_pts;                 /* 20000 */
    int32_t kept_vertex_num;             /* 800 */
    float last_frame_reliable_radius;    /* 60; accepted and unused, as in the reference body */
    int32_t map_based_dynamic_removal_on; /* 0; needs the preceding mulls_icp_run_to_map on the same context: the
                                            reference queries the kd-trees that registration left in block1 */
    char used_feature_type[8];           /* "111110" */
    float dynamic_removal_center_radius; /* 30 */
    float dynamic_dist_thre_min;         /* 0.3 */
    float dynamic_dist_thre_max;         /* 3.0 */
    float near_dist_thre;                /* 0.03 */
    int32_t recalculate_feature_on;      /* 0; 1: update_cloud_vectors (:95-115, :260-295) on the map's pillars and beams */
    uint32_t random_seed;                /* seed of the budgeted down-sampling (pcl::RandomSample in the reference) */
} mulls_map_params;

typedef struct mulls_map_info {
    double pose_lo[16];     /* local_map->pose_lo after the update (= the scan's pose), row-major */
    double local_bound[6];  /* local_map->local_bound: min_x min_y min_z max_x max_y max_z (map frame) */
    double bound[6];        /* local_map->bound (world frame, points transformed by pose_lo) */
    uint32_t n[MULLS_NUM_CLASSES];          /* points per class after the update */
    uint32_t n_appended[MULLS_NUM_CLASSES]; /* scan points appended per class (after dynamic removal) */
    int32_t feature_point_num;              /* ground + pillar + facade + beam + roof */
    float ms_update;                        /* device time of the update (CUDA events) */
} mulls_map_info;

void mulls_map_default_params(mulls_map_params *p);
/* A map whose six class clouds hold at most `max_pts_per_class` points each (map + appended scan). */
mulls_map *mulls_map_create(mulls_ctx *ctx, size_t max_pts_per_class);
void mulls_map_destroy(mulls_map *map);
/* Replace the content of the map by host clouds (e.g. a map built elsewhere) and set its pose. */
int mulls_map_set(mulls_map *map, const mulls_cloud_view cls[MULLS_NUM_CLASSES], const double pose_lo[16]);
/* update_local_map(local_map, last_target_cblock, ...): `scan_down` are last_target_cblock->pc_*_down (index 5:
 * pc_vertex), `scan_pose_lo` its pose_lo. The scan block itself is not modified (the reference leaves its down
 * clouds transformed into the old map frame and thinned by the dynamic removal). */
int mulls_map_update(mulls_map *map, const mulls_cloud_view scan_down[MULLS_NUM_CLASSES], const double scan_pose_lo[16],
                     const mulls_map_params *params, mulls_map_info *info /* may be NULL */);
int mulls_map_get_info(const mulls_map *map, mulls_map_info *info);
/* Copy class `cls` of the map to the host (48-byte rows); *n receives the point count, `cap` is the room in rows. */
int mulls_map_download(mulls_map *map, int cls, float *out_aos48, size_t cap, size_t *n);
/* mm_lls_icp with block1 = the resident map: the target views and block1->local_bound come from the map
 * (params->target_bound is ignored), only the source clouds are copied to the device. */
int mulls_icp_run_to_map(mulls_ctx *ctx, mulls_map *map, const mulls_cloud_view src[MULLS_NUM_CLASSES],
                         const mulls_icp_params *params, const double init_guess[16], mulls_icp_result *out,
                         mulls_icp_trace *trace /* may be NULL */);

/* ---- Non-ground feature classification (SURVEY §8(f) rank 2) -------------------------------------------------
 * lo::CFilter<PointT>::classify_nground_pts, include/common/cfilter.hpp:2058-2290: PCA of every pca_down_rate-th point
 * (pca.hpp:294-354, a16), linearity / planarity / direction thresholds -> pillar, beam, facade, roof (:2103-2166),
 * vertex-neighbourhood promotion (:2169-2210), keypoints with the neighbourhood-category descriptor
 * (encode_stable_points, :1071-1181), non-maximum suppression (non_max_suppress, :1243-1312) and the fixed-number
 * down-sampling (random_downsample_pcl :606-628, xy_normal_balanced_downsample :551-602). */
enum {
    MULLS_OUT_PILLAR = 0,
    MULLS_OUT_BEAM = 1,
    MULLS_OUT_FACADE = 2,
    MULLS_OUT_ROOF = 3,
    MULLS_OUT_PILLAR_DOWN = 4,
    MULLS_OUT_BEAM_DOWN = 5,
    MULLS_OUT_FACADE_DOWN = 6,
    MULLS_OUT_ROOF_DOWN = 7,
    MULLS_OUT_VERTEX = 8,   /* the keypoints this call appends to cloud_vertex */
    MULLS_OUT_UNGROUND = 9, /* cloud_in as the call leaves it (sampled, normals assigned) */
    MULLS_OUT_COUNT = 10
};

/* Arguments of classify_nground_pts (cfilter.hpp:2070-2081), same names; defaults where the reference has them,
 * otherwise the values extract_semantic_pts / test/mulls_slam.cpp pass by default. */
typedef struct mulls_classify_params {
    float neighbor_searching_radius;      /* 1.0 */
    int32_t neighbor_k;                   /* 50; 1..64 */
    int32_t neigh_k_min;                  /* 8 */
    int32_t pca_down_rate;                /* 1 */
    float edge_thre;                      /* 0.65 */
    float planar_thre;                    /* 0.65 */
    float edge_thre_down;                 /* 0.75 */
    float planar_thre_down;               /* 0.75 */
    int32_t extract_vertex_points_method; /* 2 */
    float curvature_thre;                 /* 0.12 */
    float vertex_curvature_non_max_radius; /* 1.5 * radius; unused by the reference body */
    float linear_vertical_sin_high_thre;  /* 0.94 */
    float linear_vertical_sin_low_thre;   /* 0.17 */
    float planar_vertical_sin_high_thre;  /* 0.98 */
    float planar_vertical_sin_low_thre;   /* 0.34 */
    int32_t fixed_num_downsampling;       /* 0 */
    int32_t pillar_down_fixed_num;        /* 200 */
    int32_t facade_down_fixed_num;        /* 800 */
    int32_t beam_down_fixed_num;          /* 200 */
    int32_t roof_down_fixed_num;          /* 100 */
    int32_t unground_down_fixed_num;      /* 20000 */
    float beam_height_max;                /* FLT_MAX */
    float roof_height_min;                /* -FLT_MAX */
    float feature_pts_ratio_guess;        /* 0.3 */
    int32_t sharpen_with_nms;             /* 1 */
    int32_t use_distance_adaptive_pca;    /* 0; 1 is not implemented: MULLS_E_UNSUPPORTED */
    uint32_t random_seed;                 /* seed of every random_downsample_pcl inside */
} mulls_classify_params;

typedef struct mulls_classify_out {
    float *rows[MULLS_OUT_COUNT]; /* caller buffers of `cap` 48-byte rows each (NULL: not wanted) */
    size_t cap;                   /* cloud_in.n rows are always enough */
    size_t n[MULLS_OUT_COUNT];    /* rows written */
} mulls_classify_out;

void mulls_classify_default_params(mulls_classify_params *p);
int mulls_classify_nground(mulls_ctx *ctx, mulls_cloud_view cloud_in, const mulls_classify_params *params,
                           mulls_classify_out *out);

/* ---- Ground segmentation (SURVEY §8(f) rank 2, first half) ---------------------------------------------------
 * lo::CFilter<PointT>::fast_ground_filter, include/common/cfilter.hpp:1658-2036: 2-D grid over the cloud, lowest point
 * per cell and per 3x3 neighbourhood, two height thresholds -> ground / non-ground, rate-based down-sampling by the
 * position inside the cell, and (estimate_ground_normal_method 3, the default) a RANSAC plane per ground cell
 * (estimate_ground_normal_by_ransac :2038-2054 -> CProceesing::plane_seg_ransac cprocessing.hpp:67-105 ->
 * pcl::SACSegmentation, SACMODEL_PLANE / SAC_RANSAC, optimize coefficients; PCL 1.10 semantics restated). The first
 * stage of extract_semantic_pts (:2355-2361); its `cloud_unground` is the input of mulls_classify_nground. */
typedef struct mulls_ground_params { /* argument names of :1658-1672; defaults = extract_semantic_pts / mulls_slam gflags */
    int32_t min_grid_pt_num;                     /* 10  (gf_grid_min_pt_num) */
    float grid_resolution;                       /* 3.0 (gf_grid_size) */
    float max_height_difference;                 /* 0.3 (gf_in_grid_h_thre) */
    float neighbor_height_diff;                  /* 1.5 (gf_neigh_grid_h_thre) */
    float max_ground_height;                     /* 5.0 (gf_max_h) */
    int32_t ground_random_down_rate;             /* 15  (gf_ground_down_rate) */
    int32_t ground_random_down_down_rate;        /* 2   (gf_down_down_rate) */
    int32_t nonground_random_down_rate;          /* 3   (gf_nonground_down_rate) */
    int32_t reliable_neighbor_grid_num_thre;     /* 0 */
    int32_t estimate_ground_normal_method;       /* 3; 0 = (0,0,1), 3 = RANSAC per cell; 1 and 2: MULLS_E_UNSUPPORTED */
    float normal_estimation_radius;              /* 2.0; only read by method 1 */
    int32_t distance_weight_downsampling_method; /* 2 (dist_inverse_sampling_method): 0 off, 1 linear, 2 quadratic */
    float standard_distance;                     /* 15.0 (unit_dist) */
    int32_t fixed_num_downsampling;              /* 0 */
    int32_t down_ground_fixed_num;               /* 300 (ground_down_fixed_num) */
    float intensity_thre;                        /* FLT_MAX */
    int32_t apply_grid_wise_outlier_filter;      /* 0 (extract_semantic_pts passes apply_scanner_filter here, :2361) */
    float outlier_std_scale;                     /* 3.0 */
    uint32_t random_seed; /* seed of random_downsample_pcl (fixed_num_downsampling); pcl::RandomSample is time-seeded */
} mulls_ground_params;

typedef struct mulls_ground_out {
    float *ground;      /* cloud_ground: caller buffers of `cap` 48-byte rows each (NULL: not wanted) */
    float *ground_down; /* cloud_ground_down */
    float *unground;    /* cloud_unground; row[3] = approximate height above ground (:1752, :1880, :1894) */
    size_t cap;         /* cloud_in.n rows are always enough */
    size_t n_ground, n_ground_down, n_unground;
} mulls_ground_out;

void mulls_ground_default_params(mulls_ground_params *p);
int mulls_fast_ground_filter(mulls_ctx *ctx, mulls_cloud_view cloud_in, const mulls_ground_params *params,
                             mulls_ground_out *out);

/* lo::CFilter<PointT>::voxel_downsample, include/common/cfilter.hpp:83-165: one point per occupied voxel, in voxel-index
 * order (voxel_size < 0.001 copies the cloud, :89-97). `out` receives at most cloud_in.n rows. The reference's
 * std::sort leaves open WHICH point of a voxel survives; here it is the one with the lowest index. */
int mulls_voxel_downsample(mulls_ctx *ctx, mulls_cloud_view cloud_in, float voxel_size, float *out, size_t cap, size_t *n_out);

/* lo::CFilter<PointT>::extract_semantic_pts, include/common/cfilter.hpp:2295-2413, the per-frame feature extraction:
 * voxel_downsample(pc_raw -> pc_down) (:2346), fast_ground_filter(pc_down) (:2355-2361), classify_nground_pts(pc_unground)
 * (:2378-2391) — chained in HBM: only the raw scan goes up and the feature clouds come down. Not produced: pc_sketch
 * (:2348), the scanner / semantic-mask pre-filters (:2328-2342) and update_parameters_self_adaptive (:2406-2410). */
typedef struct mulls_extract_params {
    float vf_downsample_resolution; /* cloud_down_res */
    mulls_ground_params ground;     /* the gf_* arguments */
    mulls_classify_params classify; /* the pca_* / *_thre / *_fixed_num arguments */
} mulls_extract_params;

typedef struct mulls_extract_out {
    float *pc_down;        /* in_block->pc_down; caller buffers of `cap` 48-byte rows (NULL: not wanted) */
    float *pc_ground;      /* in_block->pc_ground */
    float *pc_ground_down; /* in_block->pc_ground_down */
    size_t cap;            /* pc_raw.n rows are always enough */
    size_t n_down, n_ground, n_ground_down;
    mulls_classify_out cls; /* pc_pillar .. pc_roof_down, pc_vertex, pc_unground (MULLS_OUT_*) */
} mulls_extract_out;

int mulls_extract_semantic_pts(mulls_ctx *ctx, mulls_cloud_view pc_raw, const mulls_extract_params *params,
                               mulls_extract_out *out);

/* The wire format the library ships host clouds in when the "host_pack" tunable is on (csrc/host_pack.h): the 28 of the
 * 48 bytes of a pcl::PointXYZINormal row (utility.hpp:40) that the path reads, repacked on the host cores into pinned
 * staging before the DMA. format 1: [n x (x y z intensity)] [n x (nx ny nz)]; format 2 (motion undistortion, which also
 * reads `curvature`): [n x (x y z intensity)] [n x (nx ny nz curvature)]. `out` (16-byte aligned) receives
 * 4n + 3n floats (format 1) or 8n floats (format 2). Exposed for callers that keep their clouds packed, and for tests. */
int mulls_pack_rows(const float *aos48, size_t n, int format, float *out);

/* Scans in, poses out — the reference's DataIo on the two sides of the hot path (SURVEY 8f rank 3; csrc/scan_io.h, host
 * code only). A scan is read straight into pcl::PointXYZINormal rows (48 bytes), i.e. into the buffer every registration
 * and front-end entry point above takes; with mulls_host_alloc that buffer is pinned and crosses PCIe as it is.
 *   mulls_scan_probe   rows the file holds (KITTI .bin: one more than its records — the reference's read loop appends a
 *                      default point at end-of-file, include/common/dataio.hpp:366-373)
 *   mulls_scan_read    DataIo::read_pc_cloud_block (dataio.hpp:1732-1756) over read_pcd_file (:279-287; PCD v0.7, DATA
 *                      ascii | binary, float32 fields x y z intensity normal_x normal_y normal_z curvature, others are
 *                      ignored; binary_compressed: MULLS_E_UNSUPPORTED) and read_bin_file (:357-377; by the .bin
 *                      extension); local_bound (may be NULL) = CloudUtility::get_cloud_bbx (utility.hpp:817-848);
 *                      normalize_intensity != 0: intensity rescaled to 0..255 in float (:1738-1750)
 *   mulls_pose_write   DataIo::write_lo_pose_overwrite / write_lo_pose_append (dataio.hpp:1896-1926): the upper 3 x 4 of a
 *                      row-major 4 x 4 pose, setprecision(8), one line
 *   mulls_host_alloc / mulls_host_free   pinned host memory (cudaHostAlloc); NULL without a CUDA device */
int mulls_scan_probe(const char *path, size_t *n_points);
int mulls_scan_read(const char *path, float *rows48, size_t capacity_points, size_t *n_points, double local_bound[6],
                    int normalize_intensity);
int mulls_pose_write(const char *path, const double pose[16], int overwrite);
void *mulls_host_alloc(size_t bytes);
void mulls_host_free(void *p);

/* Runtime tunables (integers). A pipelined context passes them to its lanes, a context to the twin it double-buffers
 * one-shot batches with.
 *   "leaf_count"    search-grid cells with at most this many points are scanned, larger ones are split (default 32)
 *   "hash_slack"    grid hash tables hold at least hash_slack x cells entries; values below 2 count as 2 (default 4)
 *   "h0_min_mm"     smallest level-0 grid cell edge in mm, > 0 (default 125)
 *   "use_graph"     1: the iteration loop runs as one CUDA graph or, for small batches, as k_icp_loop; 0: the host
 *                   launch loop, one launch per kernel (default 1)
 *   "loop_kernel"   1: small batches run the whole loop as one cooperative kernel (k_icp_loop); 0: never (default 1)
 *   "host_pack"     host clouds cross PCIe packed to 28 B/point: 0 never, 1 always, 2 when a call ships at least 2^18
 *                   points (default 2)
 *   "pack_threads"  grow the process-wide packing pool to this many workers
 * Returns MULLS_E_ARG for an unknown name or a value outside the ranges above. */
int mulls_set_tunable(mulls_ctx *ctx, const char *name, int value);

#ifdef __cplusplus
}
#endif
#endif /* MULLS_B200_ABI_H */
