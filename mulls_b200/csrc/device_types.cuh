// Device-side data model of the B200 registration path (see DESIGN.md "Data layout in HBM").
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/mulls_b200/abi.h"
#include "search_core.cuh" // HashEntry, GridView

namespace mulls {

constexpr int kNumClasses = MULLS_NUM_CLASSES;
constexpr int kNumSegs = 2 * kNumClasses; // seg = side*6 + class; side 0 = target, 1 = source
constexpr int kIterBlock = 128;           // threads (= source points) per iteration-kernel block
constexpr int kIngestBlock = 256;         // input points per ingest block
constexpr int kTerms = 28;                // 21 lower-tri ATPA + 6 ATPb (+1 pad) per class partial
constexpr int kDedupMinSrc = 500;         // K_filter_distant_point (cregistration.hpp:1704)
constexpr unsigned kClaimFree = 0x7f7f7f7fu;
constexpr int kIterFlags = 256;           // per-iteration stop flags kept for the launch loop of sharded runs

enum PairStatus : int { kRunning = 0, kNeedPosterior = 1, kDone = 2 };

// Work descriptor of one block: which pair / segment (or class) and the first local point index.
struct ChunkDesc {
    uint32_t pair;
    uint32_t seg;
    uint32_t first;
};

// Immutable per-pair description, written by the host at upload time.
struct PairConst {
    // arguments of mm_lls_icp (cregistration.hpp:1114-1123) in device-friendly form
    int max_iter;
    int used[kNumClasses];
    int w_balance, w_residual, w_dist, w_intensity; // weight_strategy[0..3]
    float z_xy_ratio;
    float win_pt2pt, win_pt2pl, win_pt2li;
    float thre_unit, thre_min, thre_rate;
    float conv_t, conv_r;       // converge_translation, converge_rotation (rad, float as :1163)
    float max_t, max_r;         // max_bearable_translation / rotation (float as :1162,:1164)
    float min_ratio;            // min_neccessary_corr_ratio
    int apply_filter;
    // motion undistortion at iteration 0 (cregistration.hpp:1248-1258, cfilter.hpp:496-516): slerp(I, q, s) * p + s * t
    int undistort, ud_linear, ud_neg;
    double ud_q[4];  // quaternion (x y z w) of the inverse initial guess
    double ud_t[3];  // its translation
    double ud_theta, ud_sin_theta;
    int normal_shooting;    // normal_shooting_on: k = 10 candidates for ground / facade / roof (:1730-1739)
    int keep_less;          // keep_less_source_pts (cregistration.hpp:1191-1193, :2866-2892)
    uint32_t random_seed;
    double cos_thre;            // cos(normal_bearing/180*pi), :1818
    double sigma_thre;          // :2524
    double init[16];            // initial guess, row-major
    double tbound[6];           // block1->local_bound
    // layout
    uint32_t in_off[kNumSegs];  // offset (points) of each input cloud in the AoS48 staging array
    const float4 *in_ptr[kNumSegs]; // where the ingest kernel reads the cloud: the HBM copy, or (one-shot calls with
                                    // pinned host buffers) the caller's buffer itself, streamed over PCIe (zero-copy)
    uint32_t in_n[kNumSegs];
    uint32_t in_fmt[kNumSegs];  // layout behind in_ptr: 0 = 48-byte rows, 1 = packed 16+12 B, 2 = packed 16+16 B (host_pack.h)
    uint32_t tgt_base[kNumClasses]; // base of each class in the target SoA arrays (capacity = in_n)
    uint32_t src_base[kNumClasses]; // base of each class in the source SoA arrays
    uint32_t chunk_begin;            // iteration chunks of this pair: [chunk_begin, chunk_end)
    uint32_t chunk_end;
    uint32_t class_chunk_begin[kNumClasses + 1];
    // source sharding (mulls_icp_run_sharded): global index base and global size of each source class
    uint32_t src_index_base[kNumClasses];
    uint32_t src_global_n[kNumClasses];
    int sharded;
};

// Mutable per-pair state, lives in HBM for the whole run; updated by the last block of each phase.
struct PairState {
    double T_total[16]; // accumulated initial_guess (cregistration.hpp:1400,:1403)
    double T_inc[16];   // TempTran to be applied at the start of the next iteration (:1260)
    double x[6];
    double cofactor[36];
    double info[36];
    double sigma2;
    double ibb[6];      // intersection bounding box (utility.hpp:858-866)
    float thre;         // dis_thre_* (all six evolve identically, :1155-1160, :1855-1866)
    float confidence;
    float origin[3];    // grid origin
    float h0, inv_h0;
    int n_levels;
    int status, code, iter, iters_entered, final_buf;
    int source_feature_points_count;
    int n_src[kNumClasses];   // live source points of each class on THIS rank
    int n_src_g[kNumClasses]; // ... over all ranks (== n_src unless the source is sharded)
    int n_src_g_next[kNumClasses];
    int n_tgt[kNumClasses];
    uint32_t n_corr[kNumClasses];      // |Corr_f| of the current iteration (atomics in k_resolve)
    uint32_t n_corr_last[kNumClasses]; // same, frozen for the result
    uint32_t seg_count[kNumSegs];      // valid points per segment after the intersection filter
    uint32_t seg_start[kNumSegs];      // start of the segment in the sorted order
    uint32_t hash_entries[kNumClasses]; // cells (all levels) of each target class
    uint32_t hash_base[kNumClasses];    // table of each class inside the hash pool
    uint32_t hash_mask[kNumClasses];    // capacity-1 (power of two, load factor <= 0.5)
    int bb_src[6];                     // ordered-int encoded bbox of source ground/pillar/facade
    int bb_tgt[6];                     // ordered-int encoded bbox of all target points
    uint64_t alg_bytes;                // 28*(N_s,active + N_t) summed over executed iterations
    // random down-sampling (keep_less_source_points): radix select of the k-th smallest sampling key per cloud
    int kl_keep[kNumSegs];             // -1: cloud untouched, else the number of points to keep
    uint32_t kl_rank[kNumSegs];
    uint64_t kl_prefix[kNumSegs];
    uint32_t kl_hist[kNumSegs][256];
};

// Per-run control block in device memory: what a kernel that was recorded into a CUDA graph (fixed arguments, grids
// sized for the context's capacity) needs to know about THIS run, and the iteration counter of the device-side loop.
struct LoopCtl {
    int it;          // iteration index of the graph's WHILE loop (the host loop passes its own)
    int n_it_chunks; // iteration chunks of this upload (blocks beyond it return at once)
    int n_pairs;
    int trace_on;    // write the per-iteration trace
    int max_iter;    // max over the pairs of max_iter_num
    unsigned solved; // pairs whose k_solve block has finished this iteration
    // Work lists of the iteration kernels. live_chunks[it & 1] holds the ids of the chunks that still own live sources
    // (built after the ingest for iteration 0, by k_solve for the next iteration); the kernels run a fixed number of
    // resident blocks that fetch list positions from work[] — no block is launched for a chunk that has nothing to do.
    unsigned n_live[2];
    unsigned work[4]; // fetch counters: 0 k_search, 1 k_resolve, 2 k_accumulate, 3 k_search_shoot
};

// All device pointers of a context, passed by value to the kernels.
struct DeviceArrays {
    const float4 *in_aos;   // input clouds, 3 float4 per point (pcl::PointXYZINormal)
    float4 *stg_pos;        // staging (input order): x y z intensity  (source: initial guess applied)
    float4 *stg_nrm;        // staging: nx ny nz orig_index(bits)
    uint64_t *keys_a, *keys_b;
    uint32_t *vals_a, *vals_b;
    float4 *tgt_pos, *tgt_nrm;       // target SoA, Morton-sorted inside each (pair,class) slice
    float4 *src_pos[2], *src_nrm[2]; // source SoA ping-pong
    int *src_prevj[2];               // previous NN target (seeds the next search with a real candidate)
    float4 *src_cert[2];             // where the source stood at its last full search (xyz) and the radius inside which
                                     // its match is the only target (w; 0: no certificate) — k_search keeps matches with it
    int *nn_idx;                     // per source: matched target (index inside its class slice) or -1
    float *nn_d2;
    uint8_t *flags;                  // bit0 kept as source point, bit1 correspondence passes rejectors
    int *corr_j;                     // compacted: matched target of a surviving correspondence, else -1
    float *corr_w;                   // compacted: LLS weight stored back into Corr (:2114, :2256)
    unsigned *claim;                 // duplicate_check_table (:1760) as an atomicMin table of source indices
    HashEntry *hash;                 // pool; per-class tables are laid out on the device each run
    uint32_t hash_pool_entries;
    uint32_t *hash_used;             // [0] entries laid out this run, [1] overflow flag
    uint32_t *blk_kept;              // per iteration chunk: sources kept by the block
    double *partials;                // per iteration chunk: kTerms doubles
    double *post_partials;           // per iteration chunk: VTPV, n_obs
    PairConst *pc;
    PairState *ps;
    ChunkDesc *in_chunks;
    ChunkDesc *it_chunks;
    mulls_icp_trace *trace; // may be null
    int *xch_i32;           // exchange buffer of the sharded mode (counts / bbox), 32 ints
    double *xch_f64;        // exchange buffer of the sharded mode (per-class sums), 6*kTerms + 2 doubles
    LoopCtl *ctl;
    uint32_t *live_chunks;  // 2 x live_stride chunk ids (see LoopCtl)
    uint32_t live_stride;
    int *running;           // pairs still iterating (device counter)
    volatile int *h_running; // the same, mirrored into mapped pinned host memory for the launch loop
    volatile int *h_running_iter; // [it]: pairs still iterating at the END of iteration it (sharded runs: rank-deterministic stop)
};

} // namespace mulls
