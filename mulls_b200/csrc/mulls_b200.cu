// libmulls_b200.so — host side of the C-ABI (include/mulls_b200/abi.h) and kernel launch sequence.
// CUDA runtime only: no torch, no PCL/Eigen. One context = one device, one stream.
#include <algorithm>
#include <atomic>
#include <memory>
#include <cmath>
#include <cstdio>
#include <chrono>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <dlfcn.h>
#include <mutex>

#include "device_types.cuh"
#include "host_pack.h"
#include "scan_io.h"
#include "kernels_ingest.cuh"
#include "kernels_iterate.cuh"
#include "kernels_pca.cuh"
#include "kernels_map.cuh"
#include "kernels_classify.cuh"
#include "kernels_ground.cuh"

using namespace mulls;

namespace {
std::string g_create_error;
}

// ---- NCCL without a link-time dependency: the five entry points used, resolved from libnccl.so.2 on first use ----
namespace {
struct ncclUniqueIdBytes {
    char internal[128]; // nccl.h: ncclUniqueId
};
struct NcclApi {
    typedef int (*get_id_t)(void *);
    typedef int (*init_rank_t)(void **, int, ncclUniqueIdBytes, int);
    typedef int (*all_reduce_t)(const void *, void *, size_t, int, int, void *, cudaStream_t);
    typedef int (*destroy_t)(void *);
    typedef const char *(*err_t)(int);
    get_id_t get_id = nullptr;
    init_rank_t init_rank = nullptr;
    all_reduce_t all_reduce = nullptr;
    destroy_t destroy = nullptr;
    err_t err = nullptr;
    bool ok = false;
};
NcclApi &nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return;
        api.get_id = (NcclApi::get_id_t)dlsym(h, "ncclGetUniqueId");
        api.init_rank = (NcclApi::init_rank_t)dlsym(h, "ncclCommInitRank");
        api.all_reduce = (NcclApi::all_reduce_t)dlsym(h, "ncclAllReduce");
        api.destroy = (NcclApi::destroy_t)dlsym(h, "ncclCommDestroy");
        api.err = (NcclApi::err_t)dlsym(h, "ncclGetErrorString");
        api.ok = api.get_id && api.init_rank && api.all_reduce && api.destroy;
    });
    return api;
}
// the all-reduce hook of run_impl over NCCL: user = the communicator (nccl.h: ncclInt32 = 2, ncclFloat64 = 8; ncclSum = 0, ncclMin = 3)
int nccl_allreduce_hook(void *user, void *buf, size_t count, int dtype, int op, void *stream) {
    if (count == 0) return 0;
    return nccl_api().all_reduce(buf, buf, count, dtype == 0 ? 8 : 2, op == 0 ? 0 : 3, user, (cudaStream_t)stream);
}
} // namespace


struct mulls_map;

struct mulls_ctx {
    int device = 0;
    size_t max_pairs = 0, max_src = 0, max_tgt = 0;
    size_t cap_src = 0, cap_tgt = 0, cap_in = 0, cap_it_chunks = 0, cap_in_chunks = 0;
    cudaStream_t stream = nullptr;
    DeviceArrays A{};
    void *cub_temp = nullptr;
    size_t cub_temp_bytes = 0;
    mulls_icp_result *d_results = nullptr;
    mulls_icp_result *h_results = nullptr; // pinned
    uint32_t *h_flags = nullptr;           // pinned copy of hash_used
    int *h_running = nullptr;              // mapped pinned: pairs still iterating
    std::vector<cudaEvent_t> ev_done;      // one per iteration (launch-loop flow control)
    mulls_icp_trace *d_trace = nullptr;
    std::vector<PairConst> h_pc;
    std::vector<ChunkDesc> h_in_chunks, h_it_chunks;
    size_t n_pairs = 0, n_in = 0, n_src_total = 0, n_tgt_total = 0;
    int max_iter_max = 0;
    bool uploaded = false;
    void *nccl_comm = nullptr; // ncclComm_t created by mulls_nccl_init (destroyed with the context)
    bool any_keep_less = false;
    bool grid_valid = false; // pair 0's sorted target slices and grid are those of the last registration (mulls_nn_query)
    // tunables
    int start_level0 = 5;
    int leaf_count = 32;
    // iteration loop as a CUDA graph: WHILE(pairs running) { search, resolve, accumulate, solve } + posterior, finalize,
    // collect — one launch, the loop condition is set on the device (no host polling). Built on first use, rebuilt when a
    // tunable baked into its kernel nodes changes. 0: the host launch loop (per-kernel events for the bench's roofline).
    int use_graph = 1;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graph_exec = nullptr;
    int graph_key[6] = {-1, -1, -1, -1, -1, -1}; // the tunables baked into the kernel nodes
    LoopCtl *h_ctl = nullptr;            // pinned staging of the control block
    int num_sms = 148;
    int sort_sources = 1;    // 0: sources stay in the caller's order (study switch)
    int search_blocks = 12;  // resident k_search blocks per SM (10 / 12 / 16: register budget 48 / 40 / 32; measured 4.36 / 4.31 / 4.61 ms of search per 64-pair step)
    int defer_from_iter = 3; // k_search queues the small cells of a block (one scan loop per block) from this iteration on
    int hash_slack = 4;      // table capacity >= hash_slack x cells (power of two): load factor <= 1/hash_slack
    int reseed_cells_x4 = 16; // a previous match farther than this many quarter level-0 cells is challenged by a greedy descent
    bool any_normal_shooting = false;
    bool any_undistort = false;
    int zero_copy = 0;     // opt-in: one-shot calls read pinned host clouds in place (measured slower than DMA: 20 vs 32 GB/s)
    // repack host clouds to the 28 B/point wire format on the host cores before the DMA (host_pack.h):
    // 0 never, 1 always, 2 when a call ships at least kPackMinPoints points (small calls are latency-bound: raw rows)
    int host_pack = 2;
    int poll_pause = 64;   // _mm_pause() count between two cudaEventQuery calls of the launch loop's flow control
    int stage_wc = 0;      // allocate the pinned staging write-combined (the host only streams into it)
    float4 *h_stage = nullptr; // pinned staging of the packed clouds (allocated on first use)
    size_t h_stage_slots = 0;
    float h0_min = 0.125f;
    // timing
    cudaEvent_t ev_begin = nullptr, ev_ingest = nullptr, ev_iter = nullptr, ev_end = nullptr, ev_h2d0 = nullptr;
    bool h2d_timed = false;                 // ev_h2d0 was recorded by the upload of the current one-shot call
    float up_ms_pack = 0.f, up_ms_host = 0.f; // host-side times of that upload
    std::vector<cudaEvent_t> ev_search; // 2 per iteration
    mulls_run_stats stats{};
    std::vector<void *> allocs;
    std::string err;
    // pipelined context (mulls_create_pipelined): the batch is split over independent lane contexts, each with
    // its own stream and buffers, driven by one host thread each
    std::vector<mulls_ctx *> lanes;
    // one-shot batch calls with host buffers (mulls_icp_run_batch) are double-buffered: the second half of the batch is
    // packed and copied on the twin's stream while the first half is being registered on this one
    mulls_ctx *twin = nullptr;
    int double_buffer = 1;
    int loop_kernel = 1;       // small batches: the whole iteration loop as one cooperative kernel (k_icp_loop)
    int loop_kernel_blocks = 0; // co-resident blocks of k_icp_loop on this device (0: not yet queried, -1: unavailable)
    struct Pending {                 // a run that has been enqueued and not yet finished (run_finish)
        uint64_t launches = 0;
        int n_search_ev = 0;
        bool graphed = false, hooked = false, active = false;
    } pend;
    std::vector<size_t> lane_begin; // pair range of every lane for the resident batch
    // PCA scratch
    void *pca_buf = nullptr;
    size_t pca_buf_bytes = 0;
    // classification scratch (mulls_classify_nground)
    void *cls_buf = nullptr;
    size_t cls_buf_bytes = 0;
    // ground-filter scratch (mulls_fast_ground_filter): per-point part and per-cell part
    void *gf_buf = nullptr, *gf_cell_buf = nullptr;
    size_t gf_buf_bytes = 0, gf_cell_buf_bytes = 0;
    void *vx_buf = nullptr, *ext_buf = nullptr; // voxel filter scratch; clouds handed between the stages of extract_semantic_pts
    size_t vx_buf_bytes = 0, ext_buf_bytes = 0;
    // the local map whose clouds the target slices of pair 0 currently index (set by mulls_icp_run_to_map, cleared
    // by any other upload): what block1->tree_* are to MapManager::map_based_dynamic_close_removal
    const mulls_map *tree_map = nullptr;
    uint64_t tree_epoch = 0;
};

#define CK(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess) {                                                                      \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                            \
            return MULLS_E_CUDA;                                                                      \
        }                                                                                             \
    } while (0)

template <typename T>
static cudaError_t dev_alloc(mulls_ctx *ctx, T **p, size_t n) {
    void *v = nullptr;
    cudaError_t e = cudaMalloc(&v, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) {
        ctx->allocs.push_back(v);
        *p = (T *)v;
    }
    return e;
}

static inline size_t ceil_div(size_t a, size_t b) { return (a + b - 1) / b; }
static inline double wall_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

extern "C" {

void mulls_icp_default_params(mulls_icp_params *p) {
    std::memset(p, 0, sizeof(*p));
    p->max_iter_num = 20;
    p->dis_thre_unit = 1.5f;
    p->converge_translation = 0.002f;
    p->converge_rotation_d = 0.01f;
    p->dis_thre_min = 0.4f;
    p->dis_thre_update_rate = 1.1f;
    std::strcpy(p->used_feature_type, "111110");
    std::strcpy(p->weight_strategy, "1101");
    p->z_xy_balanced_ratio = 1.0f;
    p->pt2pt_residual_window = 0.1f;
    p->pt2pl_residual_window = 0.1f;
    p->pt2li_residual_window = 0.1f;
    p->apply_intersection_filter = 1;
    p->normal_bearing = 45.0f;
    p->sigma_thre = 0.5f;
    p->min_neccessary_corr_ratio = 0.03f;
    p->max_bearable_rotation_d = 45.0f;
    const double big = 1.7976931348623157e308;
    for (int d = 0; d < 3; ++d) {
        p->target_bound[d] = -big;
        p->target_bound[3 + d] = big;
    }
}

const char *mulls_last_error(const mulls_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

void mulls_destroy(mulls_ctx *ctx) {
    if (!ctx) return;
    for (mulls_ctx *l : ctx->lanes) mulls_destroy(l);
    ctx->lanes.clear();
    if (ctx->twin) mulls_destroy(ctx->twin), ctx->twin = nullptr;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (void *p : ctx->allocs) cudaFree(p);
    if (ctx->cub_temp) cudaFree(ctx->cub_temp);
    if (ctx->pca_buf) cudaFree(ctx->pca_buf);
    if (ctx->cls_buf) cudaFree(ctx->cls_buf);
    if (ctx->gf_buf) cudaFree(ctx->gf_buf);
    if (ctx->gf_cell_buf) cudaFree(ctx->gf_cell_buf);
    if (ctx->vx_buf) cudaFree(ctx->vx_buf);
    if (ctx->ext_buf) cudaFree(ctx->ext_buf);
    if (ctx->h_results) cudaFreeHost(ctx->h_results);
    if (ctx->h_flags) cudaFreeHost(ctx->h_flags);
    if (ctx->h_running) cudaFreeHost(ctx->h_running);
    if (ctx->nccl_comm && nccl_api().ok) nccl_api().destroy(ctx->nccl_comm);
    if (ctx->h_ctl) cudaFreeHost(ctx->h_ctl);
    if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
    if (ctx->graph) cudaGraphDestroy(ctx->graph);
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    for (cudaEvent_t e : ctx->ev_done) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->ev_search) cudaEventDestroy(e);
    if (ctx->ev_begin) cudaEventDestroy(ctx->ev_begin);
    if (ctx->ev_ingest) cudaEventDestroy(ctx->ev_ingest);
    if (ctx->ev_iter) cudaEventDestroy(ctx->ev_iter);
    if (ctx->ev_end) cudaEventDestroy(ctx->ev_end);
    if (ctx->ev_h2d0) cudaEventDestroy(ctx->ev_h2d0);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

mulls_ctx *mulls_create(int device, size_t max_pairs, size_t max_src_pts, size_t max_tgt_pts) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("mulls_create: no CUDA device (") + cudaGetErrorString(e) +
                         "); mulls_b200 has no CPU fallback";
        return nullptr;
    }
    if (device < 0 || device >= ndev || max_pairs == 0) {
        g_create_error = "mulls_create: bad device index or max_pairs";
        return nullptr;
    }
    mulls_ctx *ctx = new mulls_ctx();
    ctx->device = device;
    ctx->max_pairs = max_pairs;
    ctx->max_src = max_src_pts;
    ctx->max_tgt = max_tgt_pts;
    auto fail = [&](const char *what, cudaError_t err) -> mulls_ctx * {
        g_create_error = std::string("mulls_create: ") + what + ": " + cudaGetErrorString(err);
        mulls_destroy(ctx);
        return nullptr;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("stream", e);
    const size_t cs = ctx->cap_src = max_pairs * max_src_pts;
    const size_t ct = ctx->cap_tgt = max_pairs * max_tgt_pts;
    const size_t cin = ctx->cap_in = cs + ct;
    if (cin >= (1ull << 31)) {
        g_create_error = "mulls_create: more than 2^31 points per context";
        mulls_destroy(ctx);
        return nullptr;
    }
    // every cloud adds at most one partial chunk
    ctx->cap_it_chunks = ceil_div(cs, kIterBlock) + max_pairs * (kNumClasses + 1);
    ctx->cap_in_chunks = ceil_div(cin, kIngestBlock) + max_pairs * kNumSegs;
    DeviceArrays &A = ctx->A;
    float4 *in = nullptr;
#define ALLOC(ptr, n)                                                   \
    if ((e = dev_alloc(ctx, &(ptr), (n))) != cudaSuccess) return fail(#ptr, e)
    ALLOC(in, 3 * cin);
    A.in_aos = in;
    ALLOC(A.stg_pos, cin);
    ALLOC(A.stg_nrm, cin);
    ALLOC(A.keys_a, cin);
    ALLOC(A.keys_b, cin);
    ALLOC(A.vals_a, cin);
    ALLOC(A.vals_b, cin);
    ALLOC(A.tgt_pos, ct + kScanOverrun); // (walk_scan_leaf's last group reads past a cell)
    ALLOC(A.tgt_nrm, ct);
    for (int b = 0; b < 2; ++b) {
        ALLOC(A.src_pos[b], cs);
        ALLOC(A.src_nrm[b], cs);
        ALLOC(A.src_prevj[b], cs);
        ALLOC(A.src_cert[b], cs);
    }
    ALLOC(A.nn_idx, cs);
    ALLOC(A.nn_d2, cs);
    ALLOC(A.flags, cs);
    ALLOC(A.corr_j, cs);
    ALLOC(A.corr_w, cs);
    ALLOC(A.claim, ct);
    // hash pool: every class table has a power-of-two capacity >= 2x its cells; cells are typically
    // 2-3 per target point, so 12 entries per point (192 B) leave room for the rounding.
    {
        size_t pool = 12 * ct + 64 * max_pairs * kNumClasses;
        if (pool >= (1ull << 32)) pool = (1ull << 32) - 1;
        A.hash_pool_entries = (uint32_t)pool;
        ALLOC(A.hash, pool);
    }
    ALLOC(A.hash_used, 2);
    ALLOC(A.ctl, 1);
    ALLOC(A.blk_kept, ctx->cap_it_chunks);
    ALLOC(A.partials, ctx->cap_it_chunks * kTerms);
    ALLOC(A.post_partials, ctx->cap_it_chunks * 2);
    ALLOC(A.pc, max_pairs);
    ALLOC(A.ps, max_pairs);
    ALLOC(A.in_chunks, ctx->cap_in_chunks);
    ALLOC(A.it_chunks, ctx->cap_it_chunks);
    ALLOC(A.live_chunks, 2 * ctx->cap_it_chunks);
    A.live_stride = (uint32_t)ctx->cap_it_chunks;
    {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 148;
        ctx->num_sms = sms;
    }
    ALLOC(ctx->d_results, max_pairs + ceil_div(max_pairs * sizeof(uint64_t), sizeof(mulls_icp_result)) + 1);
    ALLOC(ctx->d_trace, max_pairs);
    ALLOC(A.running, 1);
    ALLOC(A.xch_i32, 32);
    ALLOC(A.xch_f64, kNumClasses * kTerms + 8);
#undef ALLOC
    if ((e = cudaHostAlloc((void **)&ctx->h_running, (1 + kIterFlags) * sizeof(int), cudaHostAllocMapped)) != cudaSuccess)
        return fail("mapped flag", e);
    {
        int *dptr = nullptr;
        if ((e = cudaHostGetDevicePointer((void **)&dptr, ctx->h_running, 0)) != cudaSuccess) return fail("mapped flag", e);
        A.h_running = dptr;
        A.h_running_iter = dptr + 1;
    }
    ctx->ev_done.resize(MULLS_MAX_TRACE_ITERS);
    for (auto &ev : ctx->ev_done) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    A.trace = ctx->d_trace; // written only when LoopCtl::trace_on is set for the run
    if ((e = cudaMallocHost((void **)&ctx->h_results, max_pairs * (sizeof(mulls_icp_result) + sizeof(uint64_t)))) != cudaSuccess)
        return fail("pinned results", e);
    if ((e = cudaMallocHost((void **)&ctx->h_flags, 2 * sizeof(uint32_t))) != cudaSuccess) return fail("pinned flags", e);
    if ((e = cudaMallocHost((void **)&ctx->h_ctl, sizeof(LoopCtl))) != cudaSuccess) return fail("pinned control block", e);
    // radix-sort temp storage for the largest possible sort
    {
        size_t bytes = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, bytes, A.keys_a, A.keys_b, A.vals_a, A.vals_b, (int)cin, 0, 64,
                                        ctx->stream);
        ctx->cub_temp_bytes = bytes;
        if ((e = cudaMalloc(&ctx->cub_temp, std::max<size_t>(bytes, 16))) != cudaSuccess) return fail("cub temp", e);
    }
    cudaEventCreate(&ctx->ev_begin);
    cudaEventCreate(&ctx->ev_ingest);
    cudaEventCreate(&ctx->ev_iter);
    cudaEventCreate(&ctx->ev_end);
    cudaEventCreate(&ctx->ev_h2d0);
    ctx->ev_search.resize(2 * MULLS_MAX_TRACE_ITERS);
    for (auto &ev : ctx->ev_search) cudaEventCreate(&ev);
    if ((e = cudaMemsetAsync(A.ps, 0, max_pairs * sizeof(PairState), ctx->stream)) != cudaSuccess) return fail("memset", e);
    if ((e = cudaStreamSynchronize(ctx->stream)) != cudaSuccess) return fail("sync", e);
    return ctx;
}

mulls_ctx *mulls_create_pipelined(int device, size_t max_pairs, size_t max_src_pts, size_t max_tgt_pts, int n_lanes) {
    if (n_lanes <= 1) return mulls_create(device, max_pairs, max_src_pts, max_tgt_pts);
    if ((size_t)n_lanes > max_pairs) n_lanes = (int)max_pairs;
    mulls_ctx *ctx = new mulls_ctx();
    ctx->device = device;
    ctx->max_pairs = max_pairs;
    ctx->max_src = max_src_pts;
    ctx->max_tgt = max_tgt_pts;
    const size_t per_lane = (max_pairs + n_lanes - 1) / n_lanes;
    for (int l = 0; l < n_lanes; ++l) {
        mulls_ctx *c = mulls_create(device, per_lane, max_src_pts, max_tgt_pts);
        if (!c) { // g_create_error is set by the failed create
            mulls_destroy(ctx);
            return nullptr;
        }
        ctx->lanes.push_back(c);
    }
    return ctx;
}

} // extern "C"

// Run fn(lane, first_pair, n_pairs_of_lane) on every lane of a pipelined context, one host thread per lane;
// pairs are split into contiguous, near-equal ranges. Returns the first non-zero code.
template <typename F>
static int for_each_lane(mulls_ctx *ctx, size_t n_pairs, F fn) {
    const size_t L = ctx->lanes.size();
    std::vector<int> rc(L, MULLS_OK);
    std::vector<std::thread> th;
    ctx->lane_begin.assign(L + 1, 0);
    for (size_t l = 0; l <= L; ++l) ctx->lane_begin[l] = (n_pairs * l) / L;
    for (size_t l = 0; l < L; ++l) {
        const size_t b = ctx->lane_begin[l], n = ctx->lane_begin[l + 1] - b;
        if (n == 0) continue;
        th.emplace_back([&, l, b, n]() { rc[l] = fn(ctx->lanes[l], b, n); });
    }
    for (auto &t : th) t.join();
    for (size_t l = 0; l < L; ++l)
        if (rc[l] != MULLS_OK) {
            ctx->err = ctx->lanes[l]->err;
            return rc[l];
        }
    return MULLS_OK;
}

static void merge_lane_stats(mulls_ctx *ctx) {
    mulls_run_stats &S = ctx->stats;
    S = mulls_run_stats();
    for (size_t l = 0; l < ctx->lanes.size(); ++l) {
        if (ctx->lane_begin.size() > l + 1 && ctx->lane_begin[l + 1] == ctx->lane_begin[l]) continue;
        const mulls_run_stats &s = ctx->lanes[l]->stats;
        S.kernel_launches += s.kernel_launches;
        S.algorithmic_bytes += s.algorithmic_bytes;
        S.iterations += s.iterations;
        S.search_launches += s.search_launches;
        S.ms_search += s.ms_search; // summed over concurrently running lanes: not a wall time
        S.ms_ingest = std::max(S.ms_ingest, s.ms_ingest);
        S.ms_iterate = std::max(S.ms_iterate, s.ms_iterate);
        S.ms_total = std::max(S.ms_total, s.ms_total);
    }
}

extern "C" {

int mulls_set_tunable(mulls_ctx *ctx, const char *name, int value) {
    if (!ctx || !name) return MULLS_E_ARG;
    for (mulls_ctx *l : ctx->lanes) {
        const int rc = mulls_set_tunable(l, name, value);
        if (rc != MULLS_OK) return rc;
    }
    if (ctx->twin) {
        const int rc = mulls_set_tunable(ctx->twin, name, value);
        if (rc != MULLS_OK) return rc;
    }
    std::string n(name);
    if (n == "start_level") ctx->start_level0 = value;
    else if (n == "leaf_count") ctx->leaf_count = value;
    else if (n == "reseed_cells_x4") ctx->reseed_cells_x4 = value;
    else if (n == "defer_from_iter") ctx->defer_from_iter = value;
    else if (n == "search_blocks") ctx->search_blocks = value; // (kept for old scripts: the instantiations are fixed now)
    else if (n == "sort_sources") ctx->sort_sources = value;
    else if (n == "double_buffer") ctx->double_buffer = value;
    else if (n == "loop_kernel") ctx->loop_kernel = value;
    else if (n == "hash_slack") ctx->hash_slack = std::max(2, value);
    else if (n == "use_graph") ctx->use_graph = value;
    else if (n == "zero_copy") ctx->zero_copy = value;
    else if (n == "host_pack") ctx->host_pack = value;
    else if (n == "poll_pause") ctx->poll_pause = value;
    else if (n == "stage_wc") {
        if (ctx->stage_wc != value && ctx->h_stage) { // re-allocated with the new flag on the next packed upload
            cudaFreeHost(ctx->h_stage);
            ctx->h_stage = nullptr;
            ctx->h_stage_slots = 0;
        }
        ctx->stage_wc = value;
    }
    else if (n == "pack_threads") PackPool::get().ensure_workers(value);
    else if (n == "h0_min_mm") {
        if (value <= 0) return MULLS_E_ARG; // (grid_h0 doubles it until the cloud fits)
        ctx->h0_min = (float)value / 1000.0f;
    }
    else return MULLS_E_ARG;
    return MULLS_OK;
}

int mulls_pack_rows(const float *aos48, size_t n, int format, float *out) {
    if ((n > 0 && (!aos48 || !out)) || (format != kFmtPacked28 && format != kFmtPacked32) || ((uintptr_t)out % 16) != 0)
        return MULLS_E_ARG;
    pack_rows(aos48, 0, n, format, out, out + 4 * n);
    _mm_sfence();
    return MULLS_OK;
}

// ---- scans in, poses out (csrc/scan_io.h: host code, no device involved) -------------------------------------
static int io_code(int rc) {
    switch (rc) {
    case mulls_io::kOk: return MULLS_OK;
    case mulls_io::kArg: return MULLS_E_ARG;
    case mulls_io::kCapacity: return MULLS_E_CAPACITY;
    case mulls_io::kUnsupported: return MULLS_E_UNSUPPORTED;
    default: return MULLS_E_IO;
    }
}
int mulls_scan_probe(const char *path, size_t *n_points) { return io_code(mulls_io::probe_scan(path, n_points)); }
int mulls_scan_read(const char *path, float *rows48, size_t capacity_points, size_t *n_points, double local_bound[6],
                    int normalize_intensity) {
    return io_code(mulls_io::read_scan(path, rows48, capacity_points, n_points, local_bound, normalize_intensity));
}
int mulls_pose_write(const char *path, const double pose[16], int overwrite) {
    return io_code(mulls_io::append_pose(path, pose, overwrite));
}
void *mulls_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void mulls_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

int mulls_get_stats(const mulls_ctx *ctx, mulls_run_stats *out) {
    if (!ctx || !out) return MULLS_E_ARG;
    *out = ctx->stats;
    return MULLS_OK;
}

// Inverse of the initial guess (Eigen Matrix4d::inverse: cofactors / determinant), its quaternion
// (Eigen::Quaterniond(Matrix3d)) and the per-pair constants of Eigen's slerp(Identity -> q)
// (cregistration.hpp:1248, cfilter.hpp:499-502).
static void setup_undistortion(const double *m, PairConst &pc) {
    double inv[16];
    inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
    inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
    inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
    inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
    inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
    inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
    inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
    inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
    inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
    inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
    inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
    inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
    inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
    inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
    inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
    inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
    const double det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
    double T[16];
    for (int i = 0; i < 16; ++i) T[i] = inv[i] * (1.0 / det);
    double q[4]; // x y z w
    double t = T[0] + T[5] + T[10];
    if (t > 0.0) {
        t = std::sqrt(t + 1.0);
        q[3] = 0.5 * t;
        t = 0.5 / t;
        q[0] = (T[9] - T[6]) * t;
        q[1] = (T[2] - T[8]) * t;
        q[2] = (T[4] - T[1]) * t;
    } else {
        int i = 0;
        if (T[5] > T[0]) i = 1;
        if (T[10] > T[5 * i]) i = 2;
        const int j = (i + 1) % 3, k = (j + 1) % 3;
        t = std::sqrt(T[5 * i] - T[5 * j] - T[5 * k] + 1.0);
        q[i] = 0.5 * t;
        t = 0.5 / t;
        q[3] = (T[4 * k + j] - T[4 * j + k]) * t;
        q[j] = (T[4 * j + i] + T[4 * i + j]) * t;
        q[k] = (T[4 * k + i] + T[4 * i + k]) * t;
    }
    for (int i = 0; i < 4; ++i) pc.ud_q[i] = q[i];
    pc.ud_t[0] = T[3], pc.ud_t[1] = T[7], pc.ud_t[2] = T[11];
    const double one = 1.0 - 2.220446049250313e-16;
    const double d = q[3], absD = std::fabs(d);
    pc.ud_linear = (absD >= one) ? 1 : 0;
    pc.ud_neg = (d < 0) ? 1 : 0;
    pc.ud_theta = pc.ud_linear ? 0.0 : std::acos(absD);
    pc.ud_sin_theta = pc.ud_linear ? 1.0 : std::sin(pc.ud_theta);
}

// ------------------------------------------------------------------------------------------------
static int build_pair_const(mulls_ctx *ctx, const mulls_icp_params &P, const double *init, PairConst &pc) {
    if (P.max_iter_num > MULLS_MAX_TRACE_ITERS) {
        ctx->err = "max_iter_num > 64";
        return MULLS_E_ARG;
    }
    // the threshold schedule sizes the search grid (grid_levels) and bounds every search radius
    if (!(std::isfinite(P.dis_thre_unit) && P.dis_thre_unit > 0.0f) ||
        !(std::isfinite(P.dis_thre_update_rate) && P.dis_thre_update_rate > 0.0f) ||
        !(std::isfinite(P.dis_thre_min) && P.dis_thre_min >= 0.0f)) {
        ctx->err = "dis_thre_unit and dis_thre_update_rate must be finite and > 0, dis_thre_min finite and >= 0";
        return MULLS_E_ARG;
    }
    std::memset(&pc, 0, sizeof(pc));
    pc.max_iter = P.max_iter_num;
    const size_t nu = strnlen(P.used_feature_type, 8), nw = strnlen(P.weight_strategy, 8);
    for (int c = 0; c < kNumClasses; ++c) pc.used[c] = (c < (int)nu && P.used_feature_type[c] == '1') ? 1 : 0;
    pc.w_balance = (nw > 0 && P.weight_strategy[0] == '1');
    pc.w_residual = (nw > 1 && P.weight_strategy[1] == '1');
    pc.w_dist = (nw > 2 && P.weight_strategy[2] == '1');
    pc.w_intensity = (nw > 3 && P.weight_strategy[3] == '1');
    pc.z_xy_ratio = P.z_xy_balanced_ratio;
    pc.win_pt2pt = P.pt2pt_residual_window;
    pc.win_pt2pl = P.pt2pl_residual_window;
    pc.win_pt2li = P.pt2li_residual_window;
    pc.thre_unit = P.dis_thre_unit;
    pc.thre_min = P.dis_thre_min;
    pc.thre_rate = P.dis_thre_update_rate;
    pc.conv_t = P.converge_translation;
    // the float/double mix of cregistration.hpp:1162-1164
    pc.conv_r = (float)(P.converge_rotation_d / 180.0 * M_PI);
    pc.max_t = (float)(2.0 * P.dis_thre_unit);
    pc.max_r = (float)(P.max_bearable_rotation_d / 180.0 * M_PI);
    pc.min_ratio = P.min_neccessary_corr_ratio;
    // the intersection filter is skipped in the undistortion variant (cregistration.hpp:1186)
    pc.undistort = P.apply_motion_undistortion_while_registration ? 1 : 0;
    pc.apply_filter = (P.apply_intersection_filter && !pc.undistort) ? 1 : 0;
    if (pc.undistort) setup_undistortion(init, pc);
    // :1191 keep_less_source_pts is skipped in the undistortion variant
    pc.keep_less = (P.keep_less_source_points && !pc.undistort) ? 1 : 0;
    pc.random_seed = P.random_seed;
    pc.normal_shooting = P.normal_shooting_on ? 1 : 0;
    pc.cos_thre = std::cos(P.normal_bearing / 180.0 * M_PI);
    pc.sigma_thre = (double)P.sigma_thre;
    for (int i = 0; i < 16; ++i) pc.init[i] = init[i];
    for (int i = 0; i < 6; ++i) pc.tbound[i] = P.target_bound[i];
    return MULLS_OK;
}

// resident = true: the clouds are copied into HBM (mulls_batch_upload: they must survive the caller's buffers).
// resident = false (one-shot calls): clouds in PINNED host memory are not copied at all — the ingest kernel
// streams them over PCIe itself (zero-copy through the UVA alias), pageable ones are staged with cudaMemcpy.
static int upload_impl(mulls_ctx *ctx, size_t n_pairs, const mulls_cloud_view *tgt, const mulls_cloud_view *src,
                       const mulls_icp_params *params, const double *init_guess, const uint32_t *src_index_base,
                       const uint32_t *src_global_n, bool resident = true, bool tgt_on_device = false) {
    if (!ctx || !tgt || !src || !params || !init_guess || n_pairs == 0) return MULLS_E_ARG;
    ctx->tree_map = nullptr;
    ctx->grid_valid = false;
    if (n_pairs > ctx->max_pairs) {
        ctx->err = "more pairs than the context was created for";
        return MULLS_E_CAPACITY;
    }
    CK(cudaSetDevice(ctx->device));
    ctx->uploaded = false;
    const double t_up0 = wall_ms();
    ctx->h2d_timed = false;
    ctx->up_ms_pack = 0.f;
    ctx->h_pc.assign(n_pairs, PairConst());
    ctx->h_in_chunks.clear();
    ctx->h_it_chunks.clear();
    size_t in_off = 0, s_off = 0, t_off = 0;
    int max_iter_max = 0;
    bool any_keep_less = false, any_shoot = false, any_undistort = false;
    for (size_t p = 0; p < n_pairs; ++p) {
        PairConst &pc = ctx->h_pc[p];
        int rc = build_pair_const(ctx, params[p], init_guess + 16 * p, pc);
        if (rc != MULLS_OK) return rc;
        max_iter_max = std::max(max_iter_max, pc.max_iter);
        any_keep_less = any_keep_less || pc.keep_less;
        any_shoot = any_shoot || pc.normal_shooting;
        any_undistort = any_undistort || pc.undistort;
        size_t ns = 0, nt = 0;
        for (int c = 0; c < kNumClasses; ++c) {
            nt += tgt[p * kNumClasses + c].n;
            ns += src[p * kNumClasses + c].n;
        }
        if (ns > ctx->max_src || nt > ctx->max_tgt) {
            ctx->err = "pair exceeds max_src_pts / max_tgt_pts of the context";
            return MULLS_E_CAPACITY;
        }
        for (int s = 0; s < kNumSegs; ++s) {
            const mulls_cloud_view &v = (s < kNumClasses) ? tgt[p * kNumClasses + s] : src[p * kNumClasses + (s - kNumClasses)];
            if (v.n > 0 && !v.aos48) return MULLS_E_ARG;
            pc.in_off[s] = (uint32_t)in_off;
            pc.in_n[s] = (uint32_t)v.n;
            for (size_t f = 0; f < v.n; f += kIngestBlock)
                ctx->h_in_chunks.push_back(ChunkDesc{(uint32_t)p, (uint32_t)s, (uint32_t)f});
            in_off += v.n;
        }
        pc.chunk_begin = (uint32_t)ctx->h_it_chunks.size();
        for (int c = 0; c < kNumClasses; ++c) {
            pc.tgt_base[c] = (uint32_t)t_off;
            pc.src_base[c] = (uint32_t)s_off;
            t_off += tgt[p * kNumClasses + c].n;
            const size_t n = src[p * kNumClasses + c].n;
            s_off += n;
            pc.class_chunk_begin[c] = (uint32_t)ctx->h_it_chunks.size();
            // class 0 always owns at least one chunk so that the per-pair "last block" logic (status
            // codes, iteration counter) also runs for pairs without any source point
            const size_t n_eff = (c == 0 && n == 0) ? 1 : n;
            for (size_t f = 0; f < n_eff; f += kIterBlock) ctx->h_it_chunks.push_back(ChunkDesc{(uint32_t)p, (uint32_t)c, (uint32_t)f});
            pc.src_index_base[c] = src_index_base ? src_index_base[c] : 0;
            pc.src_global_n[c] = src_global_n ? src_global_n[c] : (uint32_t)n;
        }
        pc.class_chunk_begin[kNumClasses] = (uint32_t)ctx->h_it_chunks.size();
        pc.chunk_end = (uint32_t)ctx->h_it_chunks.size();
        pc.sharded = src_index_base ? 1 : 0;
    }
    if (ctx->h_in_chunks.size() > ctx->cap_in_chunks || ctx->h_it_chunks.size() > ctx->cap_it_chunks) {
        ctx->err = "internal: chunk table capacity";
        return MULLS_E_CAPACITY;
    }
    // the clouds: repacked on the host cores and copied pair by pair (host_pack), or copied as they are, or read in
    // place (zero-copy, pinned host buffers of one-shot calls)
    size_t host_points = 0;
    for (size_t p = 0; p < n_pairs; ++p)
        for (int s = 0; s < kNumSegs; ++s)
            if (!(tgt_on_device && s < kNumClasses)) host_points += ctx->h_pc[p].in_n[s];
    const size_t kPackMinPoints = 1u << 18;
    bool tables_sent = false;
    const bool pack = ctx->host_pack == 1 || (ctx->host_pack == 2 && host_points >= kPackMinPoints);
    if (pack) {
        if (!ctx->h_stage) {
            const size_t slots = 2 * ctx->cap_in + 4 * kNumSegs * ctx->max_pairs;
            CK(cudaHostAlloc((void **)&ctx->h_stage, slots * sizeof(float4),
                             ctx->stage_wc ? cudaHostAllocWriteCombined : cudaHostAllocDefault));
            ctx->h_stage_slots = slots;
        }
        CK(cudaStreamSynchronize(ctx->stream)); // the staging may still be read by a copy of a call that failed half-way
        PackPool &pool = PackPool::get();
        pool.ensure_workers(0);
        std::unique_ptr<std::atomic<int>[]> pending(new std::atomic<int>[n_pairs]);
        std::vector<size_t> slot_begin(n_pairs + 1, 0);
        std::vector<PackJob> jobs;
        const size_t kJobPts = 16384; // multiple of 4 (pack_rows)
        size_t slot = 0;
        for (size_t p = 0; p < n_pairs; ++p) {
            PairConst &pc = ctx->h_pc[p];
            const int fmt = pc.undistort ? kFmtPacked32 : kFmtPacked28;
            slot_begin[p] = slot;
            int n_jobs = 0;
            for (int s = 0; s < kNumSegs; ++s) {
                const mulls_cloud_view &v = (s < kNumClasses) ? tgt[p * kNumClasses + s] : src[p * kNumClasses + (s - kNumClasses)];
                pc.in_ptr[s] = ctx->A.in_aos + slot;
                pc.in_fmt[s] = (uint32_t)fmt;
                if (tgt_on_device && s < kNumClasses) { // the view already points into HBM (device-resident local map)
                    pc.in_ptr[s] = (const float4 *)v.aos48;
                    pc.in_fmt[s] = kFmtRows48;
                    continue;
                }
                if (v.n == 0) continue;
                float *pos = reinterpret_cast<float *>(ctx->h_stage + slot);
                float *nrm = reinterpret_cast<float *>(ctx->h_stage + slot + v.n);
                for (size_t f = 0; f < v.n; f += kJobPts) {
                    jobs.push_back(PackJob{v.aos48, pos, nrm, f, std::min(kJobPts, v.n - f), fmt, &pending[p]});
                    ++n_jobs;
                }
                slot += packed_slots(v.n, fmt);
            }
            pending[p].store(n_jobs, std::memory_order_relaxed);
        }
        slot_begin[n_pairs] = slot;
        if (slot > ctx->h_stage_slots || slot > 3 * ctx->cap_in) {
            ctx->err = "internal: packed staging capacity";
            return MULLS_E_CAPACITY;
        }
        pool.submit(jobs); // FIFO: pair 0 is packed first, and its DMA runs while the next pairs are being packed
        // the (pageable, hence synchronously staged) tables go first: queued behind the clouds they would wait for them
        cudaError_t ce = cudaMemcpyAsync(ctx->A.pc, ctx->h_pc.data(), n_pairs * sizeof(PairConst), cudaMemcpyHostToDevice, ctx->stream);
        if (ce == cudaSuccess && !ctx->h_in_chunks.empty())
            ce = cudaMemcpyAsync(ctx->A.in_chunks, ctx->h_in_chunks.data(), ctx->h_in_chunks.size() * sizeof(ChunkDesc),
                                 cudaMemcpyHostToDevice, ctx->stream);
        if (ce == cudaSuccess && !ctx->h_it_chunks.empty())
            ce = cudaMemcpyAsync(ctx->A.it_chunks, ctx->h_it_chunks.data(), ctx->h_it_chunks.size() * sizeof(ChunkDesc),
                                 cudaMemcpyHostToDevice, ctx->stream);
        tables_sent = true; // (every job is waited for even after an error: the jobs point at `pending`)
        if (ce == cudaSuccess && cudaEventRecord(ctx->ev_h2d0, ctx->stream) == cudaSuccess) ctx->h2d_timed = true;
        const double t_pack0 = wall_ms();
        for (size_t p = 0; p < n_pairs; ++p) {
            pool.help_until_done(pending[p]);
            if (p + 1 == n_pairs) ctx->up_ms_pack = (float)(wall_ms() - t_pack0);
            const size_t b = slot_begin[p], e = slot_begin[p + 1];
            if (e > b && ce == cudaSuccess)
                ce = cudaMemcpyAsync((void *)(ctx->A.in_aos + b), ctx->h_stage + b, (e - b) * sizeof(float4), cudaMemcpyHostToDevice,
                                     ctx->stream);
        }
        CK(ce);
    } else {
    if (cudaEventRecord(ctx->ev_h2d0, ctx->stream) == cudaSuccess) ctx->h2d_timed = true;
    for (size_t p = 0; p < n_pairs; ++p) {
        PairConst &pc = ctx->h_pc[p];
        for (int s = 0; s < kNumSegs; ++s) {
            const mulls_cloud_view &v = (s < kNumClasses) ? tgt[p * kNumClasses + s] : src[p * kNumClasses + (s - kNumClasses)];
            pc.in_ptr[s] = ctx->A.in_aos + 3 * (size_t)pc.in_off[s];
            pc.in_fmt[s] = kFmtRows48;
            if (v.n == 0) continue;
            if (tgt_on_device && s < kNumClasses) { // the view already points into HBM (device-resident local map)
                pc.in_ptr[s] = (const float4 *)v.aos48;
                continue;
            }
            if (!resident && ctx->zero_copy) {
                cudaPointerAttributes attr;
                if (cudaPointerGetAttributes(&attr, v.aos48) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
                    attr.devicePointer != nullptr && ((uintptr_t)attr.devicePointer % 16) == 0) {
                    pc.in_ptr[s] = (const float4 *)attr.devicePointer;
                    continue;
                }
                cudaGetLastError(); // pageable memory: not an error, fall through to the copy
            }
            CK(cudaMemcpyAsync((void *)(ctx->A.in_aos + 3 * (size_t)pc.in_off[s]), v.aos48, v.n * 48, cudaMemcpyHostToDevice,
                               ctx->stream));
        }
    }
    }
    if (!tables_sent) {
        CK(cudaMemcpyAsync(ctx->A.pc, ctx->h_pc.data(), n_pairs * sizeof(PairConst), cudaMemcpyHostToDevice, ctx->stream));
        if (!ctx->h_in_chunks.empty())
            CK(cudaMemcpyAsync(ctx->A.in_chunks, ctx->h_in_chunks.data(), ctx->h_in_chunks.size() * sizeof(ChunkDesc),
                               cudaMemcpyHostToDevice, ctx->stream));
        if (!ctx->h_it_chunks.empty())
            CK(cudaMemcpyAsync(ctx->A.it_chunks, ctx->h_it_chunks.data(), ctx->h_it_chunks.size() * sizeof(ChunkDesc),
                               cudaMemcpyHostToDevice, ctx->stream));
    }
    // The tables above live in pageable vectors: cudaMemcpyAsync has already staged them when it returns. The clouds,
    // however, may be the caller's pinned buffers (truly asynchronous copies): a resident upload returns to the caller
    // before anything else runs, so it waits here; a one-shot call goes straight on to run_impl, which synchronises
    // before it returns — the kernels are queued while the clouds are still crossing PCIe.
    if (resident) CK(cudaStreamSynchronize(ctx->stream));
    ctx->n_pairs = n_pairs;
    ctx->n_in = in_off;
    ctx->n_src_total = s_off;
    ctx->n_tgt_total = t_off;
    ctx->max_iter_max = max_iter_max;
    ctx->any_keep_less = any_keep_less;
    ctx->any_normal_shooting = any_shoot;
    ctx->any_undistort = any_undistort;
    ctx->uploaded = true;
    ctx->up_ms_host = (float)(wall_ms() - t_up0);
    return MULLS_OK;
}

// Ingest phase on the resident inputs: state reset, initial guess, intersection filter, Morton sort,
// hashed multi-level grid. Shared by the registration path and mulls_pca_features.
static int launch_ingest(mulls_ctx *ctx, DeviceArrays &A, bool trace, uint64_t &launches, mulls_allreduce_fn hook = nullptr,
                         void *user = nullptr) {
    cudaStream_t st = ctx->stream;
    const int np = (int)ctx->n_pairs;
    const uint32_t n_in = (uint32_t)ctx->n_in;
    if (trace) CK(cudaMemsetAsync(ctx->d_trace, 0, np * sizeof(mulls_icp_trace), st));
    CK(cudaMemsetAsync(A.claim, 0x7f, std::max<size_t>(ctx->n_tgt_total, 1) * sizeof(unsigned), st));
    k_state_init<<<(unsigned)ceil_div(np, 128), 128, 0, st>>>(A, np);
    ++launches;
    const unsigned n_inc = (unsigned)ctx->h_in_chunks.size();
    if (n_inc) {
        if (ctx->any_undistort) k_ingest_transform<true><<<n_inc, kIngestBlock, 0, st>>>(A);
        else k_ingest_transform<false><<<n_inc, kIngestBlock, 0, st>>>(A);
        ++launches;
    }
    if (hook) { // sharded source: the intersection filter needs the bbox over all shards
        k_shard_pack_setup<<<1, 1, 0, st>>>(A, 0);
        if (hook(user, A.xch_i32, 6, 1, 1, (void *)st) != 0) {
            ctx->err = "all-reduce callback failed";
            return MULLS_E_COMM;
        }
        k_shard_pack_setup<<<1, 1, 0, st>>>(A, 1);
        launches += 2;
    }
    k_pair_setup<<<(unsigned)ceil_div(np, 128), 128, 0, st>>>(A, np, ctx->h0_min);
    ++launches;
    if (n_inc) {
        k_make_keys<<<n_inc, kIngestBlock, 0, st>>>(A, ctx->sort_sources);
        ++launches;
        if (ctx->any_keep_less) { // random down-sampling of :2866-2892: radix select of the k-th sampling key
            const unsigned pb = (unsigned)ceil_div(np, 64);
            k_keepless_plan<<<pb, 64, 0, st>>>(A, np);
            for (int pass = 0; pass < 8; ++pass) {
                k_keepless_hist<<<n_inc, kIngestBlock, 0, st>>>(A, pass);
                k_keepless_step<<<pb, 64, 0, st>>>(A, np, pass);
            }
            k_keepless_mark<<<n_inc, kIngestBlock, 0, st>>>(A);
            launches += 18;
        }
        int seg_bits = 1;
        while ((1ull << seg_bits) <= (uint64_t)np * kNumSegs) ++seg_bits;
        size_t bytes = ctx->cub_temp_bytes;
        CK(cub::DeviceRadixSort::SortPairs(ctx->cub_temp, bytes, A.keys_a, A.keys_b, A.vals_a, A.vals_b, (int)n_in, 0,
                                           36 + seg_bits, st));
        // (CUB's radix-sort kernels are library launches and are not counted in kernel_launches)
    }
    k_seg_offsets<<<1, 256, 0, st>>>(A, np);
    ++launches;
    if (hook) { // global class sizes (:1195-1201 counts, K_filter_distant_point test)
        k_shard_pack_setup<<<1, 1, 0, st>>>(A, 2);
        if (hook(user, A.xch_i32, kNumClasses, 1, 0, (void *)st) != 0) {
            ctx->err = "all-reduce callback failed";
            return MULLS_E_COMM;
        }
        k_shard_pack_setup<<<1, 1, 0, st>>>(A, 3);
        launches += 2;
    }
    if (n_in) {
        k_gather<<<(unsigned)ceil_div(n_in, 256), 256, 0, st>>>(A, A.keys_b, A.vals_b, n_in);
        const unsigned hb = (unsigned)ceil_div((size_t)n_in + 1, 256);
        k_hash_build<<<hb, 256, 0, st>>>(A, A.keys_b, n_in, 0);
        k_hash_layout<<<1, 32, 0, st>>>(A, np, ctx->hash_slack);
        k_hash_clear<<<1184, 256, 0, st>>>(A);
        k_hash_build<<<hb, 256, 0, st>>>(A, A.keys_b, n_in, 1);
        k_hash_build<<<hb, 256, 0, st>>>(A, A.keys_b, n_in, 2);
        launches += 6;
    } else {
        k_hash_layout<<<1, 32, 0, st>>>(A, np, ctx->hash_slack);
        ++launches;
    }
    return MULLS_OK;
}

// The iteration kernels run a fixed number of resident blocks that fetch live chunks (for_each_live_chunk): grids are
// sized by the SM count and the blocks an SM holds, never by the batch.
// ... and, for small batches, by the chunks there are (rounded up to a power of two: the grids are part of the graph)
static unsigned chunk_bucket(const mulls_ctx *ctx) {
    unsigned b = 1;
    while (b < (unsigned)ctx->h_it_chunks.size()) b <<= 1;
    return b;
}
static unsigned resident_grid(const mulls_ctx *ctx, int blocks_per_sm) {
    return std::min((unsigned)(ctx->num_sms * blocks_per_sm), chunk_bucket(ctx));
}
// it < 0 (recording the iteration graph): all three modes, each checks the device-side iteration counter; the host
// launch loop knows the iteration and launches the one that runs
static void launch_search(mulls_ctx *ctx, cudaStream_t st, const DeviceArrays &A, int buf, int it) {
    const float reseed = 0.25f * (float)ctx->reseed_cells_x4;
    const unsigned grid = resident_grid(ctx, kSearchBlocksPerSm);
    const int mode = it < 0 ? -1 : (it >= kKeepFromIter ? 2 : (it == kKeepFromIter - 1 ? 1 : 0));
    if (mode < 0 || mode == 0) k_search<0><<<grid, kIterBlock, 0, st>>>(A, buf, it, ctx->start_level0, ctx->leaf_count, ctx->defer_from_iter, reseed);
    if (mode < 0 || mode == 1) k_search<1><<<grid, kIterBlock, 0, st>>>(A, buf, it, ctx->start_level0, ctx->leaf_count, ctx->defer_from_iter, reseed);
    if (mode < 0 || mode == 2) k_search<2><<<grid, kIterBlock, 0, st>>>(A, buf, it, ctx->start_level0, ctx->leaf_count, ctx->defer_from_iter, reseed);
}
constexpr int kShootBlocksPerSm = 8, kResolveBlocksPerSm = 16, kAccumulateBlocksPerSm = 8;

// The iteration loop as a CUDA graph (CUDA 12.4+ conditional nodes): WHILE(handle) { k_search [, k_search_shoot],
// k_resolve, k_accumulate, k_solve } followed by k_posterior, k_finalize, k_collect. Kernel nodes are recorded once per
// context with grids sized for its capacity; what a run needs to know (chunk / pair counts, trace switch, loop counter)
// is read from LoopCtl in device memory. k_solve's last block sets the loop condition: no host polling, one launch.
static int build_iteration_graph(mulls_ctx *ctx) {
    const int key[6] = {ctx->start_level0, ctx->leaf_count + (ctx->reseed_cells_x4 << 12), (int)chunk_bucket(ctx),
                        ctx->any_normal_shooting ? 1 : 0, ctx->defer_from_iter, ctx->search_blocks};
    if (ctx->graph_exec && std::memcmp(key, ctx->graph_key, sizeof(key)) == 0) return MULLS_OK;
    if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec), ctx->graph_exec = nullptr;
    if (ctx->graph) cudaGraphDestroy(ctx->graph), ctx->graph = nullptr;
    cudaStream_t st = ctx->stream;
    DeviceArrays A = ctx->A;
    const unsigned cap_chunks = (unsigned)std::max<size_t>(ctx->cap_it_chunks, 1), cap_pairs = (unsigned)std::max<size_t>(ctx->max_pairs, 1);
    CK(cudaGraphCreate(&ctx->graph, 0));
    cudaGraphConditionalHandle handle;
    CK(cudaGraphConditionalHandleCreate(&handle, ctx->graph, 1, cudaGraphCondAssignDefault));
    cudaGraphNodeParams wp = {cudaGraphNodeTypeConditional};
    wp.conditional.handle = handle;
    wp.conditional.type = cudaGraphCondTypeWhile;
    wp.conditional.size = 1;
    cudaGraphNode_t while_node;
    CK(cudaGraphAddNode(&while_node, ctx->graph, nullptr, 0, &wp));
    cudaGraph_t body = wp.conditional.phGraph_out[0];
    CK(cudaStreamBeginCaptureToGraph(st, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
    launch_search(ctx, st, A, -1, -1);
    if (ctx->any_normal_shooting)
        k_search_shoot<<<resident_grid(ctx, kShootBlocksPerSm), kIterBlock, 0, st>>>(A, -1, ctx->start_level0, ctx->leaf_count);
    k_resolve<<<resident_grid(ctx, kResolveBlocksPerSm), kIterBlock, 0, st>>>(A, -1);
    k_accumulate<<<resident_grid(ctx, kAccumulateBlocksPerSm), kIterBlock, 0, st>>>(A, -1);
    k_solve<<<cap_pairs, kSolveThreads, 0, st>>>(A, -1, (unsigned long long)handle);
    CK(cudaStreamEndCapture(st, nullptr));
    CK(cudaStreamBeginCaptureToGraph(st, ctx->graph, &while_node, nullptr, 1, cudaStreamCaptureModeThreadLocal));
    k_posterior<<<std::min(cap_chunks, chunk_bucket(ctx)), kIterBlock, 0, st>>>(A);
    k_finalize<<<(unsigned)ceil_div(cap_pairs, 64), 64, 0, st>>>(A, -1);
    k_collect<<<(unsigned)ceil_div(cap_pairs, 128), 128, 0, st>>>(A, -1, ctx->d_results);
    CK(cudaStreamEndCapture(st, nullptr));
    CK(cudaGraphInstantiate(&ctx->graph_exec, ctx->graph, 0));
    std::memcpy(ctx->graph_key, key, sizeof(key));
    return MULLS_OK;
}

// Launch the whole path on the resident inputs. If `hook` is given (sharded mode) it is called between
// the phases that need a cross-rank exchange.
static int run_impl_inner(mulls_ctx *ctx, mulls_icp_result *out, mulls_icp_trace *trace, mulls_allreduce_fn hook, void *user,
                          bool finish_now);
static int run_finish_inner(mulls_ctx *ctx, mulls_icp_result *out);
// finish_now = false: everything is enqueued on the context's stream and the call returns; run_finish waits for it
static int run_impl(mulls_ctx *ctx, mulls_icp_result *out, mulls_icp_trace *trace, mulls_allreduce_fn hook, void *user,
                    bool finish_now = true) {
    const int rc = run_impl_inner(ctx, out, trace, hook, user, finish_now);
    // an error exit may leave async copies from / into the caller's buffers (clouds, trace, results) in flight:
    // nothing is handed back before the stream has drained
    if (rc != MULLS_OK && ctx && ctx->stream) cudaStreamSynchronize(ctx->stream);
    return rc;
}
static int run_finish(mulls_ctx *ctx, mulls_icp_result *out) {
    const int rc = run_finish_inner(ctx, out);
    if (rc != MULLS_OK && ctx && ctx->stream) cudaStreamSynchronize(ctx->stream);
    return rc;
}
static int run_impl_inner(mulls_ctx *ctx, mulls_icp_result *out, mulls_icp_trace *trace, mulls_allreduce_fn hook, void *user,
                          bool finish_now) {
    if (!ctx || !ctx->uploaded) return MULLS_E_ARG;
    ctx->pend.active = false;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    DeviceArrays A = ctx->A;
    const int np = (int)ctx->n_pairs;
    uint64_t launches = 0;
    CK(cudaEventRecord(ctx->ev_begin, st));
    {
        int rc = launch_ingest(ctx, A, trace != nullptr, launches, hook, user);
        if (rc != MULLS_OK) return rc;
    }
    const unsigned n_itc = (unsigned)ctx->h_it_chunks.size();
    {
        LoopCtl &c = *ctx->h_ctl; // (the previous run has been synchronised: the staging copy is free)
        c = LoopCtl();
        c.n_it_chunks = (int)n_itc, c.n_pairs = np, c.trace_on = trace ? 1 : 0, c.max_iter = ctx->max_iter_max;
        CK(cudaMemcpyAsync(A.ctl, ctx->h_ctl, sizeof(LoopCtl), cudaMemcpyHostToDevice, st));
        if (n_itc) { // the chunks that own source points after the intersection filter: work list of iteration 0
            k_live_init<<<(unsigned)ceil_div(n_itc, 256), 256, 0, st>>>(A);
            ++launches;
        }
    }
    // small batches: one cooperative kernel runs the whole loop (every chunk and every pair must find a co-resident block)
    bool looped = false;
    if (!hook && ctx->use_graph && ctx->loop_kernel && !ctx->any_normal_shooting && n_itc > 0) {
        if (ctx->loop_kernel_blocks == 0) {
            int per_sm = 0, coop = 0;
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device);
            if (coop && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_icp_loop, kIterBlock, 0) == cudaSuccess && per_sm > 0)
                ctx->loop_kernel_blocks = per_sm * ctx->num_sms;
            else
                ctx->loop_kernel_blocks = -1, cudaGetLastError();
        }
        // `loop_kernel` = how many chunks a co-resident block may have to walk per phase (1: every chunk has its block)
        looped = ctx->loop_kernel_blocks > 0 && n_itc <= (unsigned)(ctx->loop_kernel * ctx->loop_kernel_blocks) &&
                 np <= ctx->loop_kernel * ctx->loop_kernel_blocks;
    }
    const bool graphed = !hook && ctx->use_graph && !looped;
    if (graphed) {
        const int rc = build_iteration_graph(ctx);
        if (rc != MULLS_OK) return rc;
    }
    CK(cudaEventRecord(ctx->ev_ingest, st));
    int n_search_ev = 0;
    if (looped) {
        DeviceArrays Aarg = A;
        int a1 = ctx->start_level0, a2 = ctx->leaf_count, a3 = ctx->defer_from_iter;
        float a4 = 0.25f * (float)ctx->reseed_cells_x4;
        void *args[] = {&Aarg, &a1, &a2, &a3, &a4};
        const unsigned grid = std::max(1u, std::min((unsigned)ctx->loop_kernel_blocks, std::max(n_itc, (unsigned)np)));
        CK(cudaLaunchCooperativeKernel((const void *)k_icp_loop, dim3(grid), dim3(kIterBlock), args, 0, st));
        k_posterior<<<n_itc, kIterBlock, 0, st>>>(A);
        k_finalize<<<(unsigned)ceil_div(np, 64), 64, 0, st>>>(A, np);
        launches += 3;
    } else if (graphed) {
        CK(cudaGraphLaunch(ctx->graph_exec, st));
        CK(cudaMemcpyAsync(ctx->h_ctl, A.ctl, sizeof(LoopCtl), cudaMemcpyDeviceToHost, st)); // iterations executed
    } else if (n_itc) {
        for (int it = 0; it < ctx->max_iter_max; ++it) {
            // flow control: stay at most two iterations ahead of the device and stop launching as soon
            // as every pair has converged or failed (the device mirrors its counter into mapped memory)
            if (it >= 2) {
                // (poll with pauses: several lanes spinning inside the driver slow each other's launches down)
                while (cudaEventQuery(ctx->ev_done[it - 2]) == cudaErrorNotReady)
                    for (int k = 0; k < ctx->poll_pause; ++k) _mm_pause();
                // Sharded runs must take this decision identically on every rank (the ranks issue matching collectives):
                // they read the count the device recorded at the END of iteration it-2 — written once, before
                // ev_done[it-2] — never the live flag, whose value at this instant depends on each rank's timing.
                if (hook ? ((volatile int *)ctx->h_running)[1 + std::min(it - 2, kIterFlags - 1)] <= 0
                         : *(volatile int *)ctx->h_running <= 0)
                    break;
            }
            const int buf = it & 1;
            if (hook) // other ranks' claims of the previous iteration must not survive in this rank's table
                CK(cudaMemsetAsync(A.claim, 0x7f, std::max<size_t>(ctx->n_tgt_total, 1) * sizeof(unsigned), st));
            CK(cudaEventRecord(ctx->ev_search[2 * it], st));
            launch_search(ctx, st, A, buf, it);
            if (ctx->any_normal_shooting) {
                k_search_shoot<<<resident_grid(ctx, kShootBlocksPerSm), kIterBlock, 0, st>>>(A, buf, ctx->start_level0, ctx->leaf_count);
                ++launches;
            }
            CK(cudaEventRecord(ctx->ev_search[2 * it + 1], st));
            if (hook) { // exchange 1: the duplicate-check claims of all shards (min of source indices)
                if (hook(user, A.claim, ctx->n_tgt_total, 1, 1, (void *)st) != 0) {
                    ctx->err = "all-reduce callback failed";
                    return MULLS_E_COMM;
                }
            }
            k_resolve<<<resident_grid(ctx, kResolveBlocksPerSm), kIterBlock, 0, st>>>(A, buf);
            if (hook) { // exchange 2: correspondence counts (w_ground, -2 test) and surviving source counts
                k_shard_counts<<<1, kIterBlock, 0, st>>>(A, 0);
                if (hook(user, A.xch_i32, 2 * kNumClasses, 1, 0, (void *)st) != 0) {
                    ctx->err = "all-reduce callback failed";
                    return MULLS_E_COMM;
                }
                k_shard_counts<<<1, kIterBlock, 0, st>>>(A, 1);
                launches += 2;
            }
            k_accumulate<<<resident_grid(ctx, kAccumulateBlocksPerSm), kIterBlock, 0, st>>>(A, buf);
            k_solve<<<(unsigned)np, kSolveThreads, 0, st>>>(A, buf, 0ull);
            if (hook) { // exchange 3: per-class normal-equation sums; then every rank solves the same system
                if (hook(user, A.xch_f64, kNumClasses * kTerms, 0, 0, (void *)st) != 0) {
                    ctx->err = "all-reduce callback failed";
                    return MULLS_E_COMM;
                }
                k_shard_solve<<<1, 32, 0, st>>>(A, buf, std::min(it, kIterFlags - 1));
                ++launches;
            }
            CK(cudaEventRecord(ctx->ev_done[it], st));
            launches += 4;
            n_search_ev = it + 1;
        }
        k_posterior<<<n_itc, kIterBlock, 0, st>>>(A);
        if (hook) {
            k_shard_post<<<1, 32, 0, st>>>(A, 0);
            if (hook(user, A.xch_f64, 2, 0, 0, (void *)st) != 0) {
                ctx->err = "all-reduce callback failed";
                return MULLS_E_COMM;
            }
            k_shard_post<<<1, 32, 0, st>>>(A, 1);
            launches += 3;
        } else {
            k_finalize<<<(unsigned)ceil_div(np, 64), 64, 0, st>>>(A, np);
            launches += 2;
        }
    }
    CK(cudaEventRecord(ctx->ev_iter, st));
    if (!graphed) {
        k_collect<<<(unsigned)ceil_div(np, 128), 128, 0, st>>>(A, np, ctx->d_results);
        ++launches;
    }
    CK(cudaMemcpyAsync(ctx->h_results, ctx->d_results, np * (sizeof(mulls_icp_result) + sizeof(uint64_t)), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(ctx->h_flags, A.hash_used, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    if (trace) CK(cudaMemcpyAsync(trace, ctx->d_trace, np * sizeof(mulls_icp_trace), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(ctx->ev_end, st));
    ctx->pend.launches = launches, ctx->pend.n_search_ev = n_search_ev, ctx->pend.graphed = graphed, ctx->pend.hooked = hook != nullptr;
    ctx->pend.active = true;
    if (!finish_now) return MULLS_OK;
    return run_finish_inner(ctx, out);
}

static int run_finish_inner(mulls_ctx *ctx, mulls_icp_result *out) {
    if (!ctx || !ctx->pend.active) return MULLS_E_ARG;
    ctx->pend.active = false;
    cudaStream_t st = ctx->stream;
    const int np = (int)ctx->n_pairs;
    uint64_t launches = ctx->pend.launches;
    const int n_search_ev = ctx->pend.n_search_ev;
    const bool graphed = ctx->pend.graphed;
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    // (graph: three k_search forms, k_resolve, k_accumulate, k_solve per executed iteration + posterior, finalize, collect)
    if (graphed) launches += (uint64_t)ctx->h_ctl->it * (6u + (ctx->any_normal_shooting ? 1u : 0u)) + 3u;
    if (ctx->h_flags[1]) {
        ctx->err = "hash pool exhausted (target clouds produce more grid cells than the context reserves)";
        return MULLS_E_CAPACITY;
    }
    if (out) std::memcpy(out, ctx->h_results, np * sizeof(mulls_icp_result));
    // statistics
    mulls_run_stats &S = ctx->stats;
    S = mulls_run_stats();
    S.kernel_launches = launches;
    cudaEventElapsedTime(&S.ms_ingest, ctx->ev_begin, ctx->ev_ingest);
    cudaEventElapsedTime(&S.ms_iterate, ctx->ev_ingest, ctx->ev_iter);
    cudaEventElapsedTime(&S.ms_total, ctx->ev_begin, ctx->ev_end);
    if (ctx->h2d_timed) cudaEventElapsedTime(&S.ms_h2d, ctx->ev_h2d0, ctx->ev_begin);
    S.ms_host_pack = ctx->up_ms_pack, S.ms_host_upload = ctx->up_ms_host;
    ctx->h2d_timed = false;
    float ms = 0.f;
    for (int it = 0; it < n_search_ev; ++it) {
        float t = 0.f;
        cudaEventElapsedTime(&t, ctx->ev_search[2 * it], ctx->ev_search[2 * it + 1]);
        S.ms_search_iter[it] = t;
        ms += t;
    }
    S.ms_search = ms;
    S.search_launches = (uint64_t)n_search_ev;
    for (int p = 0; p < np; ++p) S.iterations += (uint64_t)ctx->h_results[p].iters;
    // algorithmic bytes are accumulated on the device per executed iteration (k_collect puts them behind the results)
    {
        const uint64_t *ab = reinterpret_cast<const uint64_t *>(ctx->h_results + np);
        for (int p = 0; p < np; ++p) S.algorithmic_bytes += ab[p];
    }
    ctx->grid_valid = !ctx->pend.hooked;
    return MULLS_OK;
}

int mulls_batch_upload(mulls_ctx *ctx, size_t n_pairs, const mulls_cloud_view *tgt, const mulls_cloud_view *src,
                       const mulls_icp_params *params, const double *init_guess) {
    if (ctx && !ctx->lanes.empty()) {
        if (!tgt || !src || !params || !init_guess || n_pairs == 0) return MULLS_E_ARG;
        if (n_pairs > ctx->max_pairs) {
            ctx->err = "more pairs than the context was created for";
            return MULLS_E_CAPACITY;
        }
        ctx->n_pairs = n_pairs;
        const int rc = for_each_lane(ctx, n_pairs, [&](mulls_ctx *lane, size_t b, size_t n) {
            return upload_impl(lane, n, tgt + b * kNumClasses, src + b * kNumClasses, params + b, init_guess + 16 * b, nullptr,
                               nullptr);
        });
        ctx->uploaded = (rc == MULLS_OK);
        return rc;
    }
    return upload_impl(ctx, n_pairs, tgt, src, params, init_guess, nullptr, nullptr);
}

int mulls_batch_run_resident(mulls_ctx *ctx, mulls_icp_result *out, mulls_icp_trace *trace) {
    if (ctx && !ctx->lanes.empty()) {
        if (!ctx->uploaded) return MULLS_E_ARG;
        const int rc = for_each_lane(ctx, ctx->n_pairs, [&](mulls_ctx *lane, size_t b, size_t) {
            return run_impl(lane, out ? out + b : nullptr, trace ? trace + b : nullptr, nullptr, nullptr);
        });
        merge_lane_stats(ctx);
        return rc;
    }
    return run_impl(ctx, out, trace, nullptr, nullptr);
}

// One-shot batch on ONE context (host buffers in, results out). With >= 2 pairs and the iteration graph the batch is
// double-buffered over the context and its twin (own stream and buffers, created on first use): the second half is
// packed and copied while the first half is being registered; both halves are collected at the end.
static int one_shot_batch(mulls_ctx *ctx, size_t n_pairs, const mulls_cloud_view *tgt, const mulls_cloud_view *src,
                          const mulls_icp_params *params, const double *init_guess, mulls_icp_result *out, mulls_icp_trace *trace) {
    const double t0 = wall_ms();
    const bool split = ctx->double_buffer && ctx->use_graph && n_pairs >= 2 && n_pairs <= ctx->max_pairs;
    if (split && !ctx->twin) {
        mulls_ctx *t = mulls_create(ctx->device, (ctx->max_pairs + 1) / 2, ctx->max_src, ctx->max_tgt);
        if (t) { // (no memory for it: the call simply runs on one context)
            t->start_level0 = ctx->start_level0, t->leaf_count = ctx->leaf_count, t->reseed_cells_x4 = ctx->reseed_cells_x4;
            t->defer_from_iter = ctx->defer_from_iter, t->sort_sources = ctx->sort_sources, t->hash_slack = ctx->hash_slack;
            t->use_graph = ctx->use_graph, t->zero_copy = ctx->zero_copy, t->host_pack = ctx->host_pack, t->poll_pause = ctx->poll_pause;
            t->stage_wc = ctx->stage_wc, t->h0_min = ctx->h0_min, t->double_buffer = 0;
            ctx->twin = t;
        }
    }
    if (!split || !ctx->twin) {
        int rc = upload_impl(ctx, n_pairs, tgt, src, params, init_guess, nullptr, nullptr, /*resident=*/false);
        if (rc != MULLS_OK) return rc;
        rc = run_impl(ctx, out, trace, nullptr, nullptr);
        ctx->uploaded = false; // nothing stays resident after a one-shot call
        ctx->stats.ms_host_call = (float)(wall_ms() - t0);
        return rc;
    }
    mulls_ctx *a = ctx, *b = ctx->twin;
    const size_t n0 = (n_pairs + 1) / 2, n1 = n_pairs - n0;
    int rc = upload_impl(a, n0, tgt, src, params, init_guess, nullptr, nullptr, /*resident=*/false);
    if (rc == MULLS_OK) rc = run_impl(a, nullptr, trace, nullptr, nullptr, /*finish_now=*/false);
    int rcb = MULLS_OK;
    if (rc == MULLS_OK) {
        rcb = upload_impl(b, n1, tgt + n0 * kNumClasses, src + n0 * kNumClasses, params + n0, init_guess + 16 * n0, nullptr, nullptr,
                          /*resident=*/false);
        if (rcb == MULLS_OK) rcb = run_impl(b, nullptr, trace ? trace + n0 : nullptr, nullptr, nullptr, /*finish_now=*/false);
    }
    // whatever happened, nothing is handed back while one of the two streams still works on the caller's buffers
    if (rc == MULLS_OK) rc = run_finish(a, out);
    else cudaStreamSynchronize(a->stream);
    if (rc == MULLS_OK && rcb == MULLS_OK) rcb = run_finish(b, out ? out + n0 : nullptr);
    else if (b->stream) cudaStreamSynchronize(b->stream), b->pend.active = false;
    a->uploaded = b->uploaded = false;
    if (rc == MULLS_OK && rcb != MULLS_OK) {
        ctx->err = b->err;
        rc = rcb;
    }
    if (rc == MULLS_OK) { // the call's statistics: both halves (device times overlap: the longer one is reported)
        mulls_run_stats &S = a->stats;
        const mulls_run_stats &T = b->stats;
        S.kernel_launches += T.kernel_launches, S.algorithmic_bytes += T.algorithmic_bytes, S.iterations += T.iterations;
        S.ms_ingest = std::max(S.ms_ingest, T.ms_ingest), S.ms_iterate = std::max(S.ms_iterate, T.ms_iterate);
        S.ms_total = std::max(S.ms_total, T.ms_total);
        S.ms_h2d += T.ms_h2d, S.ms_host_pack += T.ms_host_pack, S.ms_host_upload += T.ms_host_upload;
    }
    ctx->stats.ms_host_call = (float)(wall_ms() - t0);
    return rc;
}

int mulls_icp_run_batch(mulls_ctx *ctx, size_t n_pairs, const mulls_cloud_view *tgt, const mulls_cloud_view *src,
                        const mulls_icp_params *params, const double *init_guess, mulls_icp_result *out,
                        mulls_icp_trace *trace) {
    if (ctx && !ctx->lanes.empty()) {
        // pipelined: every lane uploads and registers its slice on its own stream — while one slice is being
        // registered the next one's clouds are already crossing PCIe
        if (!tgt || !src || !params || !init_guess || n_pairs == 0) return MULLS_E_ARG;
        if (n_pairs > ctx->max_pairs) {
            ctx->err = "more pairs than the context was created for";
            return MULLS_E_CAPACITY;
        }
        ctx->n_pairs = n_pairs;
        ctx->uploaded = false;
        const int rc = for_each_lane(ctx, n_pairs, [&](mulls_ctx *lane, size_t b, size_t n) {
            return one_shot_batch(lane, n, tgt + b * kNumClasses, src + b * kNumClasses, params + b, init_guess + 16 * b,
                                  out ? out + b : nullptr, trace ? trace + b : nullptr);
        });
        merge_lane_stats(ctx);
        return rc;
    }
    if (!ctx || !tgt || !src || !params || !init_guess || n_pairs == 0) return MULLS_E_ARG;
    return one_shot_batch(ctx, n_pairs, tgt, src, params, init_guess, out, trace);
}

int mulls_icp_run(mulls_ctx *ctx, const mulls_cloud_view tgt[MULLS_NUM_CLASSES], const mulls_cloud_view src[MULLS_NUM_CLASSES],
                  const mulls_icp_params *params, const double init_guess[16], mulls_icp_result *out,
                  mulls_icp_trace *trace) {
    return mulls_icp_run_batch(ctx, 1, tgt, src, params, init_guess, out, trace);
}

} // extern "C"

extern "C" {

int mulls_nccl_unique_id(char id[MULLS_NCCL_ID_BYTES]) {
    if (!id) return MULLS_E_ARG;
    NcclApi &api = nccl_api();
    if (!api.ok) return MULLS_E_COMM;
    ncclUniqueIdBytes u;
    if (api.get_id(&u) != 0) return MULLS_E_COMM;
    std::memcpy(id, u.internal, MULLS_NCCL_ID_BYTES);
    return MULLS_OK;
}

int mulls_nccl_init(mulls_ctx *ctx, int rank, int world, const char id[MULLS_NCCL_ID_BYTES]) {
    if (!ctx || !id || world < 1 || rank < 0 || rank >= world) return MULLS_E_ARG;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0];
    NcclApi &api = nccl_api();
    if (!api.ok) {
        ctx->err = "libnccl.so.2 not found (or too old)";
        return MULLS_E_COMM;
    }
    CK(cudaSetDevice(ctx->device));
    if (ctx->nccl_comm) api.destroy(ctx->nccl_comm), ctx->nccl_comm = nullptr;
    ncclUniqueIdBytes u;
    std::memcpy(u.internal, id, MULLS_NCCL_ID_BYTES);
    const int rc = api.init_rank(&ctx->nccl_comm, world, u, rank);
    if (rc != 0) {
        ctx->err = std::string("ncclCommInitRank: ") + (api.err ? api.err(rc) : "failed");
        ctx->nccl_comm = nullptr;
        return MULLS_E_COMM;
    }
    return MULLS_OK;
}

int mulls_icp_run_sharded_nccl(mulls_ctx *ctx, void *comm, const mulls_cloud_view tgt[MULLS_NUM_CLASSES],
                               const mulls_cloud_view src_shard[MULLS_NUM_CLASSES], const uint32_t src_index_base[MULLS_NUM_CLASSES],
                               const uint32_t src_global_n[MULLS_NUM_CLASSES], const mulls_icp_params *params,
                               const double init_guess[16], mulls_icp_result *out, mulls_icp_trace *trace) {
    if (!ctx) return MULLS_E_ARG;
    mulls_ctx *owner = ctx->lanes.empty() ? ctx : ctx->lanes[0];
    if (!comm) comm = owner->nccl_comm;
    if (!comm || !nccl_api().ok) {
        owner->err = "no NCCL communicator: call mulls_nccl_init first (or pass an ncclComm_t)";
        return MULLS_E_COMM;
    }
    return mulls_icp_run_sharded(ctx, tgt, src_shard, src_index_base, src_global_n, params, init_guess, nccl_allreduce_hook, comm, out,
                                 trace);
}

int mulls_nn_query(mulls_ctx *ctx, int cls, const float *xyz, size_t n, int32_t *idx, float *d2) {
    if (!ctx || cls < 0 || cls >= kNumClasses || (n > 0 && (!xyz || !idx || !d2))) return MULLS_E_ARG;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0]; // (a pipelined context answers for the first pair of its first lane)
    if (!ctx->grid_valid) {
        ctx->err = "mulls_nn_query: no registration has run on this context since its last upload";
        return MULLS_E_ARG;
    }
    if (n == 0) return MULLS_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    float *d_q = nullptr;
    int *d_i = nullptr;
    float *d_d = nullptr;
    CK(cudaMallocAsync((void **)&d_q, 3 * n * sizeof(float), st));
    CK(cudaMallocAsync((void **)&d_i, n * sizeof(int), st));
    CK(cudaMallocAsync((void **)&d_d, n * sizeof(float), st));
    CK(cudaMemcpyAsync(d_q, xyz, 3 * n * sizeof(float), cudaMemcpyHostToDevice, st));
    k_nn_query<<<(unsigned)ceil_div(n, kIterBlock), kIterBlock, 0, st>>>(ctx->A, cls, d_q, (uint32_t)n, ctx->start_level0,
                                                                           ctx->leaf_count, d_i, d_d);
    CK(cudaMemcpyAsync(idx, d_i, n * sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(d2, d_d, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    cudaFreeAsync(d_q, st);
    cudaFreeAsync(d_i, st);
    cudaFreeAsync(d_d, st);
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    return MULLS_OK;
}

int mulls_icp_run_sharded(mulls_ctx *ctx, const mulls_cloud_view tgt[MULLS_NUM_CLASSES],
                          const mulls_cloud_view src_shard[MULLS_NUM_CLASSES],
                          const uint32_t src_index_base[MULLS_NUM_CLASSES], const uint32_t src_global_n[MULLS_NUM_CLASSES],
                          const mulls_icp_params *params, const double init_guess[16], mulls_allreduce_fn allreduce,
                          void *user, mulls_icp_result *out, mulls_icp_trace *trace) {
    if (!ctx || !allreduce || !params) return MULLS_E_ARG;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0];
    if (params->keep_less_source_points && !params->apply_motion_undistortion_while_registration) {
        // the down-sampling quota and its sampling keys are defined over the WHOLE source cloud (:2866-2892); a
        // shard-local plan would keep ~world times too many points and a different subset than the unsharded run
        ctx->err = "keep_less_source_points is not supported for a source-sharded registration";
        return MULLS_E_UNSUPPORTED;
    }
    int rc = upload_impl(ctx, 1, tgt, src_shard, params, init_guess, src_index_base, src_global_n, /*resident=*/false);
    if (rc != MULLS_OK) return rc;
    rc = run_impl(ctx, out, trace, allreduce, user);
    ctx->uploaded = false;
    return rc;
}

} // extern "C"

// PCA features of one cloud (host rows, or rows already in HBM) into ctx->pca_buf; `args` receives the device arrays.
// Nothing is synchronised: the caller consumes the arrays on ctx->stream.
static int pca_on_device(mulls_ctx *ctx, mulls_cloud_view cloud, bool cloud_on_device, float radius, int k, int stride,
                         PcaArgs &args, uint64_t &launches, uint32_t *nbr = nullptr) {
    // the cloud becomes the only target class of a one-pair batch: same filter-less ingest, same grid
    mulls_icp_params P;
    mulls_icp_default_params(&P);
    std::strcpy(P.used_feature_type, "100000");
    P.apply_intersection_filter = 0;
    P.dis_thre_unit = radius; // the grid's top level then covers 2.5 x radius
    P.max_iter_num = 0;
    mulls_cloud_view tgt[MULLS_NUM_CLASSES] = {cloud, {nullptr, 0}, {nullptr, 0}, {nullptr, 0}, {nullptr, 0}, {nullptr, 0}};
    mulls_cloud_view src[MULLS_NUM_CLASSES] = {{nullptr, 0}, {nullptr, 0}, {nullptr, 0}, {nullptr, 0}, {nullptr, 0}, {nullptr, 0}};
    const double ident[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    int rc = upload_impl(ctx, 1, tgt, src, &P, ident, nullptr, nullptr, /*resident=*/false, cloud_on_device);
    if (rc != MULLS_OK) return rc;
    const size_t n = cloud.n;
    const size_t bytes = n * (9 * sizeof(float) + sizeof(int));
    if (bytes > ctx->pca_buf_bytes) {
        if (ctx->pca_buf) cudaFree(ctx->pca_buf);
        ctx->pca_buf = nullptr;
        ctx->pca_buf_bytes = 0;
        CK(cudaMalloc(&ctx->pca_buf, std::max<size_t>(bytes, 16)));
        ctx->pca_buf_bytes = bytes;
    }
    cudaStream_t st = ctx->stream;
    DeviceArrays A = ctx->A;
    A.trace = nullptr;
    rc = launch_ingest(ctx, A, false, launches);
    if (rc != MULLS_OK) return rc;
    args.radius = radius;
    args.r2 = (float)((double)radius * (double)radius);
    args.k = k;
    args.stride = stride;
    args.eigenvalues = (float *)ctx->pca_buf;
    args.principal = args.eigenvalues + 3 * n;
    args.normal = args.principal + 3 * n;
    args.pt_num = (int *)(args.normal + 3 * n);
    args.nbr = nbr;
    CK(cudaMemsetAsync(ctx->pca_buf, 0, std::max<size_t>(bytes, 16), st));
    if (n) {
        k_pca<<<(unsigned)ceil_div(n, kPcaWarps), kPcaWarps * 32, 0, st>>>(A, args);
        ++launches;
    }
    CK(cudaMemcpyAsync(ctx->h_flags, A.hash_used, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    ctx->uploaded = false; // the resident batch was replaced by the PCA cloud
    return MULLS_OK;
}

extern "C" {

int mulls_pca_features(mulls_ctx *ctx, mulls_cloud_view cloud, float radius, int k, int stride, mulls_pca_out *out) {
    if (!ctx || !out || !out->eigenvalues || !out->principal || !out->normal || !out->pt_num || stride < 1 ||
        !(radius > 0.f))
        return MULLS_E_ARG;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0];
    PcaArgs args;
    uint64_t launches = 0;
    const size_t n = cloud.n;
    // k within the list capacity (the reference uses 20..50): pcl::PCA's float mean / covariance accumulated in
    // radiusSearch order — bit-reproducible against the CPU path; larger or unlimited k: fp64 warp reduction
    uint32_t *nbr = nullptr;
    if (k >= 1 && k <= kPcaListCap && n > 0) {
        const size_t bytes = n * (size_t)k * sizeof(uint32_t);
        if (bytes > ctx->cls_buf_bytes) {
            if (ctx->cls_buf) cudaFree(ctx->cls_buf);
            ctx->cls_buf = nullptr;
            ctx->cls_buf_bytes = 0;
            CK(cudaMalloc(&ctx->cls_buf, bytes));
            ctx->cls_buf_bytes = bytes;
        }
        nbr = (uint32_t *)ctx->cls_buf;
    }
    int rc = pca_on_device(ctx, cloud, false, radius, k, stride, args, launches, nbr);
    if (rc != MULLS_OK) return rc;
    cudaStream_t st = ctx->stream;
    if (n) {
        CK(cudaMemcpyAsync(out->eigenvalues, args.eigenvalues, 3 * n * sizeof(float), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(out->principal, args.principal, 3 * n * sizeof(float), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(out->normal, args.normal, 3 * n * sizeof(float), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(out->pt_num, args.pt_num, n * sizeof(int), cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (ctx->h_flags[1]) {
        ctx->err = "hash pool exhausted";
        return MULLS_E_CAPACITY;
    }
    ctx->stats = mulls_run_stats();
    ctx->stats.kernel_launches = launches;
    return MULLS_OK;
}

// ================================================================================================
// Device-resident local map (MapManager::update_local_map, src/map_manager.cpp:17-145)
// ================================================================================================
} // extern "C"

struct mulls_map {
    mulls_ctx *ctx = nullptr;
    size_t cap = 0;                      // rows per class buffer
    float4 *buf[2][kNumClasses] = {};    // the map, ping-pong
    float4 *mid[kNumClasses] = {};       // after append + transform + radius crop
    float4 *scan[kNumClasses] = {};      // the scan's down clouds of the running update
    uint8_t *drop[kNumClasses] = {};     // per scan point: removed by the dynamic filter
    int cur = 0;
    uint32_t n[kNumClasses] = {};
    double pose[16];
    double local_bound[6], bound[6];
    MapState *d_state = nullptr, *h_state = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    mulls_map_info last{};
    uint64_t epoch = 0; // bumped by every change of the content
};

namespace {
// Eigen::Matrix4d::inverse(): adjugate / determinant
void host_inverse4(const double *m, double *out) {
    double inv[16];
    inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
    inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
    inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
    inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
    inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
    inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
    inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
    inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
    inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
    inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
    inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
    inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
    inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
    inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
    inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
    inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
    const double det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
    for (int i = 0; i < 16; ++i) out[i] = inv[i] * (1.0 / det);
}
void host_mul4(const double *a, const double *b, double *out) { // sequential over k
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) {
            double acc = 0.0;
            for (int k = 0; k < 4; ++k) acc += a[4 * i + k] * b[4 * k + j];
            out[4 * i + j] = acc;
        }
}
void map_fill_info(const mulls_map *m, mulls_map_info *info) {
    *info = m->last;
    for (int i = 0; i < 16; ++i) info->pose_lo[i] = m->pose[i];
    for (int i = 0; i < 6; ++i) info->local_bound[i] = m->local_bound[i], info->bound[i] = m->bound[i];
    for (int c = 0; c < kNumClasses; ++c) info->n[c] = m->n[c];
    info->feature_point_num = (int)(m->n[0] + m->n[1] + m->n[2] + m->n[3] + m->n[4]);
}
} // namespace

extern "C" {

void mulls_map_default_params(mulls_map_params *p) { // include/pgo/map_manager.h:22-32
    std::memset(p, 0, sizeof(*p));
    p->local_map_radius = 80.f;
    p->max_num_pts = 20000;
    p->kept_vertex_num = 800;
    p->last_frame_reliable_radius = 60.f;
    p->map_based_dynamic_removal_on = 0;
    std::strcpy(p->used_feature_type, "111110");
    p->dynamic_removal_center_radius = 30.0f;
    p->dynamic_dist_thre_min = 0.3f;
    p->dynamic_dist_thre_max = 3.0f;
    p->near_dist_thre = 0.03f;
    p->recalculate_feature_on = 0;
    p->random_seed = 0;
}

void mulls_map_destroy(mulls_map *m) {
    if (!m) return;
    mulls_ctx *ctx = m->ctx;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->tree_map == m) ctx->tree_map = nullptr;
    for (int c = 0; c < kNumClasses; ++c) {
        cudaFree(m->buf[0][c]);
        cudaFree(m->buf[1][c]);
        cudaFree(m->mid[c]);
        cudaFree(m->scan[c]);
        cudaFree(m->drop[c]);
    }
    cudaFree(m->d_state);
    if (m->h_state) cudaFreeHost(m->h_state);
    if (m->ev0) cudaEventDestroy(m->ev0);
    if (m->ev1) cudaEventDestroy(m->ev1);
    delete m;
}

mulls_map *mulls_map_create(mulls_ctx *ctx, size_t max_pts_per_class) {
    if (!ctx || max_pts_per_class == 0 || max_pts_per_class >= (1ull << 31)) return nullptr;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0];
    if (cudaSetDevice(ctx->device) != cudaSuccess) return nullptr;
    mulls_map *m = new mulls_map();
    m->ctx = ctx;
    m->cap = max_pts_per_class;
    bool ok = true;
    const size_t bytes = max_pts_per_class * 48;
    for (int c = 0; c < kNumClasses && ok; ++c) {
        ok = ok && cudaMalloc((void **)&m->buf[0][c], bytes) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&m->buf[1][c], bytes) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&m->mid[c], bytes) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&m->scan[c], bytes) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&m->drop[c], max_pts_per_class) == cudaSuccess;
    }
    ok = ok && cudaMalloc((void **)&m->d_state, sizeof(MapState)) == cudaSuccess;
    ok = ok && cudaMallocHost((void **)&m->h_state, sizeof(MapState)) == cudaSuccess;
    ok = ok && cudaEventCreate(&m->ev0) == cudaSuccess && cudaEventCreate(&m->ev1) == cudaSuccess;
    if (!ok) {
        ctx->err = std::string("mulls_map_create: ") + cudaGetErrorString(cudaGetLastError());
        mulls_map_destroy(m);
        return nullptr;
    }
    const double big = 1.7976931348623157e308;
    for (int i = 0; i < 16; ++i) m->pose[i] = (i % 5 == 0) ? 1.0 : 0.0; // cloudblock_t starts at the identity pose
    for (int d = 0; d < 3; ++d) {
        m->local_bound[d] = m->bound[d] = big;
        m->local_bound[3 + d] = m->bound[3 + d] = -big;
    }
    return m;
}

int mulls_map_set(mulls_map *m, const mulls_cloud_view cls[MULLS_NUM_CLASSES], const double pose_lo[16]) {
    if (!m || !cls || !pose_lo) return MULLS_E_ARG;
    mulls_ctx *ctx = m->ctx;
    CK(cudaSetDevice(ctx->device));
    for (int c = 0; c < kNumClasses; ++c) {
        if (cls[c].n > m->cap) {
            ctx->err = "mulls_map_set: class cloud larger than the map's capacity";
            return MULLS_E_CAPACITY;
        }
        if (cls[c].n > 0 && !cls[c].aos48) return MULLS_E_ARG;
    }
    const double big = 1.7976931348623157e308;
    double lb[6] = {big, big, big, -big, -big, -big};
    for (int c = 0; c < kNumClasses; ++c) {
        if (cls[c].n)
            CK(cudaMemcpyAsync(m->buf[m->cur][c], cls[c].aos48, cls[c].n * 48, cudaMemcpyHostToDevice, ctx->stream));
        m->n[c] = (uint32_t)cls[c].n;
        for (size_t i = 0; i < cls[c].n; ++i) // get_cloud_bbx, utility.hpp:817-847
            for (int d = 0; d < 3; ++d) {
                const double v = cls[c].aos48[12 * i + d];
                if (lb[d] > v) lb[d] = v;
                if (lb[3 + d] < v) lb[3 + d] = v;
            }
    }
    CK(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 16; ++i) m->pose[i] = pose_lo[i];
    for (int i = 0; i < 6; ++i) m->local_bound[i] = lb[i];
    // the world-frame box is refreshed by the next update; until then report the local one moved by the pose's translation
    for (int d = 0; d < 3; ++d) {
        m->bound[d] = lb[d] + pose_lo[4 * d + 3];
        m->bound[3 + d] = lb[3 + d] + pose_lo[4 * d + 3];
    }
    m->last = mulls_map_info();
    ++m->epoch;
    if (ctx->tree_map == m) ctx->tree_map = nullptr;
    return MULLS_OK;
}

int mulls_map_get_info(const mulls_map *m, mulls_map_info *info) {
    if (!m || !info) return MULLS_E_ARG;
    map_fill_info(m, info);
    return MULLS_OK;
}

int mulls_map_download(mulls_map *m, int cls, float *out_aos48, size_t cap, size_t *n) {
    if (!m || cls < 0 || cls >= kNumClasses || !n) return MULLS_E_ARG;
    mulls_ctx *ctx = m->ctx;
    *n = m->n[cls];
    if (!out_aos48) return MULLS_OK;
    if (cap < m->n[cls]) {
        ctx->err = "mulls_map_download: buffer too small";
        return MULLS_E_CAPACITY;
    }
    CK(cudaSetDevice(ctx->device));
    if (m->n[cls]) CK(cudaMemcpy(out_aos48, m->buf[m->cur][cls], (size_t)m->n[cls] * 48, cudaMemcpyDeviceToHost));
    return MULLS_OK;
}

int mulls_map_update(mulls_map *m, const mulls_cloud_view scan_down[MULLS_NUM_CLASSES], const double scan_pose_lo[16],
                     const mulls_map_params *params, mulls_map_info *info) {
    if (!m || !scan_down || !scan_pose_lo || !params) return MULLS_E_ARG;
    mulls_ctx *ctx = m->ctx;
    const mulls_map_params &P = *params;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    MapArgs M;
    std::memset(&M, 0, sizeof(M));
    const size_t nu = strnlen(P.used_feature_type, 8);
    for (int c = 0; c < kNumClasses; ++c) {
        M.used[c] = (c < (int)nu && P.used_feature_type[c] == '1') ? 1 : 0;
        if (scan_down[c].n > 0 && !scan_down[c].aos48) return MULLS_E_ARG;
        if (scan_down[c].n > m->cap || (size_t)m->n[c] + scan_down[c].n > m->cap) {
            ctx->err = "mulls_map_update: map + scan exceed max_pts_per_class";
            return MULLS_E_CAPACITY;
        }
    }
    // :28, :32 tran_target_map = pose_scan^-1 * pose_map and its inverse
    double inv_scan[16];
    host_inverse4(scan_pose_lo, inv_scan);
    host_mul4(inv_scan, m->pose, M.T);
    host_inverse4(M.T, M.Tinv);
    for (int i = 0; i < 16; ++i) M.pose[i] = scan_pose_lo[i];
    M.radius = (double)P.local_map_radius;
    M.max_num_pts = P.max_num_pts;
    M.kept_vertex_num = P.kept_vertex_num;
    M.seed = P.random_seed;
    M.state = m->d_state;
    const int nxt = m->cur ^ 1;
    for (int c = 0; c < kNumClasses; ++c) {
        M.old_pts[c] = m->buf[m->cur][c];
        M.scan_pts[c] = m->scan[c];
        M.scan_drop[c] = nullptr;
        M.mid[c] = m->mid[c];
        M.out[c] = m->buf[nxt][c];
        M.n_old[c] = m->n[c];
        M.n_scan[c] = (uint32_t)scan_down[c].n;
    }
    CK(cudaEventRecord(m->ev0, st));
    for (int c = 0; c < kNumClasses; ++c)
        if (scan_down[c].n)
            CK(cudaMemcpyAsync(m->scan[c], scan_down[c].aos48, scan_down[c].n * 48, cudaMemcpyHostToDevice, st));
    // :37-48 map-based dynamic object removal on the scan's pillar / beam / facade points
    const int feature_point_num = (int)(m->n[0] + m->n[1] + m->n[2] + m->n[3] + m->n[4]);
    if (P.map_based_dynamic_removal_on && feature_point_num > P.max_num_pts / 5) {
        if (ctx->tree_map != m || ctx->tree_epoch != m->epoch) {
            ctx->err = "mulls_map_update: map_based_dynamic_removal_on needs the target trees of the preceding "
                       "mulls_icp_run_to_map on this map";
            return MULLS_E_ARG;
        }
        MapDynArgs D;
        std::memset(&D, 0, sizeof(D));
        const int order[3] = {MULLS_PILLAR, MULLS_BEAM, MULLS_FACADE};
        size_t nq = 0;
        for (int k = 0; k < 3; ++k) {
            const int c = order[k];
            D.cls[k] = c;
            D.scan_pts[k] = m->scan[c];
            D.drop[k] = m->drop[c];
            D.n_scan[k] = M.used[c] ? (uint32_t)scan_down[c].n : 0u;
            if (D.n_scan[k]) {
                CK(cudaMemsetAsync(m->drop[c], 0, D.n_scan[k], st));
                M.scan_drop[c] = m->drop[c];
            }
            nq += D.n_scan[k];
        }
        for (int i = 0; i < 16; ++i) D.Tinv[i] = M.Tinv[i];
        D.center_radius = P.dynamic_removal_center_radius;
        D.dist_min = P.dynamic_dist_thre_min;
        // :34 max_(dynamic_dist_thre_max, dynamic_dist_thre_min + 0.1)
        D.dist_max = ((double)P.dynamic_dist_thre_max > (double)P.dynamic_dist_thre_min + 0.1)
                         ? P.dynamic_dist_thre_max
                         : (float)((double)P.dynamic_dist_thre_min + 0.1);
        D.near_thre = P.near_dist_thre;
        if (nq) k_map_dynamic<<<(unsigned)ceil_div(nq * 32, 256), 256, 0, st>>>(ctx->A, D);
    }
    k_map_merge<<<kNumClasses, kMapBlock, 0, st>>>(M);
    k_map_sample<<<kNumClasses, kMapBlock, 0, st>>>(M);
    CK(cudaMemcpyAsync(m->h_state, m->d_state, sizeof(MapState), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(m->ev1, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    // the map now lives in the other buffer, in the scan's frame
    m->cur = nxt;
    const MapState &S = *m->h_state;
    const double big = 1.7976931348623157e308;
    double lb[6] = {big, big, big, -big, -big, -big}, gb[6] = {big, big, big, -big, -big, -big};
    for (int c = 0; c < kNumClasses; ++c) {
        m->n[c] = S.n_out[c];
        m->last.n_appended[c] = S.n_appended[c];
        if (S.n_out[c] == 0) continue;
        for (int d = 0; d < 3; ++d) {
            lb[d] = std::min(lb[d], (double)S.lb[c][d]);
            lb[3 + d] = std::max(lb[3 + d], (double)S.lb[c][3 + d]);
            gb[d] = std::min(gb[d], (double)S.gb[c][d]);
            gb[3 + d] = std::max(gb[3 + d], (double)S.gb[c][3 + d]);
        }
    }
    for (int i = 0; i < 6; ++i) m->local_bound[i] = lb[i], m->bound[i] = gb[i];
    for (int i = 0; i < 16; ++i) m->pose[i] = scan_pose_lo[i];
    cudaEventElapsedTime(&m->last.ms_update, m->ev0, m->ev1);
    ++m->epoch;
    ctx->tree_map = nullptr; // :134 free_tree()
    // :95-115 update_cloud_vectors: re-estimate the direction of the map's pillar and beam points from the map itself
    // (PCA over at most 20 neighbours within 1.8 m) and keep the ones that still look like a pillar / a beam. The
    // bounding boxes above are not refreshed (the reference computes them before this step).
    if (P.recalculate_feature_on) {
        const float pca_radius = 1.8f, sin_high_pillar = 0.80f, sin_low_beam = 0.25f, min_linearity = 0.65f;
        const int pca_max_k = 20, pca_min_k = 6;
        const int cls[2] = {MULLS_PILLAR, MULLS_BEAM};
        const float lo[2] = {0.0f, sin_low_beam}, hi[2] = {sin_high_pillar, 1.0f};
        bool any = false;
        for (int k = 0; k < 2; ++k) {
            const int c = cls[k];
            if (!M.used[c] || m->n[c] == 0) continue;
            mulls_cloud_view v{(const float *)m->buf[m->cur][c], m->n[c]};
            PcaArgs args;
            uint64_t launches = 0;
            const size_t nbr_bytes = (size_t)m->n[c] * pca_max_k * sizeof(uint32_t);
            if (nbr_bytes > ctx->cls_buf_bytes) {
                if (ctx->cls_buf) cudaFree(ctx->cls_buf);
                ctx->cls_buf = nullptr;
                ctx->cls_buf_bytes = 0;
                CK(cudaMalloc(&ctx->cls_buf, nbr_bytes));
                ctx->cls_buf_bytes = nbr_bytes;
            }
            const int rc = pca_on_device(ctx, v, true, pca_radius, pca_max_k, 1, args, launches, (uint32_t *)ctx->cls_buf);
            if (rc != MULLS_OK) return rc;
            k_map_revector<<<1, kMapBlock, 0, st>>>(m->buf[m->cur][c], m->n[c], args, pca_min_k, lo[k], hi[k], min_linearity,
                                                   m->mid[c], &m->d_state->n_out[c]);
            std::swap(m->buf[m->cur][c], m->mid[c]);
            any = true;
        }
        if (any) {
            CK(cudaMemcpyAsync(m->h_state, m->d_state, sizeof(MapState), cudaMemcpyDeviceToHost, st));
            CK(cudaEventRecord(m->ev1, st));
            CK(cudaStreamSynchronize(st));
            CK(cudaGetLastError());
            if (ctx->h_flags[1]) {
                ctx->err = "hash pool exhausted";
                return MULLS_E_CAPACITY;
            }
            for (int k = 0; k < 2; ++k) m->n[cls[k]] = m->h_state->n_out[cls[k]];
            cudaEventElapsedTime(&m->last.ms_update, m->ev0, m->ev1);
        }
    }
    if (info) map_fill_info(m, info);
    return MULLS_OK;
}

int mulls_icp_run_to_map(mulls_ctx *ctx, mulls_map *m, const mulls_cloud_view src[MULLS_NUM_CLASSES],
                         const mulls_icp_params *params, const double init_guess[16], mulls_icp_result *out,
                         mulls_icp_trace *trace) {
    if (!ctx || !m || !src || !params || !init_guess) return MULLS_E_ARG;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0];
    if (ctx != m->ctx) {
        ctx->err = "mulls_icp_run_to_map: the map belongs to another context";
        return MULLS_E_ARG;
    }
    mulls_cloud_view tgt[MULLS_NUM_CLASSES];
    for (int c = 0; c < kNumClasses; ++c) {
        tgt[c].aos48 = (const float *)m->buf[m->cur][c];
        tgt[c].n = m->n[c];
    }
    mulls_icp_params P = *params;
    for (int i = 0; i < 6; ++i) P.target_bound[i] = m->local_bound[i]; // block1->local_bound, cregistration.hpp:2916
    int rc = upload_impl(ctx, 1, tgt, src, &P, init_guess, nullptr, nullptr, /*resident=*/false, /*tgt_on_device=*/true);
    if (rc != MULLS_OK) return rc;
    rc = run_impl(ctx, out, trace, nullptr, nullptr);
    ctx->uploaded = false;
    if (rc == MULLS_OK) { // the sorted target slices of this run stand in for block1->tree_*
        ctx->tree_map = m;
        ctx->tree_epoch = m->epoch;
    }
    return rc;
}

// ================================================================================================
// Non-ground feature classification (CFilter::classify_nground_pts, cfilter.hpp:2058-2290)
// ================================================================================================
void mulls_classify_default_params(mulls_classify_params *p) {
    std::memset(p, 0, sizeof(*p));
    p->neighbor_searching_radius = 1.0f;
    p->neighbor_k = 50;
    p->neigh_k_min = 8;
    p->pca_down_rate = 1;
    p->edge_thre = 0.65f;
    p->planar_thre = 0.65f;
    p->edge_thre_down = 0.75f;
    p->planar_thre_down = 0.75f;
    p->extract_vertex_points_method = 2;
    p->curvature_thre = 0.12f;
    p->vertex_curvature_non_max_radius = 1.5f;
    p->linear_vertical_sin_high_thre = 0.94f;
    p->linear_vertical_sin_low_thre = 0.17f;
    p->planar_vertical_sin_high_thre = 0.98f;
    p->planar_vertical_sin_low_thre = 0.34f;
    p->fixed_num_downsampling = 0;
    p->pillar_down_fixed_num = 200;
    p->facade_down_fixed_num = 800;
    p->beam_down_fixed_num = 200;
    p->roof_down_fixed_num = 100;
    p->unground_down_fixed_num = 20000;
    p->beam_height_max = FLT_MAX;
    p->roof_height_min = -FLT_MAX;
    p->feature_pts_ratio_guess = 0.3f;
    p->sharpen_with_nms = 1;
    p->use_distance_adaptive_pca = 0;
    p->random_seed = 0;
}

int mulls_classify_nground(mulls_ctx *ctx, mulls_cloud_view cloud_in, const mulls_classify_params *params,
                           mulls_classify_out *out) {
    if (!ctx || !params || !out || (cloud_in.n > 0 && !cloud_in.aos48)) return MULLS_E_ARG;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0];
    const mulls_classify_params &P = *params;
    if (P.use_distance_adaptive_pca) {
        ctx->err = "mulls_classify_nground: use_distance_adaptive_pca is not implemented";
        return MULLS_E_UNSUPPORTED;
    }
    if (P.neighbor_k < 1 || P.neighbor_k > kPcaListCap || !(P.neighbor_searching_radius > 0.f)) {
        ctx->err = "mulls_classify_nground: neighbor_k must be 1..64 and the radius positive";
        return MULLS_E_ARG;
    }
    for (int k = 0; k < MULLS_OUT_COUNT; ++k) out->n[k] = 0;
    const size_t n0 = cloud_in.n;
    if (n0 == 0) return MULLS_OK;
    if (n0 > ctx->max_tgt) {
        ctx->err = "mulls_classify_nground: cloud exceeds max_tgt_pts of the context";
        return MULLS_E_CAPACITY;
    }
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // :2086-2087 random_downsample_pcl(cloud_in, unground_down_fixed_num): the size it leaves is known up front
    size_t n = n0;
    const bool sample_in = P.fixed_num_downsampling && P.unground_down_fixed_num >= 0 && n0 > (size_t)P.unground_down_fixed_num;
    if (sample_in) n = (size_t)P.unground_down_fixed_num;
    const int stride = P.pca_down_rate > 0 ? P.pca_down_rate : 1;
    // scratch layout
    const size_t row_b = 48;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t o = off;
        off += (bytes + 255) / 256 * 256;
        return o;
    };
    const size_t o_in = take(n0 * row_b), o_rows = take(n0 * row_b);
    size_t o_cls[4], o_srt[4], o_dn[4], o_dn2[4];
    for (int c = 0; c < 4; ++c) o_cls[c] = take(n0 * row_b), o_srt[c] = take(n0 * row_b), o_dn[c] = take(n0 * row_b), o_dn2[c] = take(n0 * row_b);
    const size_t o_sect = take(2 * n0 * row_b), o_vrows = take(n0 * row_b), o_vertex = take(n0 * row_b);
    const size_t o_sel = take(4 * n0 * sizeof(float4)), o_nbr = take(n0 * (size_t)P.neighbor_k * sizeof(uint32_t));
    const size_t o_l0 = take(n0), o_l = take(n0), o_df = take(n0), o_s4 = take(n0), o_vf = take(n0), o_st = take(sizeof(ClsState));
    if (off > ctx->cls_buf_bytes) {
        if (ctx->cls_buf) cudaFree(ctx->cls_buf);
        ctx->cls_buf = nullptr;
        ctx->cls_buf_bytes = 0;
        CK(cudaMalloc(&ctx->cls_buf, off));
        ctx->cls_buf_bytes = off;
    }
    char *base = (char *)ctx->cls_buf;
    ClsArgs C;
    std::memset(&C, 0, sizeof(C));
    C.P = P;
    C.n = (uint32_t)n;
    C.stride = stride;
    C.rows = (float4 *)(base + o_rows);
    for (int c = 0; c < 4; ++c) {
        C.cls[c] = (float4 *)(base + o_cls[c]);
        C.cls_sorted[c] = (float4 *)(base + o_srt[c]);
        C.down[c] = (float4 *)(base + o_dn[c]);
        C.down2[c] = (float4 *)(base + o_dn2[c]);
    }
    C.sect = (float4 *)(base + o_sect);
    C.vrows = (float4 *)(base + o_vrows);
    C.vertex = (float4 *)(base + o_vertex);
    C.sel_pos = (float4 *)(base + o_sel);
    C.label0 = (uint8_t *)(base + o_l0);
    C.label = (uint8_t *)(base + o_l);
    C.downflag = (uint8_t *)(base + o_df);
    C.st4 = (uint8_t *)(base + o_s4);
    C.vflag = (uint8_t *)(base + o_vf);
    C.st = (ClsState *)(base + o_st);
    uint32_t *nbr = (uint32_t *)(base + o_nbr);
    CK(cudaEventRecord(ctx->ev_begin, st));
    CK(cudaMemsetAsync(C.st, 0, sizeof(ClsState), st));
    uint64_t launches = 0;
    if (sample_in) {
        CK(cudaMemcpyAsync(base + o_in, cloud_in.aos48, n0 * row_b, cudaMemcpyDefault, st)); // host or device rows
        k_rows_sample<<<1, kClsBlock, 0, st>>>((const float4 *)(base + o_in), (uint32_t)n0, P.unground_down_fixed_num, P.random_seed,
                                               18u, C.rows);
        ++launches;
    } else {
        CK(cudaMemcpyAsync(C.rows, cloud_in.aos48, n0 * row_b, cudaMemcpyDefault, st));
    }
    ClsState hs;
    std::memset(&hs, 0, sizeof(hs));
    if (n > 0) {
        // :2089-2097 PCA of every pca_down_rate-th point, with the neighbour lists
        mulls_cloud_view v{(const float *)C.rows, n};
        const int rc = pca_on_device(ctx, v, true, P.neighbor_searching_radius, P.neighbor_k, stride, C.F, launches, nbr);
        if (rc != MULLS_OK) return rc;
        C.keys_a = ctx->A.keys_a;
        C.keys_b = ctx->A.keys_b;
        const unsigned gb = (unsigned)ceil_div(n, 256);
        k_cls_label<<<gb, 256, 0, st>>>(C);
        k_cls_compact<<<8, kClsBlock, 0, st>>>(C);
        k_cls_promote_pre<<<gb, 256, 0, st>>>(C);
        k_cls_promote<<<1, kClsBlock, 0, st>>>(C);
        k_cls_promote_apply<<<gb, 256, 0, st>>>(C);
        k_cls_compact2<<<4, kClsBlock, 0, st>>>(C);
        k_cls_encode<<<gb, 256, 0, st>>>(C);
        k_cls_compact_vertex<<<1, kClsBlock, 0, st>>>(C);
        launches += 8;
        if (P.sharpen_with_nms) {
            CK(cudaMemsetAsync(C.keys_a, 0xff, n * sizeof(uint64_t), st));
            k_nms_keys<<<dim3(gb, 4), 256, 0, st>>>(C);
            size_t bytes = ctx->cub_temp_bytes;
            CK(cub::DeviceRadixSort::SortKeys(ctx->cub_temp, bytes, C.keys_a, C.keys_b, (int)n, 0, 64, st));
            k_nms_gather<<<gb, 256, 0, st>>>(C);
            k_nms_select<<<4, kClsBlock, 0, st>>>(C);
            launches += 3;
        }
        if (P.fixed_num_downsampling) {
            k_cls_fixed<<<4, kClsBlock, 0, st>>>(C);
            ++launches;
        }
        CK(cudaMemcpyAsync(&hs, C.st, sizeof(ClsState), cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (n > 0 && ctx->h_flags[1]) {
        ctx->err = "hash pool exhausted";
        return MULLS_E_CAPACITY;
    }
    // results
    const float4 *src[MULLS_OUT_COUNT];
    size_t cnt[MULLS_OUT_COUNT];
    for (int c = 0; c < 4; ++c) {
        src[c] = hs.nms_ran[c] ? C.cls_sorted[c] : C.cls[c];
        cnt[c] = hs.n_cls2[c];
        src[4 + c] = P.fixed_num_downsampling ? C.down2[c] : C.down[c];
        cnt[4 + c] = P.fixed_num_downsampling ? hs.n_down2[c] : hs.n_down[c];
    }
    src[MULLS_OUT_VERTEX] = C.vertex, cnt[MULLS_OUT_VERTEX] = hs.n_vertex;
    src[MULLS_OUT_UNGROUND] = C.rows, cnt[MULLS_OUT_UNGROUND] = n;
    for (int k = 0; k < MULLS_OUT_COUNT; ++k) {
        out->n[k] = cnt[k];
        if (!out->rows[k] || cnt[k] == 0) continue;
        if (cnt[k] > out->cap) {
            ctx->err = "mulls_classify_nground: output buffer too small";
            return MULLS_E_CAPACITY;
        }
        CK(cudaMemcpyAsync(out->rows[k], src[k], cnt[k] * row_b, cudaMemcpyDefault, st));
    }
    CK(cudaEventRecord(ctx->ev_end, st));
    CK(cudaStreamSynchronize(st));
    ctx->stats = mulls_run_stats();
    ctx->stats.kernel_launches = launches;
    cudaEventElapsedTime(&ctx->stats.ms_total, ctx->ev_begin, ctx->ev_end);
    return MULLS_OK;
}

} // extern "C"

// ------------------------------------------------------------------------------------------------
// Ground segmentation (CFilter::fast_ground_filter, cfilter.hpp:1658-2036)
// ------------------------------------------------------------------------------------------------
namespace {
// first kSacDraws outputs of boost::mt19937 seeded with 12345u (every pcl::SampleConsensusModel object starts there)
const uint32_t *sac_draw_table() {
    static std::vector<uint32_t> tab;
    if (tab.empty()) {
        std::vector<uint32_t> t(kSacDraws);
        uint32_t mt[624];
        mt[0] = 12345u;
        for (int i = 1; i < 624; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
        int idx = 624;
        for (int k = 0; k < kSacDraws; ++k) {
            if (idx >= 624) {
                for (int i = 0; i < 624; ++i) {
                    const uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7fffffffu);
                    mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
                }
                idx = 0;
            }
            uint32_t y = mt[idx++];
            y ^= y >> 11;
            y ^= (y << 7) & 0x9d2c5680u;
            y ^= (y << 15) & 0xefc60000u;
            y ^= y >> 18;
            t[k] = y;
        }
        tab.swap(t);
    }
    return tab.data();
}
int host_ord(float f) {
    int i;
    std::memcpy(&i, &f, 4);
    return i >= 0 ? i : (i ^ 0x7fffffff);
}
} // namespace

extern "C" {

void mulls_ground_default_params(mulls_ground_params *p) { // extract_semantic_pts as test/mulls_slam.cpp calls it (gflags :78-104)
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->min_grid_pt_num = 10;
    p->grid_resolution = 3.0f;
    p->max_height_difference = 0.3f;
    p->neighbor_height_diff = 1.5f;
    p->max_ground_height = 5.0f;
    p->ground_random_down_rate = 15;
    p->ground_random_down_down_rate = 2;
    p->nonground_random_down_rate = 3;
    p->reliable_neighbor_grid_num_thre = 0;
    p->estimate_ground_normal_method = 3;
    p->normal_estimation_radius = 2.0f;
    p->distance_weight_downsampling_method = 2;
    p->standard_distance = 15.0f;
    p->fixed_num_downsampling = 0;
    p->down_ground_fixed_num = 300;
    p->intensity_thre = FLT_MAX;
    p->apply_grid_wise_outlier_filter = 0;
    p->outlier_std_scale = 3.0f;
    p->random_seed = 0;
}

int mulls_fast_ground_filter(mulls_ctx *ctx, mulls_cloud_view cloud_in, const mulls_ground_params *params,
                             mulls_ground_out *out) {
    if (!ctx || !params || !out || (cloud_in.n > 0 && !cloud_in.aos48)) return MULLS_E_ARG;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0];
    const mulls_ground_params &P = *params;
    if (P.estimate_ground_normal_method != 0 && P.estimate_ground_normal_method != 3) {
        ctx->err = "mulls_fast_ground_filter: estimate_ground_normal_method 1 / 2 (pcl::NormalEstimation) are not implemented";
        return MULLS_E_UNSUPPORTED;
    }
    if (P.ground_random_down_rate < 1 || P.nonground_random_down_rate < 1 || P.ground_random_down_down_rate < 1 ||
        !(P.grid_resolution > 0.f)) {
        ctx->err = "mulls_fast_ground_filter: the down-sampling rates must be >= 1 and grid_resolution positive";
        return MULLS_E_ARG;
    }
    out->n_ground = out->n_ground_down = out->n_unground = 0;
    const size_t n = cloud_in.n;
    if (n == 0) return MULLS_OK;
    if (n > ctx->max_tgt || n >= (1ull << 31)) {
        ctx->err = "mulls_fast_ground_filter: cloud exceeds max_tgt_pts of the context";
        return MULLS_E_CAPACITY;
    }
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // temporary storage of the library sort / scans
    size_t sort_bytes = 0, scan_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (uint32_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr,
                                    (uint32_t *)nullptr, (int)n, 0, 32, st);
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (uint32_t *)nullptr, (uint32_t *)nullptr, (int)n, st);
    // per-point scratch
    const size_t row_b = 48;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t o = off;
        off += (bytes + 255) / 256 * 256;
        return o;
    };
    const size_t o_rows = take(n * row_b), o_g = take(n * row_b), o_gd = take(n * row_b), o_u = take(n * row_b);
    const size_t o_key = take(4 * n), o_idx = take(4 * n), o_keys = take(4 * n), o_idxs = take(4 * n), o_call = take(4 * n);
    const size_t o_hf = take(4 * n), o_hp = take(4 * n), o_dec = take(n), o_cand = take(16 * n), o_shuf = take(4 * n), o_inl = take(n);
    const size_t o_st = take(sizeof(GfState)), o_draws = take(kSacDraws * sizeof(uint32_t));
    const size_t o_tmp = take(std::max(sort_bytes, scan_bytes));
    if (off > ctx->gf_buf_bytes) {
        if (ctx->gf_buf) cudaFree(ctx->gf_buf);
        ctx->gf_buf = nullptr;
        ctx->gf_buf_bytes = 0;
        CK(cudaMalloc(&ctx->gf_buf, off));
        ctx->gf_buf_bytes = off;
    }
    char *base = (char *)ctx->gf_buf;
    GfArgs A;
    std::memset(&A, 0, sizeof(A));
    A.P = P;
    A.n = (uint32_t)n;
    A.rows = (const float4 *)(base + o_rows);
    A.out_ground = (float4 *)(base + o_g);
    A.out_ground_down = (float4 *)(base + o_gd);
    A.out_unground = (float4 *)(base + o_u);
    A.key = (uint32_t *)(base + o_key), A.idx = (uint32_t *)(base + o_idx);
    A.key_s = (uint32_t *)(base + o_keys), A.idx_s = (uint32_t *)(base + o_idxs);
    A.cell_all = (int *)(base + o_call);
    A.high_flag = (uint32_t *)(base + o_hf), A.high_pos = (uint32_t *)(base + o_hp);
    A.decision = (uint8_t *)(base + o_dec);
    A.cand = (float4 *)(base + o_cand);
    A.shuf = (int *)(base + o_shuf);
    A.inl = (uint8_t *)(base + o_inl);
    A.st = (GfState *)(base + o_st);
    A.draws = (const uint32_t *)(base + o_draws);
    void *tmp = base + o_tmp;
    size_t tmp_bytes = std::max(sort_bytes, scan_bytes);
    CK(cudaEventRecord(ctx->ev_begin, st));
    CK(cudaMemcpyAsync((void *)A.rows, cloud_in.aos48, n * row_b, cudaMemcpyDefault, st)); // host or device rows
    CK(cudaMemcpyAsync((void *)A.draws, sac_draw_table(), kSacDraws * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    GfState hs;
    std::memset(&hs, 0, sizeof(hs));
    hs.bb[0] = hs.bb[1] = host_ord(FLT_MAX);
    hs.bb[2] = hs.bb[3] = host_ord(-FLT_MAX);
    CK(cudaMemcpyAsync(A.st, &hs, sizeof(GfState), cudaMemcpyHostToDevice, st));
    uint64_t launches = 0;
    const unsigned pb = (unsigned)ceil_div(n, kGfBlock);
    k_gf_bbox<<<pb, kGfBlock, 0, st>>>(A);
    k_gf_setup<<<1, 32, 0, st>>>(A);
    launches += 2;
    CK(cudaMemcpyAsync(&hs, A.st, sizeof(GfState), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (hs.num_grid < 0 || hs.num_grid > (1 << 26)) {
        ctx->err = "mulls_fast_ground_filter: the cloud spans more than 2^26 grid cells (outliers far from the scan?)";
        return MULLS_E_CAPACITY;
    }
    const int num_grid = hs.num_grid;
    if (num_grid > 0) { // (a degenerate cloud with zero extent along x or y has no cell: every point fails the id test)
        const size_t g = (size_t)num_grid;
        size_t coff = 0;
        auto ctake = [&](size_t bytes) {
            const size_t o = coff;
            coff += (bytes + 255) / 256 * 256;
            return o;
        };
        const size_t c_start = ctake(4 * g), c_end = ctake(4 * g), c_minz = ctake(4 * g), c_nb = ctake(4 * g), c_oth = ctake(4 * g);
        const size_t c_rel = ctake(4 * g), c_nrm = ctake(16 * g), c_ng = ctake(4 * g), c_nu = ctake(4 * g), c_og = ctake(4 * g),
                     c_ou = ctake(4 * g);
        size_t cscan = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, cscan, (uint32_t *)nullptr, (uint32_t *)nullptr, num_grid, st);
        const size_t c_tmp = ctake(cscan);
        if (coff > ctx->gf_cell_buf_bytes) {
            if (ctx->gf_cell_buf) cudaFree(ctx->gf_cell_buf);
            ctx->gf_cell_buf = nullptr;
            ctx->gf_cell_buf_bytes = 0;
            CK(cudaMalloc(&ctx->gf_cell_buf, coff));
            ctx->gf_cell_buf_bytes = coff;
        }
        char *cb = (char *)ctx->gf_cell_buf;
        A.cell_start = (uint32_t *)(cb + c_start), A.cell_end = (uint32_t *)(cb + c_end);
        A.min_z = (float *)(cb + c_minz), A.neighbor_min_z = (float *)(cb + c_nb), A.outlier_thre = (float *)(cb + c_oth);
        A.reliable = (int *)(cb + c_rel);
        A.cell_normal = (float4 *)(cb + c_nrm);
        A.cell_ng = (uint32_t *)(cb + c_ng), A.cell_nu = (uint32_t *)(cb + c_nu);
        A.cell_og = (uint32_t *)(cb + c_og), A.cell_ou = (uint32_t *)(cb + c_ou);
        void *ctmp = cb + c_tmp;
        CK(cudaMemsetAsync(A.cell_start, 0, 4 * g, st));
        CK(cudaMemsetAsync(A.cell_end, 0, 4 * g, st));
        const unsigned wb = (unsigned)ceil_div(g * 32, kGfBlock), cbk = (unsigned)ceil_div(g, kGfBlock);
        k_gf_assign<<<pb, kGfBlock, 0, st>>>(A);
        size_t b1 = tmp_bytes;
        CK(cub::DeviceRadixSort::SortPairs(tmp, b1, A.key, A.key_s, A.idx, A.idx_s, (int)n, 0, 32, st));
        k_gf_bounds<<<pb, kGfBlock, 0, st>>>(A);
        k_gf_cell_min<<<wb, kGfBlock, 0, st>>>(A, num_grid);
        k_gf_neighbors<<<cbk, kGfBlock, 0, st>>>(A, num_grid);
        k_gf_high<<<pb, kGfBlock, 0, st>>>(A);
        size_t b2 = tmp_bytes;
        CK(cub::DeviceScan::ExclusiveSum(tmp, b2, A.high_flag, A.high_pos, (int)n, st));
        k_gf_high_emit<<<pb, kGfBlock, 0, st>>>(A);
        k_gf_cell_decide<<<wb, kGfBlock, 0, st>>>(A, num_grid);
        size_t b3 = cscan;
        CK(cub::DeviceScan::ExclusiveSum(ctmp, b3, A.cell_ng, A.cell_og, num_grid, st));
        b3 = cscan;
        CK(cub::DeviceScan::ExclusiveSum(ctmp, b3, A.cell_nu, A.cell_ou, num_grid, st));
        k_gf_totals<<<1, 1, 0, st>>>(A, num_grid);
        k_gf_cell_emit<<<wb, kGfBlock, 0, st>>>(A, num_grid);
        k_gf_down<<<1, kClsBlock, 0, st>>>(A);
        launches += 11;
        CK(cudaMemcpyAsync(&hs, A.st, sizeof(GfState), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
        out->n_ground = hs.n_ground, out->n_ground_down = hs.n_ground_down, out->n_unground = hs.n_unground;
        if (hs.n_ground > out->cap || hs.n_unground > out->cap) {
            ctx->err = "mulls_fast_ground_filter: output buffer too small";
            return MULLS_E_CAPACITY;
        }
        if (out->ground && hs.n_ground)
            CK(cudaMemcpyAsync(out->ground, A.out_ground, hs.n_ground * row_b, cudaMemcpyDefault, st));
        if (out->ground_down && hs.n_ground_down)
            CK(cudaMemcpyAsync(out->ground_down, A.out_ground_down, hs.n_ground_down * row_b, cudaMemcpyDefault, st));
        if (out->unground && hs.n_unground)
            CK(cudaMemcpyAsync(out->unground, A.out_unground, hs.n_unground * row_b, cudaMemcpyDefault, st));
    }
    CK(cudaEventRecord(ctx->ev_end, st));
    CK(cudaStreamSynchronize(st));
    ctx->stats = mulls_run_stats();
    ctx->stats.kernel_launches = launches;
    cudaEventElapsedTime(&ctx->stats.ms_total, ctx->ev_begin, ctx->ev_end);
    return MULLS_OK;
}

} // extern "C"

// ------------------------------------------------------------------------------------------------
// CFilter::voxel_downsample (cfilter.hpp:83-165) and the chain of CFilter::extract_semantic_pts (:2295-2413)
// ------------------------------------------------------------------------------------------------
extern "C" {

int mulls_voxel_downsample(mulls_ctx *ctx, mulls_cloud_view cloud_in, float voxel_size, float *out, size_t cap, size_t *n_out) {
    if (!ctx || !n_out || (cloud_in.n > 0 && (!cloud_in.aos48 || !out))) return MULLS_E_ARG;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0];
    *n_out = 0;
    const size_t n = cloud_in.n;
    if (n == 0) return MULLS_OK;
    if (n > ctx->max_tgt || n >= (1ull << 31)) {
        ctx->err = "mulls_voxel_downsample: cloud exceeds max_tgt_pts of the context";
        return MULLS_E_CAPACITY;
    }
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t row_b = 48;
    if (voxel_size < 0.001) { // :89-97 disabled: cloud_out = cloud_in
        if (n > cap) {
            ctx->err = "mulls_voxel_downsample: output buffer too small";
            return MULLS_E_CAPACITY;
        }
        CK(cudaMemcpyAsync(out, cloud_in.aos48, n * row_b, cudaMemcpyDefault, st));
        CK(cudaStreamSynchronize(st));
        *n_out = n;
        return MULLS_OK;
    }
    size_t sort_bytes = 0, scan_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (uint32_t *)nullptr, (uint32_t *)nullptr, (int)n, 0, 64, st);
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (uint32_t *)nullptr, (uint32_t *)nullptr, (int)n, st);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t o = off;
        off += (bytes + 255) / 256 * 256;
        return o;
    };
    const size_t o_rows = take(n * row_b), o_out = take(n * row_b), o_key = take(8 * n), o_keys = take(8 * n);
    const size_t o_idx = take(4 * n), o_idxs = take(4 * n), o_head = take(4 * n), o_pos = take(4 * n), o_st = take(sizeof(VxState));
    const size_t o_tmp = take(std::max(sort_bytes, scan_bytes));
    if (off > ctx->vx_buf_bytes) {
        if (ctx->vx_buf) cudaFree(ctx->vx_buf);
        ctx->vx_buf = nullptr;
        ctx->vx_buf_bytes = 0;
        CK(cudaMalloc(&ctx->vx_buf, off));
        ctx->vx_buf_bytes = off;
    }
    char *base = (char *)ctx->vx_buf;
    VxArgs V;
    V.n = (uint32_t)n;
    V.voxel_size = voxel_size;
    V.rows = (const float4 *)(base + o_rows);
    V.out = (float4 *)(base + o_out);
    V.key = (unsigned long long *)(base + o_key), V.key_s = (unsigned long long *)(base + o_keys);
    V.idx = (uint32_t *)(base + o_idx), V.idx_s = (uint32_t *)(base + o_idxs);
    V.head = (uint32_t *)(base + o_head), V.pos = (uint32_t *)(base + o_pos);
    V.st = (VxState *)(base + o_st);
    void *tmp = base + o_tmp;
    const size_t tmp_bytes = std::max(sort_bytes, scan_bytes);
    VxState hs;
    std::memset(&hs, 0, sizeof(hs));
    for (int d = 0; d < 3; ++d) hs.bb[d] = host_ord(FLT_MAX), hs.bb[3 + d] = host_ord(-FLT_MAX);
    CK(cudaEventRecord(ctx->ev_begin, st));
    CK(cudaMemcpyAsync((void *)V.rows, cloud_in.aos48, n * row_b, cudaMemcpyDefault, st));
    CK(cudaMemcpyAsync(V.st, &hs, sizeof(VxState), cudaMemcpyHostToDevice, st));
    const unsigned pb = (unsigned)ceil_div(n, kGfBlock);
    k_vx_bbox<<<pb, kGfBlock, 0, st>>>(V);
    k_vx_setup<<<1, 1, 0, st>>>(V);
    k_vx_keys<<<pb, kGfBlock, 0, st>>>(V);
    size_t b1 = tmp_bytes;
    CK(cub::DeviceRadixSort::SortPairs(tmp, b1, V.key, V.key_s, V.idx, V.idx_s, (int)n, 0, 64, st));
    k_vx_heads<<<pb, kGfBlock, 0, st>>>(V);
    size_t b2 = tmp_bytes;
    CK(cub::DeviceScan::ExclusiveSum(tmp, b2, V.head, V.pos, (int)n, st));
    k_vx_gather<<<pb, kGfBlock, 0, st>>>(V);
    CK(cudaMemcpyAsync(&hs, V.st, sizeof(VxState), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    *n_out = hs.n_out;
    if (hs.n_out > cap) {
        ctx->err = "mulls_voxel_downsample: output buffer too small";
        return MULLS_E_CAPACITY;
    }
    CK(cudaMemcpyAsync(out, V.out, (size_t)hs.n_out * row_b, cudaMemcpyDefault, st));
    CK(cudaEventRecord(ctx->ev_end, st));
    CK(cudaStreamSynchronize(st));
    ctx->stats = mulls_run_stats();
    ctx->stats.kernel_launches = 5;
    cudaEventElapsedTime(&ctx->stats.ms_total, ctx->ev_begin, ctx->ev_end);
    return MULLS_OK;
}

int mulls_extract_semantic_pts(mulls_ctx *ctx, mulls_cloud_view pc_raw, const mulls_extract_params *params,
                               mulls_extract_out *out) {
    if (!ctx || !params || !out || (pc_raw.n > 0 && !pc_raw.aos48)) return MULLS_E_ARG;
    if (!ctx->lanes.empty()) ctx = ctx->lanes[0];
    out->n_down = out->n_ground = out->n_ground_down = 0;
    for (int k = 0; k < MULLS_OUT_COUNT; ++k) out->cls.n[k] = 0;
    const size_t n = pc_raw.n;
    if (n == 0) return MULLS_OK;
    if ((out->pc_down || out->pc_ground || out->pc_ground_down) && out->cap < n) {
        ctx->err = "mulls_extract_semantic_pts: the output buffers must hold pc_raw.n rows";
        return MULLS_E_ARG;
    }
    CK(cudaSetDevice(ctx->device));
    // the clouds handed from stage to stage stay in HBM: pc_down and the ground filter's cloud_unground
    const size_t row_b = 48, need = 2 * n * row_b;
    if (need > ctx->ext_buf_bytes) {
        if (ctx->ext_buf) cudaFree(ctx->ext_buf);
        ctx->ext_buf = nullptr;
        ctx->ext_buf_bytes = 0;
        CK(cudaMalloc(&ctx->ext_buf, need));
        ctx->ext_buf_bytes = need;
    }
    float *d_down = (float *)ctx->ext_buf, *d_ung = (float *)((char *)ctx->ext_buf + n * row_b);
    float ms = 0.f;
    uint64_t launches = 0;
    // :2346 voxel_downsample(pc_raw, pc_down) (pc_sketch, :2348, is not a feature cloud and is not produced)
    size_t n_down = 0;
    int rc = mulls_voxel_downsample(ctx, pc_raw, params->vf_downsample_resolution, d_down, n, &n_down);
    if (rc != MULLS_OK) return rc;
    ms += ctx->stats.ms_total, launches += ctx->stats.kernel_launches;
    out->n_down = n_down;
    if (out->pc_down && n_down) {
        CK(cudaMemcpyAsync(out->pc_down, d_down, n_down * row_b, cudaMemcpyDefault, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    // :2355-2361 fast_ground_filter(pc_down -> pc_ground, pc_ground_down, pc_unground)
    mulls_ground_out g;
    std::memset(&g, 0, sizeof(g));
    g.ground = out->pc_ground, g.ground_down = out->pc_ground_down, g.unground = d_ung;
    g.cap = n;
    rc = mulls_fast_ground_filter(ctx, mulls_cloud_view{d_down, n_down}, &params->ground, &g);
    if (rc != MULLS_OK) return rc;
    ms += ctx->stats.ms_total, launches += ctx->stats.kernel_launches;
    out->n_ground = g.n_ground, out->n_ground_down = g.n_ground_down;
    // :2378-2391 classify_nground_pts(pc_unground -> pillar, beam, facade, roof, their down clouds, vertex)
    rc = mulls_classify_nground(ctx, mulls_cloud_view{d_ung, g.n_unground}, &params->classify, &out->cls);
    if (rc != MULLS_OK) return rc;
    ms += ctx->stats.ms_total, launches += ctx->stats.kernel_launches;
    ctx->stats.ms_total = ms;
    ctx->stats.kernel_launches = launches;
    return MULLS_OK;
}

} // extern "C"
