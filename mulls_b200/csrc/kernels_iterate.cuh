// Iteration phase: one pass of the loop body of mm_lls_icp (cregistration.hpp:1239-1401) as four kernels; the first
// three run over (pair, class, 128-source chunk) work items, the fourth over pairs:
//   k_search      I1+I2a  apply the previous increment to the source (:1260), exact radius-bounded 1-NN on the hashed
//                         multi-level grid (replaces the kd-tree query of :1745), claim the target
//   k_resolve     I2b     duplicate check (:1755-1792), distance rejector (:1794-1796), normal check (:1798-1830),
//                         per-class correspondence counts
//   k_accumulate  I3-I5   order-preserving source compaction (:1776-1789), 21+6 normal-equation terms per
//                         correspondence (:1976-2275), fixed-order block reduction -> one partial per chunk
//   k_solve       I5-I9   per pair: partials summed in chunk order, 6x6 solve, Euler/Jacobian, convergence and
//                         status logic (:1301-1400) — the iteration driver lives on the device
// After the loop: k_posterior + k_finalize (:2518-2677, :1386). Source-sharded registrations (k_shard_*) insert the
// caller's all-reduce between these phases.
#pragma once
#include <cooperative_groups.h>

#include "device_math.cuh"
#include "device_types.cuh"
#include "kernels_ingest.cuh"

namespace mulls {

// kernels recorded into the iteration graph are launched over the context's CAPACITY and take the double-buffer index
// from the device-side loop counter (buf < 0); the host loop passes exact grids and buf = it & 1
__device__ __forceinline__ bool chunk_in_run(const DeviceArrays &A) { return blockIdx.x < (unsigned)A.ctl->n_it_chunks; }
__device__ __forceinline__ int loop_buf(const DeviceArrays &A, int buf) { return buf >= 0 ? buf : (A.ctl->it & 1); }
__device__ __forceinline__ mulls_icp_trace *trace_of(const DeviceArrays &A, uint32_t pair) {
    return (A.trace && A.ctl->trace_on) ? &A.trace[pair] : nullptr;
}

// The iteration kernels run a fixed number of resident blocks; each block fetches positions of the live-chunk list of
// this iteration (LoopCtl::n_live / work, device_types.cuh) until the list is exhausted. `body(chunk)` is executed by
// the whole block; a body may leave early per thread, but only before any barrier it contains.
template <class Body>
__device__ __forceinline__ void for_each_live_chunk(const DeviceArrays &A, int parity, int which, Body body) {
    __shared__ uint32_t s_fetch;
    LoopCtl &ctl = *A.ctl;
    const uint32_t n = ctl.n_live[parity];
    const uint32_t *list = A.live_chunks + (size_t)parity * A.live_stride;
    for (;;) {
        __syncthreads(); // the previous chunk is finished with and s_fetch has been read by everyone
        if (threadIdx.x == 0) s_fetch = atomicAdd(&ctl.work[which], 1u);
        __syncthreads();
        const uint32_t w = s_fetch;
        if (w >= n) break;
        body(list[w]);
    }
}

// warp-aggregated append of the chunks [first, first + count) of one (pair, class) to a live list
__device__ __forceinline__ void append_live_chunks(const DeviceArrays &A, int parity, uint32_t first, uint32_t count, uint32_t base) {
    uint32_t *list = A.live_chunks + (size_t)parity * A.live_stride;
    for (uint32_t k = threadIdx.x; k < count; k += blockDim.x) list[base + k] = first + k;
}

// after the ingest: the chunks that own at least one source point form the list of iteration 0
__global__ void __launch_bounds__(256) k_live_init(DeviceArrays A) {
    LoopCtl &ctl = *A.ctl;
    const uint32_t chunk = blockIdx.x * blockDim.x + threadIdx.x;
    bool live = false;
    if (chunk < (uint32_t)ctl.n_it_chunks) {
        const ChunkDesc cd = A.it_chunks[chunk];
        live = (int)cd.first < A.ps[cd.pair].n_src[cd.seg];
    }
    const unsigned m = __ballot_sync(0xffffffffu, live);
    if (!m) return;
    const int lane = threadIdx.x & 31;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(&ctl.n_live[0], (unsigned)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (live) A.live_chunks[base + __popc(m & ((1u << lane) - 1u))] = chunk;
}

// ------------------------------------------------------------------------------------------------
// exact 1-NN within radius on the multi-level hashed grid of one target class: search_core.cuh
// (__host__ __device__; the CPU suite runs the same functions against a brute-force scan)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ GridView grid_of(const DeviceArrays &A, const PairConst &pc, const PairState &ps, int c, int leaf_count) {
    GridView g;
    g.table = A.hash + ps.hash_base[c];
    g.mask = ps.hash_mask[c];
    g.pos = A.tgt_pos + pc.tgt_base[c];
    g.nrm = A.tgt_nrm + pc.tgt_base[c];
    g.ox = ps.origin[0], g.oy = ps.origin[1], g.oz = ps.origin[2];
    g.h0 = ps.h0, g.inv_h0 = ps.inv_h0;
    g.n_levels = ps.n_levels;
    g.leaf_count = leaf_count;
    g.level_slack2 = 1.002001f;
    return g;
}

// squared distance from p to the (slightly inflated) box of cell (x,y,z) at a level with cell size hl
__device__ __forceinline__ float cell_dist2(const GridView &g, float px, float py, float pz, float hl, int x, int y,
                                            int z, float margin) {
    const float ax = slab_dist(g.ox + (float)x * hl, g.ox + (float)(x + 1) * hl, px, margin);
    const float ay = slab_dist(g.oy + (float)y * hl, g.oy + (float)(y + 1) * hl, py, margin);
    const float az = slab_dist(g.oz + (float)z * hl, g.oz + (float)(z + 1) * hl, pz, margin);
    return ax * ax + ay * ay + az * az;
}

// ------------------------------------------------------------------------------------------------
// exact k nearest targets (k = 10) for the normal-shooting correspondences of :1732-1737
// (pcl::registration::CorrespondenceEstimationNormalShooting): same hierarchy as nn_search, the pruning bound is
// the current k-th best distance and there is no search radius — the level pyramid of a pair that uses normal
// shooting goes up to a block that spans the whole grid, so the result is exact however far the targets are.
// Total order (d2, original index). A rarely used option: plain per-thread DFS with its stack in local memory,
// kept out of k_search (own kernel, k_search_shoot).
// ------------------------------------------------------------------------------------------------
constexpr int kShootK = 10;
constexpr int kShootStack = 48; // DFS entries: at most 7 stay behind per descended level

struct KnnList {
    float d2[kShootK];
    int j[kShootK];
    int n;
};
__device__ __forceinline__ float knn_bound(const KnnList &kl) { return kl.n < kShootK ? INFINITY : kl.d2[kShootK - 1]; }

__device__ __forceinline__ void knn_insert(const GridView &g, KnnList &kl, float d2, int j) {
    if (kl.n == kShootK) {
        const float w = kl.d2[kShootK - 1];
        if (d2 > w) return;
        if (d2 == w && __float_as_int(__ldg(&g.nrm[j]).w) >= __float_as_int(__ldg(&g.nrm[kl.j[kShootK - 1]]).w)) return;
    }
    for (int i = 0; i < kl.n; ++i)
        if (kl.j[i] == j) return; // a point is met again when the search ascends a level
    int pos = (kl.n < kShootK) ? kl.n : kShootK - 1;
    while (pos > 0) {
        const float dp = kl.d2[pos - 1];
        bool before = d2 < dp;
        if (d2 == dp) before = __float_as_int(__ldg(&g.nrm[j]).w) < __float_as_int(__ldg(&g.nrm[kl.j[pos - 1]]).w);
        if (!before) break;
        kl.d2[pos] = kl.d2[pos - 1];
        kl.j[pos] = kl.j[pos - 1];
        --pos;
    }
    kl.d2[pos] = d2;
    kl.j[pos] = j;
    if (kl.n < kShootK) ++kl.n;
}

__device__ __forceinline__ void knn_search(const GridView &g, float px, float py, float pz, int start_level, KnnList &kl) {
    kl.n = 0;
    const int c0x = (int)floorf((px - g.ox) * g.inv_h0);
    const int c0y = (int)floorf((py - g.oy) * g.inv_h0);
    const int c0z = (int)floorf((pz - g.oz) * g.inv_h0);
    const int L = g.n_levels;
    const float margin = 1e-3f * g.h0;
    uint2 st_cell[kShootStack]; // pack_cell(x, y, z, level, 0)
    float st_d2[kShootStack];
    for (int l = min(max(start_level, 1), L - 1);; ++l) {
        const float H = g.h0 * (float)(1 << l);
        const int ncell = (1 << kCoordBits) >> l;
        for (int k = 0; k < 8; ++k) { // own cell first, then the half-side neighbours
            int x = (c0x >> l) + ((k & 1) ? ((((c0x >> (l - 1)) & 1) ? 1 : -1)) : 0);
            int y = (c0y >> l) + ((k & 2) ? ((((c0y >> (l - 1)) & 1) ? 1 : -1)) : 0);
            int z = (c0z >> l) + ((k & 4) ? ((((c0z >> (l - 1)) & 1) ? 1 : -1)) : 0);
            if (ncell == 2) x = k & 1, y = (k >> 1) & 1, z = k >> 2; // top of the full pyramid: the 8 cells ARE the grid
            if (x < 0 || y < 0 || z < 0 || x >= ncell || y >= ncell || z >= ncell) continue;
            int sp = 0;
            st_cell[0] = pack_cell((uint32_t)x, (uint32_t)y, (uint32_t)z, l, 0u);
            st_d2[0] = cell_dist2(g, px, py, pz, H, x, y, z, margin);
            sp = 1;
            while (sp > 0) {
                --sp;
                if (st_d2[sp] > knn_bound(kl) * 1.0001f + 1e-12f) continue;
                const uint2 ce = st_cell[sp];
                const int lv = (int)((ce.y >> 4) & 0xfu);
                const int cx = (int)(ce.x & 0xfffu), cy = (int)((ce.x >> 12) & 0xfffu), cz = (int)((ce.x >> 24) | ((ce.y & 0xfu) << 8));
                uint32_t start, count, cmask;
                if (!probe_cell(g, (uint32_t)cx, (uint32_t)cy, (uint32_t)cz, lv, start, count, cmask)) continue;
                if (count <= (uint32_t)g.leaf_count || lv == 0 || sp + 8 > kShootStack) {
                    for (uint32_t jj = start; jj < start + count; ++jj) {
                        const float4 q = __ldg(&g.pos[jj]);
                        knn_insert(g, kl, flann_l2(px, py, pz, q.x, q.y, q.z), (int)jj);
                    }
                } else {
                    const float hc = 0.5f * g.h0 * (float)(1 << lv);
                    for (int ch = 7; ch >= 0; --ch) {
                        if (!((cmask >> ch) & 1u)) continue;
                        const int x2 = 2 * cx + (ch & 1), y2 = 2 * cy + ((ch >> 1) & 1), z2 = 2 * cz + (ch >> 2);
                        const float d2c = cell_dist2(g, px, py, pz, hc, x2, y2, z2, margin);
                        if (d2c > knn_bound(kl) * 1.0001f + 1e-12f) continue;
                        st_cell[sp] = pack_cell((uint32_t)x2, (uint32_t)y2, (uint32_t)z2, lv - 1, 0u);
                        st_d2[sp] = d2c;
                        ++sp;
                    }
                }
            }
        }
        const float cover = 0.999f * 0.5f * H; // every target closer than this has been examined
        if (kl.n == kShootK && kl.d2[kShootK - 1] <= cover * cover) break;
        if (l == L - 1) break; // the top block spans the whole grid: everything has been examined
    }
}

// ---- k_search ----------------------------------------------------------------------------------
// what every search kernel does first: cregistration.hpp:1260 — incremental in-place update of the float source
// cloud by the previous iteration's TempTran (double math, float store, as pcl::transformPointCloudWithNormals)
__device__ __forceinline__ void load_and_advance(DeviceArrays &A, const PairState &ps, int buf, uint32_t gi, bool valid,
                                                 float4 &p, float4 &n) {
    p = A.src_pos[buf][gi];
    n = A.src_nrm[buf][gi];
    if (valid && ps.iter > 0) {
        const double *t = ps.T_inc;
        const double px = p.x, py = p.y, pz = p.z, qx = n.x, qy = n.y, qz = n.z;
        p.x = (float)(t[0] * px + t[1] * py + t[2] * pz + t[3]);
        p.y = (float)(t[4] * px + t[5] * py + t[6] * pz + t[7]);
        p.z = (float)(t[8] * px + t[9] * py + t[10] * pz + t[11]);
        n.x = (float)(t[0] * qx + t[1] * qy + t[2] * qz);
        n.y = (float)(t[4] * qx + t[5] * qy + t[6] * qz);
        n.z = (float)(t[8] * qx + t[9] * qy + t[10] * qz);
        A.src_pos[buf][gi] = p;
        A.src_nrm[buf][gi] = n;
    }
}

// shoot = 0: every class except the normal-shooting ones; shoot = 1 (k_search_shoot): only those
__device__ __forceinline__ bool shoots(const PairConst &pc, int c) {
    return pc.normal_shooting && (c == MULLS_GROUND || c == MULLS_FACADE || c == MULLS_ROOF);
}

// ---- k_search: I1 + I2a of the iteration — apply the previous increment to the source (:1260), exact
//      radius-bounded 1-NN on the hashed multi-level grid (nn_search_walk, search_core.cuh — replaces the kd-tree query
//      of :1745), claim the target for the duplicate check. Resident blocks fetch their work from the live list.
// Iterations 0 .. kKeepFromIter-1 ("direct"): work unit = a quarter chunk (32 sources) per WARP, one query per lane,
//   no cooperation and no barrier; the last of them also leaves a certificate per query (src_cert: where the query
//   stood, and a radius inside which its match is the only target).
// From iteration kKeepFromIter on ("keep"): work unit = a chunk per BLOCK, two passes:
//   A  every source: transform, then try to KEEP the previous match without a search: if |p - q| + |p - p_ref| stays
//      below the certificate radius, q is still the unique nearest target and its distance is computed directly (the
//      result a search would return, bit for bit). Queries that cannot be kept are listed in shared memory;
//   B  the listed queries, densely packed into the first threads of the block: seeded exact search, new certificate.
//   Late iterations keep most matches (measured on the C2 pair: 41 / 54 / 86 % in iterations 3 / 4 / 5; ~100 % once
//   converged), and what is kept costs the streaming pass A only. (A variant with pass B fed from ONE queue in HBM —
//   dense warps whatever chunk a source comes from, no barrier — measured slower: 0.58 / 0.46 / 0.28 ms against
//   0.37 / 0.28 / 0.16 for iterations 3 / 4 / 5; the queue interleaves chunks, and the locality of a warp's 32 queries
//   is worth more than its density.)
constexpr int kKeepFromIter = 3;
// search parameters (profiles/r2_search_ab_scan4_occupancy.txt: other deferral iterations and reseed distances are
// no faster)
constexpr int kStartLevel = 5;       // grid level at which a walk starts
constexpr int kDeferFromIter = 3;    // from this iteration on a block queues its small cells (one scan loop per block)
constexpr float kReseedCells = 4.0f; // a previous match farther than this many level-0 cells is challenged by a greedy descent

struct SearchArgs {
    int leaf_count;
};

// what is fixed for all queries of one (pair, class): grid, radius
struct SearchFrame {
    GridView g;
    double max_dist_sqr; // CorrespondenceEstimation keeps d2 <= (2.5*thre)^2, evaluated in double (:1745, PCL)
    float r2_prune;
    bool defer;
};
__device__ __forceinline__ SearchFrame search_frame(const DeviceArrays &A, const PairConst &pc, const PairState &ps, int c, const SearchArgs &sa) {
    SearchFrame f;
    f.g = grid_of(A, pc, ps, c, sa.leaf_count);
    const float max_distance_f = 2.5f * ps.thre;
    f.max_dist_sqr = (double)max_distance_f * (double)max_distance_f;
    f.r2_prune = (float)f.max_dist_sqr * 1.0001f;
    f.defer = ps.iter >= kDeferFromIter; // queueing a block's small cells pays once the seeds are good
    return f;
}

// keep test of CorrespondenceEstimation + claim + result of one query
__device__ __forceinline__ void search_finish(DeviceArrays &A, const PairConst &pc, int c, uint32_t gi, int best_j, float best_d2,
                                              double max_dist_sqr, float orig_index_bits) {
    if (best_j >= 0 && !((double)best_d2 <= max_dist_sqr)) best_j = -1;
    if (best_j >= 0) {
        // duplicate_check_table as a claim: the lowest source index wins (:1762-1786, Q5)
        atomicMin(&A.claim[pc.tgt_base[c] + best_j], (unsigned)__float_as_int(orig_index_bits));
    }
    A.nn_idx[gi] = best_j;
    A.nn_d2[gi] = best_d2;
}

// seeded exact search of one query (p already advanced). Seeds: the previous iteration's match (a real candidate, so
// the box-distance pruning bites from the first cell on and the search only has to prove that nothing is closer); a
// match that the last increment left far away (the big first corrections) is challenged by a fresh greedy descent.
template <class Bounds>
__device__ __forceinline__ void search_one(DeviceArrays &A, const PairConst &pc, int c, int buf, uint32_t gi, const float4 p,
                                           float orig_bits, const SearchFrame &f, bool write_cert) {
    NoStats st;
    int best_j = -1;
    float best_d2 = INFINITY;
    const int pj = A.src_prevj[buf][gi];
    if (pj >= 0) {
        const float4 q = __ldg(&f.g.pos[pj]);
        best_d2 = flann_l2(p.x, p.y, p.z, q.x, q.y, q.z);
        best_j = pj;
    }
    {
        const float rs = kReseedCells * f.g.h0;
        if (best_j < 0 || best_d2 > rs * rs) {
            float d2 = INFINITY;
            int j = -1;
            walk_greedy_seed(f.g, p.x, p.y, p.z, kStartLevel, d2, j, st);
            if (j >= 0 && d2 < best_d2) best_d2 = d2, best_j = j;
        }
    }
    const float cert2 = nn_search_walk_b<Bounds>(f.g, p.x, p.y, p.z, f.r2_prune, kStartLevel, f.defer, best_d2, best_j, st);
    if (write_cert) A.src_cert[buf][gi] = make_float4(p.x, p.y, p.z, sqrtf(cert2));
    search_finish(A, pc, c, gi, best_j, best_d2, f.max_dist_sqr, orig_bits);
}

// direct mode: one warp, 32 consecutive sources of a chunk
template <class Bounds>
__device__ __forceinline__ void search_quarter(DeviceArrays &A, int buf, uint32_t chunk, uint32_t sub, const SearchArgs &sa, bool write_cert) {
    const ChunkDesc cd = A.it_chunks[chunk];
    const PairConst &pc = A.pc[cd.pair];
    const PairState &ps = A.ps[cd.pair];
    if (ps.status != kRunning || A.hash_used[1]) return;
    const int c = (int)cd.seg;
    const int ns = ps.n_src[c], nt = ps.n_tgt[c], nsg = ps.n_src_g[c];
    if ((int)cd.first >= ns) return; // warp-uniform
    if (shoots(pc, c)) return;       // warp-uniform: k_search_shoot's work
    const uint32_t local = cd.first + 32u * sub + (threadIdx.x & 31u);
    const bool valid = (int)local < ns;
    const uint32_t gi = pc.src_base[c] + (valid ? local : 0);
    float4 p, n;
    load_and_advance(A, ps, buf, gi, valid, p, n);
    if (!valid) return;
    // determine_corres needs >= 3 points on both sides (:1727-1728)
    if (!(pc.used[c] && nsg >= 3 && nt >= 3)) {
        A.nn_idx[gi] = -1;
        A.nn_d2[gi] = INFINITY;
        return;
    }
    const SearchFrame f = search_frame(A, pc, ps, c, sa);
    search_one<Bounds>(A, pc, c, buf, gi, p, n.w, f, write_cert);
}

// keep mode: one block, one chunk. need_list / n_need live in shared memory.
__device__ __forceinline__ void search_keep_chunk(DeviceArrays &A, int buf, uint32_t chunk, const SearchArgs &sa, uint8_t *need_list,
                                                  uint32_t *n_need) {
    const ChunkDesc cd = A.it_chunks[chunk];
    const PairConst &pc = A.pc[cd.pair];
    const PairState &ps = A.ps[cd.pair];
    if (ps.status != kRunning || A.hash_used[1]) return; // block-uniform, like the two below
    const int c = (int)cd.seg;
    const int ns = ps.n_src[c], nt = ps.n_tgt[c], nsg = ps.n_src_g[c];
    if ((int)cd.first >= ns) return;
    if (shoots(pc, c)) return;
    const int lane = threadIdx.x & 31;
    const bool active = pc.used[c] && nsg >= 3 && nt >= 3;
    const SearchFrame f = search_frame(A, pc, ps, c, sa);
    if (threadIdx.x == 0) *n_need = 0u;
    __syncthreads();
    // ---- pass A
    {
        const uint32_t local = cd.first + threadIdx.x;
        const bool valid = (int)local < ns;
        const uint32_t gi = pc.src_base[c] + (valid ? local : 0);
        float4 p, n;
        load_and_advance(A, ps, buf, gi, valid, p, n);
        bool need = false;
        if (valid) {
            if (!active) {
                A.nn_idx[gi] = -1;
                A.nn_d2[gi] = INFINITY;
            } else {
                need = true;
                const int pj = A.src_prevj[buf][gi];
                const float4 ce = A.src_cert[buf][gi]; // p_ref, certificate radius (0: none)
                if (pj >= 0 && ce.w > 0.0f) {
                    const float4 q = __ldg(&f.g.pos[pj]);
                    const float d1 = flann_l2(p.x, p.y, p.z, q.x, q.y, q.z);
                    const float mv = flann_l2(p.x, p.y, p.z, ce.x, ce.y, ce.z);
                    // every other target t: |p - t| >= |p_ref - t| - |p - p_ref| >= radius - moved. The factors and the
                    // 3e-5 m absorb the float evaluation of all the distances involved (coordinates < 1 km)
                    if ((sqrtf(d1) + sqrtf(mv)) * 1.0001f + 3e-5f < ce.w * 0.9999f) {
                        search_finish(A, pc, c, gi, pj, d1, f.max_dist_sqr, n.w);
                        need = false;
                    }
                }
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, need);
        uint32_t base = 0;
        if (lane == 0 && m) base = atomicAdd(n_need, (uint32_t)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (need) need_list[base + __popc(m & ((1u << lane) - 1u))] = (uint8_t)threadIdx.x;
    }
    __syncthreads();
    // ---- pass B: the listed queries fill the first threads (whole warps stay out when few are left)
    if (threadIdx.x < *n_need) {
        const uint32_t gi = pc.src_base[c] + cd.first + need_list[threadIdx.x];
        const float4 p = A.src_pos[buf][gi]; // (advanced by pass A)
        search_one<WalkBounds>(A, pc, c, buf, gi, p, A.src_nrm[buf][gi].w, f, true);
    }
}

// One kernel per mode (own register allocation each): 0 = direct, 1 = direct + certificate, 2 = keep. The iteration
// graph holds all three; the two that are not this iteration's return at once.
constexpr int kSearchBlocksPerSm = 12; // 40 registers (measured against 10 / 16 blocks: 4.36 / 4.31 / 4.61 ms per 64-pair step)
__device__ __forceinline__ int search_mode_of(int it) { return it >= kKeepFromIter ? 2 : (it == kKeepFromIter - 1 ? 1 : 0); }

template <int kMode>
__global__ void __launch_bounds__(kIterBlock, kSearchBlocksPerSm) k_search(DeviceArrays A, int buf, int it, int leaf_count) {
    buf = loop_buf(A, buf);
    if (it < 0) it = A.ctl->it; // (graph: the device-side loop counter; every running pair is in this iteration)
    if (blockIdx.x == 0 && threadIdx.x == 0) { // first kernel(s) of the iteration: counters and list the later ones use
        LoopCtl &ctl = *A.ctl;
        ctl.work[1] = ctl.work[2] = ctl.work[3] = 0u;
        ctl.n_live[buf ^ 1] = 0u;
    }
    if (search_mode_of(it) != kMode) return;
    const SearchArgs sa = {leaf_count};
    if (kMode == 2) {
        __shared__ uint8_t s_need[kIterBlock];
        __shared__ uint32_t s_n_need;
        for_each_live_chunk(A, buf, 0, [&](uint32_t chunk) { search_keep_chunk(A, buf, chunk, sa, s_need, &s_n_need); });
    } else {
        const uint32_t n_units = (kIterBlock / 32) * A.ctl->n_live[buf];
        const uint32_t *list = A.live_chunks + (size_t)buf * A.live_stride;
        for (;;) { // fetched per warp: no barrier, a warp that finishes early moves on
            uint32_t u = 0;
            if ((threadIdx.x & 31) == 0) u = atomicAdd(&A.ctl->work[0], 1u);
            u = __shfl_sync(0xffffffffu, u, 0);
            if (u >= n_units) break;
            if (kMode == 1) search_quarter<WalkBounds>(A, buf, list[u / (kIterBlock / 32)], u % (kIterBlock / 32), sa, true);
            else search_quarter<NoBounds>(A, buf, list[u / (kIterBlock / 32)], u % (kIterBlock / 32), sa, false);
            __syncwarp();
        }
    }
}

// :1732-1737 normal shooting [PCL CorrespondenceEstimationNormalShooting, k = 10]: among the 10 nearest targets
// the one with the smallest squared distance to the line through the source point along its normal; dropped
// if that value exceeds max_distance (NOT squared); correspondence distance = its squared NN distance.
// Launched only when a pair of the batch asked for normal shooting.
__device__ __forceinline__ void search_shoot_chunk(DeviceArrays &A, int buf, uint32_t chunk, int leaf_count) {
    const ChunkDesc cd = A.it_chunks[chunk];
    const PairConst &pc = A.pc[cd.pair];
    const PairState &ps = A.ps[cd.pair];
    if (ps.status != kRunning || A.hash_used[1]) return;
    const int c = (int)cd.seg;
    const int ns = ps.n_src[c], nt = ps.n_tgt[c], nsg = ps.n_src_g[c];
    if ((int)cd.first >= ns || !shoots(pc, c)) return; // block-uniform
    const uint32_t local = cd.first + threadIdx.x;
    const bool valid = (int)local < ns;
    const uint32_t gi = pc.src_base[c] + (valid ? local : 0);
    float4 p, n;
    load_and_advance(A, ps, buf, gi, valid, p, n);
    if (!valid) return;
    if (!(pc.used[c] && nsg >= 3 && nt >= 3)) {
        A.nn_idx[gi] = -1;
        A.nn_d2[gi] = INFINITY;
        return;
    }
    const GridView g = grid_of(A, pc, ps, c, leaf_count);
    const float max_distance_f = 2.5f * ps.thre;
    int sj = -1;
    float sd2 = INFINITY;
    KnnList kl;
    knn_search(g, p.x, p.y, p.z, kStartLevel, kl);
    double min_dist = 1.7976931348623157e308;
    for (int t = 0; t < kl.n; ++t) {
        const float4 q = __ldg(&g.pos[kl.j[t]]);
        const float ptx = q.x - p.x, pty = q.y - p.y, ptz = q.z - p.z;
        const double Nx = n.x, Ny = n.y, Nz = n.z, Vx = ptx, Vy = pty, Vz = ptz;
        const double Cx = Ny * Vz - Nz * Vy, Cy = Nz * Vx - Nx * Vz, Cz = Nx * Vy - Ny * Vx;
        const double dist = Cx * Cx + (Cy * Cy + Cz * Cz);
        if (dist < min_dist) {
            min_dist = dist;
            sj = kl.j[t];
            sd2 = kl.d2[t];
        }
    }
    if (sj >= 0 && min_dist > (double)max_distance_f) sj = -1;
    if (sj >= 0) atomicMin(&A.claim[pc.tgt_base[c] + sj], (unsigned)__float_as_int(n.w));
    A.nn_idx[gi] = sj;
    A.nn_d2[gi] = sd2;
}
__global__ void __launch_bounds__(kIterBlock) k_search_shoot(DeviceArrays A, int buf, int leaf_count) {
    buf = loop_buf(A, buf);
    for_each_live_chunk(A, buf, 3, [&](uint32_t chunk) { search_shoot_chunk(A, buf, chunk, leaf_count); });
}

// ---- k_resolve ---------------------------------------------------------------------------------
__device__ __forceinline__ void resolve_body(DeviceArrays &A, int buf, uint32_t chunk) {
    const ChunkDesc cd = A.it_chunks[chunk];
    const PairConst &pc = A.pc[cd.pair];
    PairState &ps = A.ps[cd.pair];
    if (ps.status != kRunning) return;
    const int c = (int)cd.seg;
    const int ns = ps.n_src[c], nt = ps.n_tgt[c], nsg = ps.n_src_g[c];
    const uint32_t local = cd.first + threadIdx.x;
    const bool valid = (int)local < ns;
    const bool active = pc.used[c] && nsg >= 3 && nt >= 3; // determine_corres ran for this class
    const bool dedup = active && nsg >= kDedupMinSrc;
    bool kept = false, pass = false;
    if (valid) {
        const uint32_t gi = pc.src_base[c] + local;
        const int j = A.nn_idx[gi];
        const bool matched = active && j >= 0;
        bool corr = matched;
        kept = true;
        if (dedup) {
            const float4 n = A.src_nrm[buf][gi];
            const bool winner = matched && A.claim[pc.tgt_base[c] + j] == (unsigned)__float_as_int(n.w);
            kept = winner;
            corr = winner;
        }
        if (corr) {
            // CorrespondenceRejectorDistance: distance < thre*thre, both float (:1794-1796, PCL)
            const float d2 = A.nn_d2[gi];
            pass = d2 < ps.thre * ps.thre;
            if (pass && c != MULLS_VERTEX) {
                const float4 n = A.src_nrm[buf][gi];
                const float4 m = A.tgt_nrm[pc.tgt_base[c] + j];
                const double dot = (double)n.x * (double)m.x + (double)n.y * (double)m.y + (double)n.z * (double)m.z;
                const float cos_angle = (float)fabs(dot);
                if ((double)cos_angle < pc.cos_thre) pass = false;
            }
        }
        A.flags[gi] = (uint8_t)((kept ? 1 : 0) | (pass ? 2 : 0));
    }
    const unsigned kb = __ballot_sync(0xffffffffu, kept);
    const unsigned pb = __ballot_sync(0xffffffffu, pass);
    __shared__ unsigned s_kept[kIterBlock / 32], s_pass[kIterBlock / 32];
    if ((threadIdx.x & 31) == 0) {
        s_kept[threadIdx.x >> 5] = __popc(kb);
        s_pass[threadIdx.x >> 5] = __popc(pb);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned k = 0, p = 0;
        for (int w = 0; w < kIterBlock / 32; ++w) {
            k += s_kept[w];
            p += s_pass[w];
        }
        A.blk_kept[chunk] = k;
        if (p) atomicAdd(&ps.n_corr[c], p);
    }
}
__global__ void __launch_bounds__(kIterBlock) k_resolve(DeviceArrays A, int buf) {
    buf = loop_buf(A, buf);
    for_each_live_chunk(A, buf, 1, [&](uint32_t chunk) { resolve_body(A, buf, chunk); });
}

// ------------------------------------------------------------------------------------------------
// per-correspondence normal-equation terms. Layout of the kTerms doubles of a partial:
//   [0..20]  lower triangle of ATPA, column by column: (0,0)(1,0)..(5,0)(1,1)(2,1)..(5,5)
//   [21..26] ATPb
// ------------------------------------------------------------------------------------------------
// `t`: anything indexable that takes the 27 terms (k_accumulate: a column of the block's shared-memory term matrix)
template <class Sink>
__device__ __forceinline__ void terms_pt2pl(const float4 p, const float pi, const float4 q, const float4 qn,
                                            float weight, int iter_num, bool dist_w, bool resid_w, bool inten_w,
                                            float window, Sink t, float &w_out) {
    // cregistration.hpp:2080-2151
    const float px = p.x, py = p.y, pz = p.z, qx = q.x, qy = q.y, qz = q.z;
    const float ntx = qn.x, nty = qn.y, ntz = qn.z;
    float w = weight;
    const float a = ntz * py - nty * pz;
    const float b = ntx * pz - ntz * px;
    const float c = nty * px - ntx * py;
    const float d = ntx * qx + nty * qy + ntz * qz - ntx * px - nty * py - ntz * pz;
    const float dist = sqrtf(qx * qx + qy * qy + qz * qz);
    if (dist_w) w = w * weight_by_dist_adaptive(dist, iter_num);
    if (resid_w) w = w * weight_by_residual(fabsf(d), window);
    if (inten_w) w = w * weight_by_intensity((float)((double)pi + 0.0001), (float)((double)q.w + 0.0001));
    w_out = w;
    t[0] = w * ntx * ntx;
    t[1] = w * ntx * nty;
    t[2] = w * ntx * ntz;
    t[3] = w * a * ntx;
    t[4] = w * b * ntx;
    t[5] = w * c * ntx;
    t[6] = w * nty * nty;
    t[7] = w * nty * ntz;
    t[8] = w * a * nty;
    t[9] = w * b * nty;
    t[10] = w * c * nty;
    t[11] = w * ntz * ntz;
    t[12] = w * a * ntz;
    t[13] = w * b * ntz;
    t[14] = w * c * ntz;
    t[15] = w * a * a;
    t[16] = w * a * b;
    t[17] = w * a * c;
    t[18] = w * b * b;
    t[19] = w * b * c;
    t[20] = w * c * c;
    t[21] = w * d * ntx;
    t[22] = w * d * nty;
    t[23] = w * d * ntz;
    t[24] = w * d * a;
    t[25] = w * d * b;
    t[26] = w * d * c;
}

// diagonal index of column j in the lower-triangle layout
__device__ __forceinline__ int diag_index(int j) {
    const int d[6] = {0, 6, 11, 15, 18, 20};
    return d[j];
}

template <class Sink>
__device__ __forceinline__ void terms_pt2li(const float4 p, const float pi, const float4 q, const float4 qv,
                                            float weight, int iter_num, bool dist_w, bool resid_w, bool inten_w,
                                            float window, Sink t, float &w_out) {
    // cregistration.hpp:2174-2271; only the diagonal of this block survives the symmetrisation (Q1)
    const float px = p.x, py = p.y, pz = p.z, qx = q.x, qy = q.y, qz = q.z;
    const float vx = qv.x, vy = qv.y, vz = qv.z;
    const float dx = px - qx, dy = py - qy, dz = pz - qz;
    double Am[3][6], bv[3];
    Am[0][0] = 0;
    Am[0][1] = (double)(-vz);
    Am[0][2] = (double)vy;
    Am[0][3] = (double)(vy * py + vz * pz);
    Am[0][4] = (double)(-vy * px);
    Am[0][5] = (double)(-vz * px);
    Am[1][0] = (double)vz;
    Am[1][1] = 0;
    Am[1][2] = (double)(-vx);
    Am[1][3] = (double)(-vx * py);
    Am[1][4] = (double)(vz * pz + vx * px);
    Am[1][5] = (double)(-vz * py);
    Am[2][0] = (double)(-vy);
    Am[2][1] = (double)vx;
    Am[2][2] = 0;
    Am[2][3] = (double)(-vx * pz);
    Am[2][4] = (double)(-vy * pz);
    Am[2][5] = (double)(vx * px + vy * py);
    bv[0] = (double)(-vy * dz + vz * dy);
    bv[1] = (double)(-vz * dx + vx * dz);
    bv[2] = (double)(-vx * dy + vy * dx);
    const float ex = (float)fabs(bv[0]), ey = (float)fabs(bv[1]), ez = (float)fabs(bv[2]);
    const float ed = sqrtf(ex * ex + ey * ey + ez * ez);
    float wx = weight;
    const float dist = sqrtf(qx * qx + qy * qy + qz * qz);
    if (dist_w) wx = wx * weight_by_dist_adaptive(dist, iter_num);
    if (inten_w) wx = wx * weight_by_intensity((float)((double)pi + 0.0001), (float)((double)q.w + 0.0001));
    if (resid_w) wx = wx * weight_by_residual(ed, window);
    w_out = wx;
    const double sw = (double)sqrtf(wx);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int cc = 0; cc < 6; ++cc) Am[r][cc] = sw * Am[r][cc];
        bv[r] = sw * bv[r];
    }
#pragma unroll
    for (int k = 0; k < 21; ++k) t[k] = 0.0;
    const int dg[6] = {0, 6, 11, 15, 18, 20};
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        t[dg[j]] = Am[0][j] * Am[0][j] + (Am[1][j] * Am[1][j] + Am[2][j] * Am[2][j]);
        t[21 + j] = Am[0][j] * bv[0] + (Am[1][j] * bv[1] + Am[2][j] * bv[2]);
    }
}

template <class Sink>
__device__ __forceinline__ void terms_pt2pt(const float4 p, const float pi, const float4 q, float weight,
                                            int iter_num, bool dist_w, bool resid_w, bool inten_w, float window,
                                            Sink t) {
    // cregistration.hpp:1991-2058
    const float px = p.x, py = p.y, pz = p.z, qx = q.x, qy = q.y, qz = q.z;
    const float dx = px - qx, dy = py - qy, dz = pz - qz;
    float wx = weight;
    const float dist = sqrtf(qx * qx + qy * qy + qz * qz);
    if (dist_w) wx = wx * weight_by_dist_adaptive(dist, iter_num);
    if (resid_w) wx = wx * weight_by_residual(sqrtf(dx * dx + dy * dy + dz * dz), window);
    if (inten_w) wx = wx * weight_by_intensity((float)((double)pi + 0.0001), (float)((double)q.w + 0.0001));
    const float wy = wx, wz = wx;
#pragma unroll
    for (int k = 0; k < 27; ++k) t[k] = 0.0;
    t[0] = wx;
    t[4] = wx * pz;
    t[5] = (-wx * py);
    t[6] = wy;
    t[8] = (-wy * pz);
    t[10] = wy * px;
    t[11] = wz;
    t[12] = wz * py;
    t[13] = (-wz * px);
    t[15] = wy * pz * pz + wz * py * py;
    t[16] = (-wz * px * py);
    t[17] = (-wy * px * pz);
    t[18] = wx * pz * pz + wz * px * px;
    t[19] = (-wx * py * pz);
    t[20] = wx * py * py + wy * px * px;
    t[21] = (-wx * dx);
    t[22] = (-wy * dy);
    t[23] = (-wz * dz);
    t[24] = wy * pz * dy - wz * py * dz;
    t[25] = wz * px * dz - wx * pz * dx;
    t[26] = wx * py * dx - wy * px * dy;
}

// w_ground of cregistration.hpp:1892-1900 from the per-class correspondence counts
__device__ __forceinline__ float balanced_ground_weight(const PairConst &pc, const uint32_t *n_corr) {
    if (!pc.w_balance) return 1.0f;
    const int m1 = (int)(n_corr[MULLS_GROUND] + n_corr[MULLS_ROOF]);
    const int m2 = (int)n_corr[MULLS_FACADE], m3 = (int)n_corr[MULLS_PILLAR], m4 = (int)n_corr[MULLS_BEAM];
    const float num = pc.z_xy_ratio * (float)(m2 + 2 * m3 - m4);
    const double v = (double)num / (0.0001 + 2.0 * (double)m1);
    return (float)((0.01 > v) ? 0.01 : v);
}

// :1301-1305 — too few correspondences?
__device__ __forceinline__ bool too_few(const PairConst &pc, const PairState &ps, const uint32_t *n_corr, float &ratio) {
    int total = 0;
    for (int c = 0; c < kNumClasses; ++c) total += (int)n_corr[c];
    const int nec = (int)(n_corr[MULLS_PILLAR] + n_corr[MULLS_BEAM] + n_corr[MULLS_FACADE]);
    ratio = (float)(1.0 * (double)nec / (double)ps.source_feature_points_count);
    return total < 40 || nec < 20 || ratio < pc.min_ratio;
}

// A pair stops iterating: publish the number of pairs still running to the host's launch loop.
__device__ __forceinline__ void pair_left_running(DeviceArrays &A) {
    const int left = atomicSub(A.running, 1) - 1;
    *A.h_running = left;
    __threadfence_system();
}

// Solve + state update of one pair; executed by thread 0 of the last block of k_accumulate
// (cregistration.hpp:1301-1400 after the summations). S = per-class sums [6][kTerms] in shared memory.
__device__ __noinline__ void solve_and_advance(DeviceArrays &A, uint32_t pair, const double *S, double *sm /*>= 150 doubles*/,
                                  int buf_written) {
    const PairConst &pc = A.pc[pair];
    PairState &ps = A.ps[pair];
    const int i = ps.iter;
    ps.iters_entered = i + 1;
    for (int c = 0; c < kNumClasses; ++c) ps.n_corr_last[c] = ps.n_corr[c];
    // bytes touched by this iteration's correspondence search: 28 B per active source and target point
    {
        uint64_t pts = 0;
        for (int c = 0; c < kNumClasses; ++c)
            if (pc.used[c]) pts += (uint64_t)ps.n_tgt[c];
        ps.alg_bytes += 28ull * pts; // sources added by the caller of this function (pre-compaction counts)
    }
    mulls_icp_trace *tr = trace_of(A, pair);
    if (tr && i < MULLS_MAX_TRACE_ITERS) {
        tr->n_iter = i + 1;
        for (int c = 0; c < kNumClasses; ++c) tr->n_corr[i][c] = ps.n_corr[c];
        for (int k = 0; k < 36; ++k) tr->atpa[i][k] = 0.0;
        for (int k = 0; k < 6; ++k) tr->atpb[i][k] = tr->x[i][k] = 0.0;
    }
    float ratio;
    const bool few = too_few(pc, ps, ps.n_corr, ratio);
    ps.confidence = ratio;
    if (few) {
        ps.code = -2;
        ps.status = kDone;
        pair_left_running(A);
        return; // TempTran = identity: T_total stays (:1307-1310, :1403)
    }
    // :1314-1315 threshold update
    {
        const double t = 1.0 * (double)ps.thre / (double)pc.thre_rate;
        ps.thre = (t > (double)pc.thre_min) ? (float)t : pc.thre_min;
    }
    // ATPA/ATPb: classes in the order of :1914-1921 (ground, facade, roof, pillar, beam, vertex)
    double *ATPA = sm;       // 36
    double *ATPb = sm + 36;  // 6
    double *inv = sm + 42;   // 36
    double *lu = sm + 78;    // 36
    double *Tmp = sm + 114;  // 16
    double low[21];
    for (int k = 0; k < 21; ++k) low[k] = 0.0;
    for (int k = 0; k < 6; ++k) ATPb[k] = 0.0;
    const int order[6] = {MULLS_GROUND, MULLS_FACADE, MULLS_ROOF, MULLS_PILLAR, MULLS_BEAM, MULLS_VERTEX};
    for (int o = 0; o < 6; ++o) {
        const double *s = S + order[o] * kTerms;
        for (int k = 0; k < 21; ++k) low[k] += s[k];
        for (int k = 0; k < 6; ++k) ATPb[k] += s[21 + k];
    }
    {
        int k = 0;
        for (int col = 0; col < 6; ++col)
            for (int row = col; row < 6; ++row, ++k) {
                ATPA[6 * row + col] = low[k];
                ATPA[6 * col + row] = low[k]; // :1924-1938 lower -> upper
            }
    }
    inverse6(ATPA, inv, lu);
    double x[6];
    for (int r = 0; r < 6; ++r) {
        double s = inv[6 * r] * ATPb[0];
        for (int cc = 1; cc < 6; ++cc) s = s + inv[6 * r + cc] * ATPb[cc];
        x[r] = s;
        ps.x[r] = s;
    }
    if (tr && i < MULLS_MAX_TRACE_ITERS) {
        for (int k = 0; k < 36; ++k) tr->atpa[i][k] = ATPA[k];
        for (int k = 0; k < 6; ++k) {
            tr->atpb[i][k] = ATPb[k];
            tr->x[i][k] = x[k];
        }
    }
    // :1953-1964 cofactor with the Euler->quaternion Jacobian (half-angle sines/cosines in FLOAT, :2797)
    {
        const float sr = (float)sin(0.5 * x[3]), sp = (float)sin(0.5 * x[4]), sy = (float)sin(0.5 * x[5]);
        const float cr = (float)cos(0.5 * x[3]), cp = (float)cos(0.5 * x[4]), cy = (float)cos(0.5 * x[5]);
        double J[3][3];
        J[0][0] = 0.5 * (double)(cr * cp * cy + sr * sp * sy);
        J[0][1] = 0.5 * (double)(-sr * sp * cy - cr * cp * sy);
        J[0][2] = 0.5 * (double)(-sr * cp * sy - cr * sp * cy);
        J[1][0] = 0.5 * (double)(-sr * sp * cy + cr * cp * sy);
        J[1][1] = 0.5 * (double)(cr * cp * cy - sr * sp * sy);
        J[1][2] = 0.5 * (double)(-cr * sp * sy + sr * cp * cy);
        J[2][0] = 0.5 * (double)(-sr * cp * sy - cr * sp * cy);
        J[2][1] = 0.5 * (double)(-cr * sp * sy - sr * cp * cy);
        J[2][2] = 0.5 * (double)(cr * cp * cy + sr * sp * sy);
        double *cof = ps.cofactor;
        for (int k = 0; k < 36; ++k) cof[k] = inv[k];
        double tmp[3][3];
        for (int r = 0; r < 3; ++r)
            for (int cc = 0; cc < 3; ++cc)
                tmp[r][cc] = J[r][0] * inv[6 * 3 + 3 + cc] + J[r][1] * inv[6 * 4 + 3 + cc] + J[r][2] * inv[6 * 5 + 3 + cc];
        for (int r = 0; r < 3; ++r)
            for (int cc = 0; cc < 3; ++cc)
                cof[6 * (3 + r) + 3 + cc] = tmp[r][0] * J[cc][0] + tmp[r][1] * J[cc][1] + tmp[r][2] * J[cc][2];
        for (int r = 0; r < 3; ++r)
            for (int cc = 0; cc < 3; ++cc)
                cof[6 * r + 3 + cc] = inv[6 * r + 3] * J[cc][0] + inv[6 * r + 4] * J[cc][1] + inv[6 * r + 5] * J[cc][2];
        for (int r = 0; r < 3; ++r)
            for (int cc = 0; cc < 3; ++cc)
                cof[6 * (3 + r) + cc] = J[r][0] * inv[6 * 3 + cc] + J[r][1] * inv[6 * 4 + cc] + J[r][2] * inv[6 * 5 + cc];
    }
    // :1333 TempTran
    double *Tt = ps.T_inc;
    construct_trans_a(x, Tt);
    const double ts_norm = sqrt(Tt[3] * Tt[3] + Tt[7] * Tt[7] + Tt[11] * Tt[11]);
    const double rs_angle = fabs(rotation_angle(Tt));
    if (ts_norm > (double)pc.max_t || rs_angle > (double)pc.max_r) { // :1348-1354
        ps.code = -1;
        ps.status = kDone;
        pair_left_running(A);
        return;
    }
    // :1400 / :1403 — the increment is always folded into the accumulated transform
    mat4_mul(Tt, ps.T_total, Tmp);
    for (int k = 0; k < 16; ++k) ps.T_total[k] = Tmp[k];
    if (i == pc.max_iter - 1 || (i > 2 && ts_norm < (double)pc.conv_t && rs_angle < (double)pc.conv_r)) { // :1357
        ps.status = kNeedPosterior;
        ps.final_buf = buf_written;
        pair_left_running(A);
        return;
    }
    ps.iter = i + 1;
}

// ---- k_accumulate ------------------------------------------------------------------------------
__device__ __forceinline__ void accumulate_body(DeviceArrays &A, int buf, uint32_t chunk) {
    const ChunkDesc cd = A.it_chunks[chunk];
    const PairConst &pc = A.pc[cd.pair];
    PairState &ps = A.ps[cd.pair];
    if (ps.status != kRunning) return;
    const int c = (int)cd.seg;
    const int ns = ps.n_src[c];
    const uint32_t local = cd.first + threadIdx.x;
    const bool valid = (int)local < ns;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int kWarps = kIterBlock / 32;
    // the block's term matrix: 27 rows of 128 doubles, one column per thread (27 KB: 8 blocks per SM)
    __shared__ double s_terms[27 * kIterBlock];
    __shared__ uint32_t s_off[kWarps + 1];
    __shared__ uint32_t s_base;

    // blocks entirely past the live part of the class have nothing to contribute (k_solve skips them)
    if ((int)cd.first >= ns) return;
    uint32_t dst_local = 0;
    uint8_t fl = 0;
    uint32_t gi = 0;
    bool kept = false, pass = false;
    struct Column { // row k of this thread's column
        double *base;
        __device__ __forceinline__ double &operator[](int k) const { return base[k * kIterBlock]; }
    } t = {s_terms + threadIdx.x};
    // (1) destination of the kept sources: blocks before this one in the same (pair, class)
    {
        uint32_t acc = 0;
        const uint32_t first_chunk = pc.class_chunk_begin[c];
        for (uint32_t b = first_chunk + threadIdx.x; b < chunk; b += kIterBlock) acc += A.blk_kept[b];
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) s_off[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tt = 0;
            for (int w = 0; w < kWarps; ++w) tt += s_off[w];
            s_base = tt;
        }
        __syncthreads();
    }
    if (valid) {
        gi = pc.src_base[c] + local;
        fl = A.flags[gi];
    }
    kept = (fl & 1) != 0, pass = (fl & 2) != 0;
    const unsigned kb = __ballot_sync(0xffffffffu, kept);
    if (lane == 0) s_off[warp] = __popc(kb);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (int w = 0; w < kWarps; ++w) {
            const uint32_t tt = s_off[w];
            s_off[w] = run;
            run += tt;
        }
        s_off[kWarps] = run;
    }
    __syncthreads();
    dst_local = s_base + s_off[warp] + __popc(kb & ((1u << lane) - 1u));

    // (2) terms of the surviving correspondences
    float w_store = 0.0f;
    int j = -1;
    float4 p = make_float4(0, 0, 0, 0), n = make_float4(0, 0, 0, 0);
    float d2 = 0.0f;
    if (valid) {
        p = A.src_pos[buf][gi];
        n = A.src_nrm[buf][gi];
        j = A.nn_idx[gi];
        d2 = A.nn_d2[gi];
        if (j >= 0) A.claim[pc.tgt_base[c] + j] = kClaimFree; // reset the table for the next iteration
    }
    uint32_t n_corr[kNumClasses]; // complete since every k_resolve block of the pair has finished
#pragma unroll
    for (int k = 0; k < kNumClasses; ++k) n_corr[k] = ps.n_corr[k];
    float ratio_unused;
    const bool few = too_few(pc, ps, n_corr, ratio_unused);
    if (pass && !few) {
        const float4 q = A.tgt_pos[pc.tgt_base[c] + j];
        const float4 qn = A.tgt_nrm[pc.tgt_base[c] + j];
        const int it = ps.iter;
        const bool resid_w = pc.w_residual && it > 2; // :1905-1907
        const bool dist_w = pc.w_dist != 0, inten_w = pc.w_intensity != 0;
        if (c == MULLS_GROUND || c == MULLS_FACADE || c == MULLS_ROOF) {
            const float wc = (c == MULLS_FACADE) ? 1.0f : balanced_ground_weight(pc, n_corr);
            terms_pt2pl(p, p.w, q, qn, wc, it, dist_w, resid_w, inten_w, pc.win_pt2pl, t, w_store);
        } else if (c == MULLS_PILLAR || c == MULLS_BEAM) {
            terms_pt2li(p, p.w, q, qn, 1.0f, it, dist_w, resid_w, inten_w, pc.win_pt2li, t, w_store);
        } else {
            terms_pt2pt(p, p.w, q, 1.0f, it, dist_w, resid_w, inten_w, pc.win_pt2pt, t);
            w_store = d2; // pt2pt never stores a weight: the posterior reads the squared NN distance (Q2)
        }
    } else {
#pragma unroll
        for (int k = 0; k < 27; ++k) t[k] = 0.0;
    }
    // (3) compaction into the other buffer (order preserved: :1776-1789)
    if (kept) {
        const uint32_t gd = pc.src_base[c] + dst_local;
        A.src_pos[buf ^ 1][gd] = p;
        A.src_nrm[buf ^ 1][gd] = n;
        A.src_prevj[buf ^ 1][gd] = j;
        A.src_cert[buf ^ 1][gd] = A.src_cert[buf][gi];
        A.corr_j[gd] = pass ? j : -1;
        A.corr_w[gd] = w_store;
    }
    // (4) block reduction in a fixed order: warp w sums rows w, w + 4, ... of the term matrix — four columns per lane,
    // then a butterfly over the lanes (every lane ends with the same total): bit-reproducible, independent of the
    // order in which blocks fetch chunks
    __syncthreads();
#pragma unroll 1
    for (int k = warp; k < 27; k += kWarps) {
        const double *row = s_terms + k * kIterBlock;
        double v = ((row[lane] + row[lane + 32]) + row[lane + 64]) + row[lane + 96];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) A.partials[(size_t)chunk * kTerms + k] = v;
    }
}
__global__ void __launch_bounds__(kIterBlock, 8) k_accumulate(DeviceArrays A, int buf) {
    buf = loop_buf(A, buf);
    if (blockIdx.x == 0 && threadIdx.x == 0) A.ctl->work[0] = 0u; // the next iteration's k_search starts its list at 0
    for_each_live_chunk(A, buf, 2, [&](uint32_t chunk) { accumulate_body(A, buf, chunk); });
}

// the chunks of this pair that still own live sources go onto the next iteration's list (whole block; the pair's state
// has just been advanced by thread 0)
__device__ __forceinline__ void publish_live_chunks(const DeviceArrays &A, uint32_t pair, int next_parity) {
    __shared__ uint32_t s_base;
    __syncthreads();
    const PairConst &pc = A.pc[pair];
    const PairState &ps = A.ps[pair];
    if (ps.status != kRunning) return; // block-uniform
    uint32_t count[kNumClasses], total = 0;
#pragma unroll
    for (int c = 0; c < kNumClasses; ++c) {
        count[c] = (uint32_t)((ps.n_src[c] + kIterBlock - 1) / kIterBlock);
        total += count[c];
    }
    if (threadIdx.x == 0) s_base = atomicAdd(&A.ctl->n_live[next_parity], total);
    __syncthreads();
    uint32_t base = s_base;
#pragma unroll
    for (int c = 0; c < kNumClasses; ++c) {
        append_live_chunks(A, next_parity, pc.class_chunk_begin[c], count[c], base);
        base += count[c];
    }
}

// ---- solve: one block per pair, after every k_accumulate block of the pair. Sums the per-chunk partials of every
//      class in chunk order (fixed order => bit-reproducible), then one thread solves and advances the pair state.
//      Any block size that is a multiple of 32: the warps take the classes in turn.
__device__ __forceinline__ void solve_body(DeviceArrays &A, int buf, uint32_t pair) {
    const PairConst &pc = A.pc[pair];
    PairState &ps = A.ps[pair];
    if (ps.status != kRunning) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    __shared__ double s_S[kNumClasses][kTerms];
    __shared__ double s_scratch[160];
    __shared__ int s_newn[kNumClasses];
    __shared__ uint32_t s_ncorr[kNumClasses];
    for (int cc = warp; cc < kNumClasses; cc += n_warps) {
        const uint32_t b0 = pc.class_chunk_begin[cc];
        // only the chunks that held live sources this iteration wrote a partial
        const uint32_t live = (uint32_t)((ps.n_src[cc] + kIterBlock - 1) / kIterBlock);
        const uint32_t b1 = min(pc.class_chunk_begin[cc + 1], b0 + live);
        // lane = term; chunks in order, four independent accumulators combined in a fixed order
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
        if (lane < 27) {
            uint32_t b = b0;
            for (; b + 4 <= b1; b += 4) {
                a0 += A.partials[(size_t)(b + 0) * kTerms + lane];
                a1 += A.partials[(size_t)(b + 1) * kTerms + lane];
                a2 += A.partials[(size_t)(b + 2) * kTerms + lane];
                a3 += A.partials[(size_t)(b + 3) * kTerms + lane];
            }
            for (; b < b1; ++b) a0 += A.partials[(size_t)b * kTerms + lane];
        }
        if (lane < kTerms) s_S[cc][lane] = (lane < 27) ? ((a0 + a1) + (a2 + a3)) : 0.0;
        uint32_t acc = 0; // kept sources of the class = its new size
        for (uint32_t b = b0 + lane; b < b1; b += 32) acc += A.blk_kept[b];
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) {
            s_newn[cc] = (int)acc;
            s_ncorr[cc] = ps.n_corr[cc];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t srcpts = 0;
        for (int cc = 0; cc < kNumClasses; ++cc)
            if (pc.used[cc]) srcpts += (uint64_t)ps.n_src_g[cc];
        ps.alg_bytes += 28ull * srcpts;
        if (pc.sharded) {
            // source-sharded registration: publish this rank's per-class sums; the all-reduce and
            // k_shard_solve (identical on every rank) finish the iteration
            for (int cc = 0; cc < kNumClasses; ++cc) {
                ps.n_src[cc] = s_newn[cc];
                for (int k = 0; k < kTerms; ++k) A.xch_f64[cc * kTerms + k] = (k < 27) ? s_S[cc][k] : 0.0;
            }
        } else {
        mulls_icp_trace *tr = trace_of(A, pair);
        for (int cc = 0; cc < kNumClasses; ++cc) {
            ps.n_src[cc] = s_newn[cc]; // classes that skipped determine_corres keep everything (k_resolve)
            ps.n_src_g[cc] = s_newn[cc];
            ps.n_corr[cc] = s_ncorr[cc];
            if (tr && ps.iter < MULLS_MAX_TRACE_ITERS) tr->n_src[ps.iter][cc] = (uint32_t)ps.n_src[cc];
        }
        solve_and_advance(A, pair, &s_S[0][0], s_scratch, buf ^ 1);
        for (int cc = 0; cc < kNumClasses; ++cc) ps.n_corr[cc] = 0;
        }
    }
    // (a sharded pair is advanced by k_shard_solve, after the exchange of the sums: it publishes the list)
    if (!pc.sharded) publish_live_chunks(A, pair, buf ^ 1);
}
constexpr int kSolveThreads = kNumClasses * 32; // one warp per feature class
// loop_handle != 0: the launch is the last kernel of the iteration graph's WHILE body — the block that finishes last
// advances the loop counter and tells the graph whether another iteration is needed (pairs still running)
__global__ void __launch_bounds__(kSolveThreads) k_solve(DeviceArrays A, int buf, unsigned long long loop_handle) {
    LoopCtl &ctl = *A.ctl;
    if (blockIdx.x >= (unsigned)ctl.n_pairs) return;
    solve_body(A, loop_buf(A, buf), blockIdx.x);
    if (loop_handle == 0ull) return;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&ctl.solved, 1u) == (unsigned)ctl.n_pairs - 1u) {
            ctl.solved = 0;
            const int it = ctl.it + 1;
            ctl.it = it;
            __threadfence();
            const bool again = *(volatile int *)A.running > 0 && it < ctl.max_iter;
            cudaGraphSetConditional((cudaGraphConditionalHandle)loop_handle, again ? 1u : 0u);
        }
    }
}

// ---- k_icp_loop: the WHOLE iteration loop of a small batch as one cooperative kernel. For registrations whose chunks fit
//      the co-resident grid (the reference's own operating point: a few thousand source points against a 20k-point local
//      map, test/mulls_slam.cpp:477-482) an iteration is seven short kernels at the launch-latency floor; here the four
//      phases are the same device functions over the same work lists, separated by grid-wide barriers instead of kernel
//      boundaries. Every block executes the same number of barriers: the loop bounds (LoopCtl::max_iter, the running
//      counter read after a barrier) are grid-uniform.
__global__ void __launch_bounds__(kIterBlock, 4) k_icp_loop(DeviceArrays A, int leaf_count) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    LoopCtl &ctl = *A.ctl;
    const SearchArgs sa = {leaf_count};
    __shared__ uint8_t s_need[kIterBlock];
    __shared__ uint32_t s_n_need;
    const int n_pairs = ctl.n_pairs, max_iter = ctl.max_iter;
    for (int it = 0; it < max_iter; ++it) {
        const int buf = it & 1;
        const uint32_t *list = A.live_chunks + (size_t)buf * A.live_stride;
        const uint32_t n_live = ctl.n_live[buf];
        if (blockIdx.x == 0 && threadIdx.x == 0) ctl.n_live[buf ^ 1] = 0u; // (k_solve's phase fills it, three barriers later)
        // phase 1: transform + search (+ keep) + claim
        for (uint32_t w = blockIdx.x; w < n_live; w += gridDim.x) {
            const uint32_t chunk = list[w];
            if (it >= kKeepFromIter) search_keep_chunk(A, buf, chunk, sa, s_need, &s_n_need);
            else if (it == kKeepFromIter - 1) search_quarter<WalkBounds>(A, buf, chunk, threadIdx.x >> 5, sa, true);
            else search_quarter<NoBounds>(A, buf, chunk, threadIdx.x >> 5, sa, false);
            __syncthreads();
        }
        grid.sync();
        // phase 2: duplicate check, rejectors, counts
        for (uint32_t w = blockIdx.x; w < n_live; w += gridDim.x) {
            resolve_body(A, buf, list[w]);
            __syncthreads();
        }
        grid.sync();
        // phase 3: compaction + normal-equation partials
        for (uint32_t w = blockIdx.x; w < n_live; w += gridDim.x) {
            accumulate_body(A, buf, list[w]);
            __syncthreads();
        }
        grid.sync();
        // phase 4: per pair — sum, solve, advance, publish the next work list
        for (int pair = blockIdx.x; pair < n_pairs; pair += gridDim.x) {
            solve_body(A, buf, (uint32_t)pair);
            __syncthreads();
        }
        grid.sync();
        if (*(volatile int *)A.running <= 0) break; // (grid-uniform: nothing writes it between this barrier and the next solve)
    }
}

// ---- sharded mode (mulls_icp_run_sharded, BASELINE config 5): one pair, the target replicated, the source
//      classes split over ranks in contiguous index ranges. Three tiny exchange steps per iteration, each an
//      all-reduce supplied by the caller (NCCL): claim table (min), counts (sum), per-class sums (sum).
// after ingest: global class sizes and the global bbox of source ground/pillar/facade
__global__ void k_shard_pack_setup(DeviceArrays A, int phase) {
    PairState &ps = A.ps[0];
    if (phase == 0) { // bbox: min over [min_xyz, -max_xyz] in the ordered-int encoding
        for (int d = 0; d < 3; ++d) {
            A.xch_i32[d] = ps.bb_src[d];
            A.xch_i32[3 + d] = ~ps.bb_src[3 + d]; // max(x) = ~min(~x), no overflow for INT_MIN
        }
    } else if (phase == 1) {
        for (int d = 0; d < 3; ++d) {
            ps.bb_src[d] = A.xch_i32[d];
            ps.bb_src[3 + d] = ~A.xch_i32[3 + d];
        }
    } else if (phase == 2) {
        for (int c = 0; c < kNumClasses; ++c) A.xch_i32[c] = ps.n_src[c];
    } else {
        const PairConst &pc = A.pc[0];
        int cnt = 0;
        for (int c = 0; c < kNumClasses; ++c) ps.n_src_g[c] = A.xch_i32[c];
        if (pc.used[MULLS_PILLAR]) cnt += ps.n_src_g[MULLS_PILLAR];
        if (pc.used[MULLS_FACADE]) cnt += ps.n_src_g[MULLS_FACADE];
        if (pc.used[MULLS_BEAM]) cnt += ps.n_src_g[MULLS_BEAM];
        ps.source_feature_points_count = cnt;
    }
}
// after k_resolve: this rank's correspondence and kept-source counts -> exchange buffer; and back
__global__ void __launch_bounds__(kIterBlock) k_shard_counts(DeviceArrays A, int phase) {
    const PairConst &pc = A.pc[0];
    PairState &ps = A.ps[0];
    if (ps.status != kRunning) {
        if (phase == 0 && threadIdx.x < 2 * kNumClasses) A.xch_i32[threadIdx.x] = 0;
        return;
    }
    if (phase == 0) {
        __shared__ uint32_t s_w[kIterBlock / 32];
        for (int cc = 0; cc < kNumClasses; ++cc) {
            const uint32_t b0 = pc.class_chunk_begin[cc];
            const uint32_t live = (uint32_t)((ps.n_src[cc] + kIterBlock - 1) / kIterBlock);
            const uint32_t b1 = min(pc.class_chunk_begin[cc + 1], b0 + live);
            uint32_t acc = 0;
            for (uint32_t b = b0 + threadIdx.x; b < b1; b += kIterBlock) acc += A.blk_kept[b];
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            __syncthreads();
            if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
            __syncthreads();
            if (threadIdx.x == 0) {
                uint32_t tot = 0;
                for (int w = 0; w < kIterBlock / 32; ++w) tot += s_w[w];
                A.xch_i32[kNumClasses + cc] = (int)tot;
                A.xch_i32[cc] = (int)ps.n_corr[cc];
            }
        }
    } else if (threadIdx.x == 0) {
        for (int cc = 0; cc < kNumClasses; ++cc) {
            ps.n_corr[cc] = (uint32_t)A.xch_i32[cc];
            ps.n_src_g_next[cc] = A.xch_i32[kNumClasses + cc]; // the class size after this iteration's shrinking
        }
    }
}
// after the all-reduce of the per-class sums: every rank solves the same system and advances identically
__global__ void k_shard_solve(DeviceArrays A, int buf, int it_flag) {
    PairState &ps = A.ps[0];
    __shared__ double s_scratch[160];
    if (threadIdx.x == 0) {
        if (ps.status != kRunning) {
            A.h_running_iter[it_flag] = *A.running;
            __threadfence_system();
        } else {
            mulls_icp_trace *tr = trace_of(A, 0);
            for (int cc = 0; cc < kNumClasses; ++cc) {
                ps.n_src_g[cc] = ps.n_src_g_next[cc];
                if (tr && ps.iter < MULLS_MAX_TRACE_ITERS) tr->n_src[ps.iter][cc] = (uint32_t)ps.n_src_g[cc];
            }
            solve_and_advance(A, 0, A.xch_f64, s_scratch, buf ^ 1);
            for (int cc = 0; cc < kNumClasses; ++cc) ps.n_corr[cc] = 0;
            A.h_running_iter[it_flag] = *A.running; // what the launch loop of every rank reads two iterations later
            __threadfence_system();
        }
    }
    publish_live_chunks(A, 0, buf ^ 1); // this rank's shard: its own live chunks
}
// posterior in sharded mode: VTPV / n_obs of this rank -> exchange buffer
__global__ void k_shard_post(DeviceArrays A, int phase) {
    const PairConst &pc = A.pc[0];
    PairState &ps = A.ps[0];
    if (threadIdx.x != 0) return;
    if (phase == 0) {
        double VTPV = 0.0, nob = 0.0;
        if (ps.status == kNeedPosterior) {
            const int order[6] = {MULLS_GROUND, MULLS_FACADE, MULLS_ROOF, MULLS_PILLAR, MULLS_BEAM, MULLS_VERTEX};
            for (int o = 0; o < 6; ++o) {
                const uint32_t b0 = pc.class_chunk_begin[order[o]];
                const uint32_t live = (uint32_t)((ps.n_src[order[o]] + kIterBlock - 1) / kIterBlock);
                const uint32_t b1 = min(pc.class_chunk_begin[order[o] + 1], b0 + live);
                for (uint32_t b = b0; b < b1; ++b) {
                    VTPV += A.post_partials[2 * (size_t)b];
                    nob += A.post_partials[2 * (size_t)b + 1];
                }
            }
        }
        A.xch_f64[0] = VTPV;
        A.xch_f64[1] = nob;
    } else if (ps.status == kNeedPosterior) {
        const double sigma2 = A.xch_f64[0] / (double)((int)A.xch_f64[1] - 6);
        ps.sigma2 = sigma2;
        ps.code = (sqrt(sigma2) < pc.sigma_thre) ? 1 : -3;
        double inv[36], lu[36];
        inverse6(ps.cofactor, inv, lu);
        for (int k = 0; k < 36; ++k) ps.info[k] = (1.0 / sigma2) * inv[k];
        ps.status = kDone;
    }
}

// ---- k_posterior -------------------------------------------------------------------------------
// cregistration.hpp:2518-2544: VTPV and observation count over the correspondences of the converged
// iteration with its estimate x; sigma^2, code 1 / -3, information matrix (:1386).
__global__ void __launch_bounds__(kIterBlock) k_posterior(DeviceArrays A) {
    if (!chunk_in_run(A)) return;
    const ChunkDesc cd = A.it_chunks[blockIdx.x];
    const PairConst &pc = A.pc[cd.pair];
    PairState &ps = A.ps[cd.pair];
    if (ps.status != kNeedPosterior) return;
    const int c = (int)cd.seg;
    const int buf = ps.final_buf;
    if ((int)cd.first >= ps.n_src[c]) return; // k_finalize only sums the live chunks
    const uint32_t local = cd.first + threadIdx.x;
    const bool valid = (int)local < ps.n_src[c];
    double vtpv = 0.0;
    int nobs = 0;
    if (valid) {
        const uint32_t gi = pc.src_base[c] + local;
        const int j = A.corr_j[gi];
        if (j >= 0) {
            const float4 p = A.src_pos[buf][gi];
            const float4 q = A.tgt_pos[pc.tgt_base[c] + j];
            const float4 qn = A.tgt_nrm[pc.tgt_base[c] + j];
            const float w = A.corr_w[gi];
            const double *x = ps.x;
            const float px = p.x, py = p.y, pz = p.z, qx = q.x, qy = q.y, qz = q.z;
            if (c == MULLS_GROUND || c == MULLS_FACADE || c == MULLS_ROOF) { // :2602-2623
                const float ntx = qn.x, nty = qn.y, ntz = qn.z;
                const float a = ntz * py - nty * pz;
                const float b = ntx * pz - ntz * px;
                const float cc = nty * px - ntx * py;
                const float d = ntx * qx + nty * qy + ntz * qz - ntx * px - nty * py - ntz * pz;
                const float residual = (float)((double)ntx * x[0] + (double)nty * x[1] + (double)ntz * x[2] +
                                               (double)a * x[3] + (double)b * x[4] + (double)cc * x[5] - (double)d);
                vtpv = (double)(w * residual * residual);
                nobs = 1;
            } else {
                const float dx = px - qx, dy = py - qy, dz = pz - qz;
                double Am[3][6], bv[3];
                if (c == MULLS_PILLAR || c == MULLS_BEAM) { // :2643-2673
                    const float vx = qn.x, vy = qn.y, vz = qn.z;
                    Am[0][0] = 0, Am[0][1] = (double)vz, Am[0][2] = (double)(-vy), Am[0][3] = (double)(-vz * pz - vy * py),
                    Am[0][4] = (double)(vy * px), Am[0][5] = (double)(vz * px);
                    Am[1][0] = (double)(-vz), Am[1][1] = 0, Am[1][2] = (double)vx, Am[1][3] = (double)(vx * py),
                    Am[1][4] = (double)(-vx * px - vz * pz), Am[1][5] = (double)(vz * py);
                    Am[2][0] = (double)vy, Am[2][1] = (double)(-vx), Am[2][2] = 0, Am[2][3] = (double)(vx * pz),
                    Am[2][4] = (double)(vy * pz), Am[2][5] = (double)(-vy * py - vx * px);
                    bv[0] = (double)(-vz * dy + vy * dz);
                    bv[1] = (double)(-vx * dz + vz * dx);
                    bv[2] = (double)(-vy * dx + vx * dy);
                } else { // :2559-2583
                    Am[0][0] = 1, Am[0][1] = 0, Am[0][2] = 0, Am[0][3] = 0, Am[0][4] = (double)pz, Am[0][5] = (double)(-py);
                    Am[1][0] = 0, Am[1][1] = 1, Am[1][2] = 0, Am[1][3] = (double)(-pz), Am[1][4] = 0, Am[1][5] = (double)px;
                    Am[2][0] = 0, Am[2][1] = 0, Am[2][2] = 1, Am[2][3] = (double)py, Am[2][4] = (double)(-px), Am[2][5] = 0;
                    bv[0] = (double)(-dx), bv[1] = (double)(-dy), bv[2] = (double)(-dz);
                }
                double r[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    double s = Am[k][0] * x[0];
#pragma unroll
                    for (int jj = 1; jj < 6; ++jj) s = s + Am[k][jj] * x[jj];
                    r[k] = s - bv[k];
                }
                vtpv = (double)w * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
                nobs = 3;
            }
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int kWarps = kIterBlock / 32;
    __shared__ double s_v[kWarps];
    __shared__ int s_n[kWarps];
    for (int o = 16; o > 0; o >>= 1) {
        vtpv += __shfl_xor_sync(0xffffffffu, vtpv, o);
        nobs += __shfl_xor_sync(0xffffffffu, nobs, o);
    }
    if (lane == 0) {
        s_v[warp] = vtpv;
        s_n[warp] = nobs;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double v = 0.0;
        int n = 0;
        for (int w = 0; w < kWarps; ++w) {
            v += s_v[w];
            n += s_n[w];
        }
        A.post_partials[2 * (size_t)blockIdx.x] = v;
        A.post_partials[2 * (size_t)blockIdx.x + 1] = (double)n;
    }
}

// ---- k_finalize: one thread per pair: sigma^2 = VTPV/(n-6) (:2536), code 1 / -3 (:2540-2543), information
//      matrix = cofactor^-1 / sigma^2 (:1386). Partials are summed in the class order of :2529-2534.
__global__ void k_finalize(DeviceArrays A, int n_pairs) {
    if (n_pairs < 0) n_pairs = A.ctl->n_pairs; // recorded into the iteration graph: launched over the capacity
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= n_pairs) return;
    const PairConst &pc = A.pc[pair];
    PairState &ps = A.ps[pair];
    if (ps.status != kNeedPosterior) return;
    const int order[6] = {MULLS_GROUND, MULLS_FACADE, MULLS_ROOF, MULLS_PILLAR, MULLS_BEAM, MULLS_VERTEX};
    double VTPV = 0.0;
    long long nob = 0;
    for (int o = 0; o < 6; ++o) {
        const uint32_t b0 = pc.class_chunk_begin[order[o]];
        const uint32_t live = (uint32_t)((ps.n_src[order[o]] + kIterBlock - 1) / kIterBlock);
        const uint32_t b1 = min(pc.class_chunk_begin[order[o] + 1], b0 + live);
        for (uint32_t b = b0; b < b1; ++b) {
            VTPV += A.post_partials[2 * (size_t)b];
            nob += (long long)A.post_partials[2 * (size_t)b + 1];
        }
    }
    const double sigma2 = VTPV / (double)((int)nob - 6);
    ps.sigma2 = sigma2;
    ps.code = (sqrt(sigma2) < pc.sigma_thre) ? 1 : -3;
    double inv[36], lu[36];
    inverse6(ps.cofactor, inv, lu);
    for (int k = 0; k < 36; ++k) ps.info[k] = (1.0 / sigma2) * inv[k];
    ps.status = kDone;
}

// ---- k_nn_query: mulls_nn_query — exact 1-NN of arbitrary query points in one target class of pair 0, on the grid
//      the last registration built (what block1->tree_*->nearestKSearch(p, 1) answers in the reference)
__global__ void __launch_bounds__(kIterBlock) k_nn_query(DeviceArrays A, int cls, const float *xyz, uint32_t n, int leaf_count,
                                                        int *out_idx, float *out_d2) {
    const uint32_t i = blockIdx.x * kIterBlock + threadIdx.x;
    if (i >= n) return;
    const PairConst &pc = A.pc[0];
    const PairState &ps = A.ps[0];
    int best_j = -1;
    float best_d2 = INFINITY;
    if (ps.n_tgt[cls] > 0 && !A.hash_used[1]) {
        const GridView g = grid_of(A, pc, ps, cls, leaf_count);
        const float px = xyz[3 * i], py = xyz[3 * i + 1], pz = xyz[3 * i + 2];
        const float rmax = 2.5f * pc.thre_unit;
        const float r2 = rmax * rmax * 1.0001f;
        NoStats st;
        walk_greedy_seed(g, px, py, pz, kStartLevel, best_d2, best_j, st);
        nn_search_walk(g, px, py, pz, r2, kStartLevel, false, best_d2, best_j, st);
        if (best_j >= 0 && !((double)best_d2 <= (double)rmax * (double)rmax)) best_j = -1;
        if (best_j >= 0) best_j = __float_as_int(__ldg(&g.nrm[best_j]).w);
    }
    out_idx[i] = best_j;
    out_d2[i] = best_j >= 0 ? best_d2 : INFINITY;
}

// ---- k_state_init: reset the per-pair accumulators that the ingest kernels update atomically
__global__ void k_state_init(DeviceArrays A, int n_pairs) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    PairState &ps = A.ps[p];
    for (int d = 0; d < 3; ++d) {
        ps.bb_src[d] = ps.bb_tgt[d] = 0x7fffffff;
        ps.bb_src[3 + d] = ps.bb_tgt[3 + d] = (int)0x80000000;
    }
    for (int s = 0; s < kNumSegs; ++s) ps.seg_count[s] = ps.seg_start[s] = 0;
    for (int c = 0; c < kNumClasses; ++c) ps.hash_entries[c] = ps.n_corr[c] = 0;
    ps.status = kRunning;
    if (p == 0) {
        *A.running = n_pairs;
        *A.h_running = n_pairs;
    }
}

// ---- k_collect: pair state -> mulls_icp_result (device copy, then one D2H)
__global__ void k_collect(DeviceArrays A, int n_pairs, mulls_icp_result *out) {
    if (n_pairs < 0) n_pairs = A.ctl->n_pairs;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const PairState &ps = A.ps[p];
    mulls_icp_result &r = out[p];
    for (int k = 0; k < 16; ++k) r.T[k] = ps.T_total[k];
    for (int k = 0; k < 36; ++k) r.info[k] = ps.info[k];
    r.sigma = (float)sqrt(ps.sigma2);
    r.confidence = ps.confidence;
    r.code = ps.code;
    r.iters = ps.iters_entered;
    for (int c = 0; c < kNumClasses; ++c) {
        r.n_corr[c] = ps.n_corr_last[c];
        r.n_src[c] = (uint32_t)ps.n_src_g[c];
    }
    // (the per-pair algorithmic-byte counters ride behind the results: one D2H fetches both)
    reinterpret_cast<uint64_t *>(out + A.ctl->n_pairs)[p] = ps.alg_bytes;
}

} // namespace mulls
