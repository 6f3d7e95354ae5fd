// Ingest phase: what mm_lls_icp does before its iteration loop (cregistration.hpp:1180-1232) —
// clone + apply initial guess, intersection filter, and (instead of six FLANN kd-trees) a spatial
// sort of every cloud plus a multi-level hashed grid over each target class.
#pragma once
#include "device_math.cuh"
#include "device_types.cuh"

namespace mulls {

// ---- k_ingest_transform: AoS48 -> staging SoA; source gets the initial guess (double math, float store,
//      pcl::transformPointCloudWithNormals semantics); bbox reductions for the intersection filter.
// kUndistort = false: the instantiation for batches in which no pair asks for motion undistortion (no slerp code, 32
// registers, 8 blocks per SM — the kernel is a latency-bound stream: 28 B read + 32 B written per point)
template <bool kUndistort>
__global__ void __launch_bounds__(kIngestBlock, kUndistort ? 4 : 6) k_ingest_transform(DeviceArrays A) {
    const ChunkDesc cd = A.in_chunks[blockIdx.x];
    const PairConst &pc = A.pc[cd.pair];
    const uint32_t seg = cd.seg;
    const uint32_t local = cd.first + threadIdx.x;
    const bool valid = local < pc.in_n[seg];
    const bool is_src = seg >= kNumClasses;
    const int cls = seg % kNumClasses;
    float x = 0, y = 0, z = 0;
    if (valid) {
        const size_t gi = (size_t)pc.in_off[seg] + local;
        // three layouts behind in_ptr (block-uniform): the caller's 48-byte rows, or the host-packed wire formats
        float nx, ny, nz, intensity, curvature = 0.0f;
        const uint32_t fmt = pc.in_fmt[seg];
        if (fmt == 0u) {
            const float4 *in = pc.in_ptr[seg] + 3 * (size_t)local;
            const float4 a = in[0]; // x y z _
            const float4 b = in[1]; // nx ny nz _
            const float4 c = in[2]; // intensity curvature _ _
            x = a.x, y = a.y, z = a.z;
            nx = b.x, ny = b.y, nz = b.z;
            intensity = c.x, curvature = c.y;
        } else {
            const float4 *in = pc.in_ptr[seg];
            const float4 a = in[local]; // x y z intensity
            x = a.x, y = a.y, z = a.z, intensity = a.w;
            if (fmt == 1u) {
                const float *nr = reinterpret_cast<const float *>(in + pc.in_n[seg]) + 3 * (size_t)local;
                nx = nr[0], ny = nr[1], nz = nr[2];
            } else {
                const float4 b = in[(size_t)pc.in_n[seg] + local]; // nx ny nz curvature
                nx = b.x, ny = b.y, nz = b.z, curvature = b.w;
            }
        }
        if (is_src) {
            const double *t = pc.init;
            int n_apply = 1;
            if (kUndistort && pc.undistort) {
                if (cls == MULLS_VERTEX) {
                    n_apply = 2; // not undistorted and not re-cloned: the initial guess lands twice (reference behaviour)
                } else {
                    const float curv = curvature; // timestamp ratio of the point inside its frame
                    if (!(curv < 0.0f || (double)curv > 1.0)) {
                        const double s = (double)curv;
                        double scale0, scale1;
                        if (pc.ud_linear) {
                            scale0 = 1.0 - s;
                            scale1 = s;
                        } else {
                            scale0 = sin((1.0 - s) * pc.ud_theta) / pc.ud_sin_theta;
                            scale1 = sin(s * pc.ud_theta) / pc.ud_sin_theta;
                        }
                        if (pc.ud_neg) scale1 = -scale1;
                        const double qx = scale1 * pc.ud_q[0], qy = scale1 * pc.ud_q[1], qz = scale1 * pc.ud_q[2],
                                     qw = scale0 + scale1 * pc.ud_q[3];
                        const double vx = x, vy = y, vz = z;
                        double ux = qy * vz - qz * vy, uy = qz * vx - qx * vz, uz = qx * vy - qy * vx;
                        ux += ux, uy += uy, uz += uz;
                        const double rx = vx + qw * ux + (qy * uz - qz * uy);
                        const double ry = vy + qw * uy + (qz * ux - qx * uz);
                        const double rz = vz + qw * uz + (qx * uy - qy * ux);
                        x = (float)(rx + s * pc.ud_t[0]);
                        y = (float)(ry + s * pc.ud_t[1]);
                        z = (float)(rz + s * pc.ud_t[2]);
                    }
                }
            }
            for (int rep = 0; rep < n_apply; ++rep) {
                const double px = x, py = y, pz = z, qx = nx, qy = ny, qz = nz;
                x = (float)(t[0] * px + t[1] * py + t[2] * pz + t[3]);
                y = (float)(t[4] * px + t[5] * py + t[6] * pz + t[7]);
                z = (float)(t[8] * px + t[9] * py + t[10] * pz + t[11]);
                nx = (float)(t[0] * qx + t[1] * qy + t[2] * qz);
                ny = (float)(t[4] * qx + t[5] * qy + t[6] * qz);
                nz = (float)(t[8] * qx + t[9] * qy + t[10] * qz);
            }
        }
        A.stg_pos[gi] = make_float4(x, y, z, intensity);
        A.stg_nrm[gi] = make_float4(nx, ny, nz, __int_as_float((int)local));
    }
    // bbox: source ground/pillar/facade (cregistration.hpp:2912-2915) and all target points (grid extent)
    const bool want = is_src ? (cls == MULLS_GROUND || cls == MULLS_PILLAR || cls == MULLS_FACADE) : true;
    if (!want) return; // block-uniform
    float mn[3] = {valid ? x : FLT_MAX, valid ? y : FLT_MAX, valid ? z : FLT_MAX};
    float mx[3] = {valid ? x : -FLT_MAX, valid ? y : -FLT_MAX, valid ? z : -FLT_MAX};
#pragma unroll
    for (int d = 0; d < 3; ++d)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn[d] = fminf(mn[d], __shfl_xor_sync(0xffffffffu, mn[d], o));
            mx[d] = fmaxf(mx[d], __shfl_xor_sync(0xffffffffu, mx[d], o));
        }
    __shared__ float s_mn[kIngestBlock / 32][3], s_mx[kIngestBlock / 32][3];
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int d = 0; d < 3; ++d) s_mn[threadIdx.x >> 5][d] = mn[d], s_mx[threadIdx.x >> 5][d] = mx[d];
    }
    __syncthreads();
    if (threadIdx.x < 6) { // one atomic per block and bound
        const int d = threadIdx.x % 3;
        const bool is_max = threadIdx.x >= 3;
        float v = is_max ? s_mx[0][d] : s_mn[0][d];
        for (int w = 1; w < kIngestBlock / 32; ++w) v = is_max ? fmaxf(v, s_mx[w][d]) : fminf(v, s_mn[w][d]);
        int *bb = is_src ? A.ps[cd.pair].bb_src : A.ps[cd.pair].bb_tgt;
        if (is_max) atomicMax(&bb[3 + d], float_to_ordered(v));
        else atomicMin(&bb[d], float_to_ordered(v));
    }
}

// ---- k_pair_setup: one thread per pair. Intersection bbox (utility.hpp:858-866, pad 1.0,
//      cregistration.hpp:2907-2916), grid geometry, initial state (:1144-1164).
__global__ void k_pair_setup(DeviceArrays A, int n_pairs, float h0_min) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const PairConst &pc = A.pc[p];
    PairState &ps = A.ps[p];
    double smin[3], smax[3], tmin[3], tmax[3];
    for (int d = 0; d < 3; ++d) {
        smin[d] = (double)ordered_to_float(ps.bb_src[d]);
        smax[d] = (double)ordered_to_float(ps.bb_src[3 + d]);
        tmin[d] = (double)ordered_to_float(ps.bb_tgt[d]);
        tmax[d] = (double)ordered_to_float(ps.bb_tgt[3 + d]);
    }
    const double big = 1.7976931348623157e308;
    double gmin[3], gmax[3];
    if (pc.apply_filter) {
        const float pad = 1.0f;
        for (int d = 0; d < 3; ++d) {
            // an empty source bbox stays at +/-FLT_MAX here (DBL_MAX in the reference): either way
            // the intersection is empty and every point is filtered out.
            double lo = (pc.tbound[d] > smin[d]) ? pc.tbound[d] : smin[d];
            double hi = (pc.tbound[3 + d] < smax[d]) ? pc.tbound[3 + d] : smax[d];
            ps.ibb[d] = lo - (double)pad;
            ps.ibb[3 + d] = hi + (double)pad;
            gmin[d] = fmax(tmin[d], ps.ibb[d]);
            gmax[d] = fmin(tmax[d], ps.ibb[3 + d]);
        }
    } else {
        for (int d = 0; d < 3; ++d) {
            ps.ibb[d] = -big;
            ps.ibb[3 + d] = big;
            gmin[d] = tmin[d];
            gmax[d] = tmax[d];
        }
    }
    double ext = 0.0;
    for (int d = 0; d < 3; ++d) {
        if (!(gmax[d] >= gmin[d])) {
            gmin[d] = 0.0;
            gmax[d] = 0.0;
        }
        ext = fmax(ext, gmax[d] - gmin[d]);
    }
    const float h0 = grid_h0(ext, h0_min); // (search_core.cuh)
    ps.h0 = h0;
    ps.inv_h0 = 1.0f / h0; // power of two times h0_min: exact when h0_min is a power of two
    for (int d = 0; d < 3; ++d) ps.origin[d] = (float)gmin[d] - 2.0f * h0;
    // number of levels: the top level's guaranteed coverage 0.999 * h_top / 2 must reach the largest search radius
    // 2.5 * thre that the threshold schedule reaches in max_iter iterations (grid_levels, search_core.cuh)
    int L = grid_levels(h0, pc.thre_unit, pc.thre_min, pc.thre_rate, pc.max_iter);
    // normal shooting needs the exact 10 nearest targets with no distance bound: full pyramid, whose top 2x2x2
    // block (2 x 2048 level-0 cells per axis) spans the whole grid
    if (pc.normal_shooting) L = kMaxLevels;
    ps.n_levels = L;

    for (int i = 0; i < 16; ++i) {
        ps.T_total[i] = pc.init[i];
        ps.T_inc[i] = (i % 5 == 0) ? 1.0 : 0.0;
    }
    for (int i = 0; i < 36; ++i) ps.cofactor[i] = ps.info[i] = (i % 7 == 0) ? 1.0 : 0.0;
    for (int i = 0; i < 6; ++i) ps.x[i] = 0.0;
    ps.sigma2 = 1.0;
    ps.thre = pc.thre_unit;
    ps.confidence = 1.0f;
    ps.status = kRunning;
    ps.code = 0;
    ps.iter = 0;
    ps.iters_entered = 0;
    ps.final_buf = 0;
    ps.alg_bytes = 0;
    if (pc.max_iter <= 0) {
        ps.status = kDone;
        const int left = atomicSub(A.running, 1) - 1;
        *A.h_running = left;
        __threadfence_system();
    }
}

// ---- k_make_keys: intersection filter (cfilter.hpp:950-981: strictly inside) + 64-bit sort key
//      [pair*12+seg | morton36(cell)]; filtered-out points sort to the very end.
__global__ void __launch_bounds__(kIngestBlock) k_make_keys(DeviceArrays A, int sort_sources) {
    const ChunkDesc cd = A.in_chunks[blockIdx.x];
    const PairConst &pc = A.pc[cd.pair];
    PairState &ps = A.ps[cd.pair];
    const uint32_t seg = cd.seg;
    const uint32_t local = cd.first + threadIdx.x;
    const bool valid = local < pc.in_n[seg];
    bool inside = false;
    if (valid) {
        const size_t gi = (size_t)pc.in_off[seg] + local;
        const float4 p = A.stg_pos[gi];
        const double *b = ps.ibb;
        inside = (double)p.x > b[0] && (double)p.x < b[3] && (double)p.y > b[1] && (double)p.y < b[4] &&
                 (double)p.z > b[2] && (double)p.z < b[5];
        uint64_t key = ~0ull;
        if (inside) {
            const int hi = (1 << kCoordBits) - 1;
            int cx = (int)floorf((p.x - ps.origin[0]) * ps.inv_h0);
            int cy = (int)floorf((p.y - ps.origin[1]) * ps.inv_h0);
            int cz = (int)floorf((p.z - ps.origin[2]) * ps.inv_h0);
            // targets are inside the grid by construction; sources may stick out (clamped: the
            // source key only orders threads for locality, it never enters a distance decision)
            cx = min(max(cx, 0), hi);
            cy = min(max(cy, 0), hi);
            cz = min(max(cz, 0), hi);
            key = ((uint64_t)(cd.pair * kNumSegs + seg) << 36) | morton36((uint32_t)cx, (uint32_t)cy, (uint32_t)cz);
            // (study switch: sources left in the caller's order — nothing but the search's locality depends on it)
            if (!sort_sources && seg >= kNumClasses) key = ((uint64_t)(cd.pair * kNumSegs + seg) << 36) | (uint64_t)local;
        }
        A.keys_a[gi] = key;
        A.vals_a[gi] = (uint32_t)gi;
    }
    const unsigned ballot = __ballot_sync(0xffffffffu, inside);
    if ((threadIdx.x & 31) == 0 && ballot) atomicAdd(&ps.seg_count[seg], (unsigned)__popc(ballot));
}

// ---- keep_less_source_pts (cregistration.hpp:2866-2892) -> random_downsample_pcl (cfilter.hpp:606-628) --------
// The reference samples with pcl::RandomSample seeded by time(NULL); here the kept subset of a cloud is the k
// points with the smallest key splitmix64(seed, cloud, original index) (uniform, reproducible, order preserved).
// k-th smallest key per cloud = 8-pass radix select (256-bin histogram per pass), then one marking pass.
__device__ __forceinline__ uint64_t sample_key(uint32_t seed, uint32_t cloud_id, uint32_t index) {
    uint64_t z = (((uint64_t)seed << 40) ^ ((uint64_t)cloud_id << 32) ^ (uint64_t)index) + 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

__global__ void k_keepless_plan(DeviceArrays A, int n_pairs) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const PairConst &pc = A.pc[p];
    PairState &ps = A.ps[p];
    for (int s = 0; s < kNumSegs; ++s) {
        ps.kl_keep[s] = -1;
        ps.kl_prefix[s] = 0;
        ps.kl_rank[s] = 0;
        for (int b = 0; b < 256; ++b) ps.kl_hist[s][b] = 0;
    }
    if (!pc.keep_less) return;
    const int S = kNumClasses; // source segments follow the six target segments
    auto plan = [&](int seg, int keep) { // random_downsample_pcl: untouched if size <= keep_number
        if ((int)ps.seg_count[seg] > keep) {
            ps.kl_keep[seg] = keep;
            ps.kl_rank[seg] = (uint32_t)keep;
        }
        return ((int)ps.seg_count[seg] > keep) ? keep : (int)ps.seg_count[seg];
    };
    // order and rates of :2882-2890 (target_down_rate 2, ground_down_rate 4, facade_down_rate 2)
    const int tg = plan(MULLS_GROUND, (int)(ps.seg_count[MULLS_GROUND] / 2));
    const int tf = plan(MULLS_FACADE, (int)(ps.seg_count[MULLS_FACADE] / 2));
    plan(S + MULLS_GROUND, tg / 4);
    plan(S + MULLS_FACADE, tf / 2);
    plan(S + MULLS_PILLAR, (int)ps.seg_count[MULLS_PILLAR]);
    plan(S + MULLS_BEAM, (int)ps.seg_count[MULLS_BEAM]);
    plan(S + MULLS_ROOF, (int)ps.seg_count[MULLS_ROOF]);
    plan(S + MULLS_VERTEX, (int)ps.seg_count[MULLS_VERTEX]);
}

// pass = 0..7: histogram of byte `pass` (from the top) of the keys whose higher bytes equal the prefix found so far
__global__ void __launch_bounds__(kIngestBlock) k_keepless_hist(DeviceArrays A, int pass) {
    const ChunkDesc cd = A.in_chunks[blockIdx.x];
    const PairConst &pc = A.pc[cd.pair];
    PairState &ps = A.ps[cd.pair];
    const uint32_t seg = cd.seg;
    if (ps.kl_keep[seg] <= 0) return; // untouched, or cleared entirely
    __shared__ uint32_t s_hist[256];
    s_hist[threadIdx.x] = 0; // kIngestBlock == 256
    __syncthreads();
    const uint32_t local = cd.first + threadIdx.x;
    if (local < pc.in_n[seg]) {
        const size_t gi = (size_t)pc.in_off[seg] + local;
        if (A.keys_a[gi] != ~0ull) {
            const uint64_t key = sample_key(pc.random_seed, seg, local);
            const int shift = 56 - 8 * pass;
            const bool match = (pass == 0) || ((key >> (shift + 8)) == (ps.kl_prefix[seg] >> (shift + 8)));
            if (match) atomicAdd(&s_hist[(key >> shift) & 0xff], 1u);
        }
    }
    __syncthreads();
    if (s_hist[threadIdx.x]) atomicAdd(&ps.kl_hist[seg][threadIdx.x], s_hist[threadIdx.x]);
}

__global__ void k_keepless_step(DeviceArrays A, int n_pairs, int pass) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    PairState &ps = A.ps[p];
    for (int s = 0; s < kNumSegs; ++s) {
        if (ps.kl_keep[s] <= 0) continue;
        uint32_t cum = 0, rank = ps.kl_rank[s];
        int d = 0;
        for (; d < 256; ++d) {
            const uint32_t h = ps.kl_hist[s][d];
            if (cum + h >= rank) break;
            cum += h;
        }
        ps.kl_prefix[s] |= (uint64_t)d << (56 - 8 * pass);
        ps.kl_rank[s] = rank - cum;
        for (int b = 0; b < 256; ++b) ps.kl_hist[s][b] = 0;
    }
}

// drop the points whose key exceeds the k-th smallest one (keys are a bijection of the index: exactly k remain)
__global__ void __launch_bounds__(kIngestBlock) k_keepless_mark(DeviceArrays A) {
    const ChunkDesc cd = A.in_chunks[blockIdx.x];
    const PairConst &pc = A.pc[cd.pair];
    PairState &ps = A.ps[cd.pair];
    const uint32_t seg = cd.seg;
    const int keep = ps.kl_keep[seg];
    if (keep < 0) return;
    const uint32_t local = cd.first + threadIdx.x;
    bool drop = false;
    if (local < pc.in_n[seg]) {
        const size_t gi = (size_t)pc.in_off[seg] + local;
        if (A.keys_a[gi] != ~0ull) {
            drop = (keep == 0) || sample_key(pc.random_seed, seg, local) > ps.kl_prefix[seg];
            if (drop) A.keys_a[gi] = ~0ull;
        }
    }
    const unsigned b = __ballot_sync(0xffffffffu, drop);
    if ((threadIdx.x & 31) == 0 && b) atomicSub(&ps.seg_count[seg], (unsigned)__popc(b));
}

// ---- k_seg_offsets: single block; exclusive scan of the valid counts in (pair, seg) order gives the
//      start of every segment in the sorted array; also per-class sizes and :1195-1201.
__global__ void k_seg_offsets(DeviceArrays A, int n_pairs) {
    __shared__ uint32_t carry;
    __shared__ uint32_t warp_sums[32];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int total = n_pairs * kNumSegs;
    for (int base = 0; base < total; base += blockDim.x) {
        const int i = base + threadIdx.x;
        uint32_t v = 0;
        if (i < total) v = A.ps[i / kNumSegs].seg_count[i % kNumSegs];
        uint32_t incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= o) incl += t;
        }
        if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t w = (threadIdx.x < (blockDim.x >> 5)) ? warp_sums[threadIdx.x] : 0;
            uint32_t wi = w;
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
                if (threadIdx.x >= o) wi += t;
            }
            warp_sums[threadIdx.x] = wi - w; // exclusive
        }
        __syncthreads();
        const uint32_t excl = carry + warp_sums[threadIdx.x >> 5] + incl - v;
        if (i < total) A.ps[i / kNumSegs].seg_start[i % kNumSegs] = excl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = excl + v;
        __syncthreads();
    }
    for (int p = threadIdx.x; p < n_pairs; p += blockDim.x) {
        PairState &ps = A.ps[p];
        const PairConst &pc = A.pc[p];
        for (int c = 0; c < kNumClasses; ++c) {
            ps.n_tgt[c] = (int)ps.seg_count[c];
            ps.n_src[c] = (int)ps.seg_count[kNumClasses + c];
            ps.n_src_g[c] = ps.n_src[c];
            ps.n_corr[c] = 0;
            ps.n_corr_last[c] = 0;
        }
        int cnt = 0;
        if (pc.used[MULLS_PILLAR]) cnt += ps.n_src[MULLS_PILLAR];
        if (pc.used[MULLS_FACADE]) cnt += ps.n_src[MULLS_FACADE];
        if (pc.used[MULLS_BEAM]) cnt += ps.n_src[MULLS_BEAM];
        ps.source_feature_points_count = cnt;
    }
}

// ---- k_gather: sorted order -> final SoA slices (targets, and source buffer 0)
__global__ void __launch_bounds__(256) k_gather(DeviceArrays A, const uint64_t *keys, const uint32_t *vals, uint32_t n_total) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_total) return;
    const uint64_t key = keys[i];
    if (key == ~0ull) return;
    const uint32_t sg = (uint32_t)(key >> 36);
    const uint32_t pair = sg / kNumSegs, seg = sg % kNumSegs;
    const PairConst &pc = A.pc[pair];
    const uint32_t local = i - A.ps[pair].seg_start[seg];
    const uint32_t v = vals[i];
    const float4 pos = A.stg_pos[v];
    const float4 nrm = A.stg_nrm[v];
    if (seg < kNumClasses) {
        const uint32_t d = pc.tgt_base[seg] + local;
        A.tgt_pos[d] = pos;
        A.tgt_nrm[d] = nrm;
    } else {
        const uint32_t d = pc.src_base[seg - kNumClasses] + local;
        float4 n2 = nrm;
        if (pc.sharded) n2.w = __int_as_float(__float_as_int(nrm.w) + (int)pc.src_index_base[seg - kNumClasses]);
        A.src_pos[0][d] = pos;
        A.src_nrm[0][d] = n2;
        A.src_prevj[0][d] = -1;
        A.src_cert[0][d] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// ---- hashed multi-level grid over a target class --------------------------------------------
// Entry = {key_lo, key_hi | child mask << 16, start, count} (grid_key.cuh); (0, 0) marks an empty slot.
__device__ __forceinline__ void hash_insert(HashEntry *table, uint32_t mask, uint32_t klo, uint32_t khi, uint32_t start) {
    uint32_t slot = cell_hash(klo, khi) & mask;
    const unsigned long long packed = (unsigned long long)klo | ((unsigned long long)khi << 32);
    while (true) {
        unsigned long long *kp = reinterpret_cast<unsigned long long *>(&table[slot]);
        unsigned long long old = atomicCAS(kp, 0ull, packed);
        if (old == 0ull) {
            table[slot].start = start;
            return;
        }
        slot = (slot + 1) & mask;
    }
}
// key_hi carries, above the 16 key bits, the 8-bit mask of existing children (set while closing cells)
__device__ __forceinline__ HashEntry *hash_find(HashEntry *table, uint32_t mask, uint32_t klo, uint32_t khi) {
    uint32_t slot = cell_hash(klo, khi) & mask;
    while (true) {
        const uint32_t lo = *reinterpret_cast<volatile uint32_t *>(&table[slot].key_lo);
        const uint32_t hi = *reinterpret_cast<volatile uint32_t *>(&table[slot].key_hi);
        if (lo == klo && (hi & kKeyHiMask) == khi) return &table[slot];
        if (lo == 0u && hi == 0u) return nullptr;
        slot = (slot + 1) & mask;
    }
}

// k_hash_build: thread i looks at the boundary between sorted elements i-1 and i. Where the Morton
// prefix changes, a new cell starts at every level up to the highest differing one.
//   mode 0: count the cells per (pair, class)          -> PairState::hash_entries
//   mode 1: open cells: insert {key, start}
//   mode 2: close cells: write the count of every cell the previous point ended
__global__ void __launch_bounds__(256) k_hash_build(DeviceArrays A, const uint64_t *keys, uint32_t n_total, int mode) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = i <= n_total;
    const uint64_t kcur = (in_range && i < n_total) ? keys[i] : ~0ull;
    const uint64_t kprev = (in_range && i > 0) ? keys[i - 1] : ~0ull;
    const bool cur_t = kcur != ~0ull && ((uint32_t)(kcur >> 36) % kNumSegs) < kNumClasses;
    const bool prev_t = kprev != ~0ull && ((uint32_t)(kprev >> 36) % kNumSegs) < kNumClasses;
    const bool same_seg = cur_t && prev_t && (kcur >> 36) == (kprev >> 36);
    const uint64_t mmask = (1ull << 36) - 1;
    int top = kMaxLevels - 1; // highest level at which the cell changes
    bool boundary = true;
    if (same_seg) {
        const uint64_t diff = (kcur ^ kprev) & mmask;
        if (diff == 0) boundary = false; // same finest cell: no boundary at any level
        else top = (63 - __clzll((long long)diff)) / 3;
    }
    if (mode == 0) {
        uint32_t sg = cur_t ? (uint32_t)(kcur >> 36) : 0xffffffffu;
        int cnt = 0;
        if (cur_t && boundary) {
            const int L = A.ps[sg / kNumSegs].n_levels;
            cnt = min(top, L - 1) + 1;
        }
        const unsigned grp = __match_any_sync(0xffffffffu, sg);
        if (grp == 0xffffffffu) {
            const int tot = __reduce_add_sync(0xffffffffu, cnt);
            if ((threadIdx.x & 31) == 0 && tot > 0 && cur_t)
                atomicAdd(&A.ps[sg / kNumSegs].hash_entries[sg % kNumSegs], (unsigned)tot);
        } else if (cnt > 0) {
            atomicAdd(&A.ps[sg / kNumSegs].hash_entries[sg % kNumSegs], (unsigned)cnt);
        }
        return;
    }
    if (!boundary || A.hash_used[1]) return;
    if (mode == 1) {
        if (!cur_t) return;
        const uint32_t sg = (uint32_t)(kcur >> 36);
        const uint32_t pair = sg / kNumSegs, cls = sg % kNumSegs;
        const PairState &ps = A.ps[pair];
        const int L = ps.n_levels;
        const uint32_t local = i - ps.seg_start[cls];
        HashEntry *table = A.hash + ps.hash_base[cls];
        const uint64_t m = kcur & mmask;
        const uint32_t x0 = compact12(m), y0 = compact12(m >> 1), z0 = compact12(m >> 2);
        for (int l = 0; l <= top && l < L; ++l)
            hash_insert(table, ps.hash_mask[cls], cell_key_lo(x0 >> l, y0 >> l, z0 >> l), cell_key_hi(z0 >> l, l), local);
    } else {
        if (!prev_t) return;
        const uint32_t sg = (uint32_t)(kprev >> 36);
        const uint32_t pair = sg / kNumSegs, cls = sg % kNumSegs;
        const PairState &ps = A.ps[pair];
        const int L = ps.n_levels;
        const uint32_t local_end = i - ps.seg_start[cls];
        HashEntry *table = A.hash + ps.hash_base[cls];
        const uint64_t m = kprev & mmask;
        const uint32_t x0 = compact12(m), y0 = compact12(m >> 1), z0 = compact12(m >> 2);
        for (int l = 0; l <= top && l < L; ++l) {
            const uint32_t x = x0 >> l, y = y0 >> l, z = z0 >> l;
            HashEntry *e = hash_find(table, ps.hash_mask[cls], cell_key_lo(x, y, z), cell_key_hi(z, l));
            if (e) e->count = local_end - e->start;
            if (l + 1 < L) { // tell the parent which of its 8 children exists (child = x bit | y bit << 1 | z bit << 2)
                HashEntry *par = hash_find(table, ps.hash_mask[cls], cell_key_lo(x >> 1, y >> 1, z >> 1), cell_key_hi(z >> 1, l + 1));
                if (par) atomicOr(&par->key_hi, 1u << (16 + ((x & 1u) | ((y & 1u) << 1) | ((z & 1u) << 2))));
            }
        }
    }
}

// k_hash_layout: single block. Power-of-two table per (pair, class) with load factor <= 0.5, carved out
// of the pool in order; flags overflow instead of writing out of bounds.
__global__ void k_hash_layout(DeviceArrays A, int n_pairs, int slack) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    // load factor <= 1/slack if the pool allows it (slack 4: a miss costs ~1.4 probes instead of 2.5 at 1/2), else
    // <= 0.5, else <= 0.8 (longer probe chains, same results), else give up
    for (int attempt = 0; attempt < 3; ++attempt) {
        uint64_t used = 0;
        bool overflow = false;
        for (int p = 0; p < n_pairs && !overflow; ++p) {
            PairState &ps = A.ps[p];
            for (int c = 0; c < kNumClasses; ++c) {
                const uint64_t want = (attempt == 0) ? (uint64_t)slack * ps.hash_entries[c] : (attempt == 1) ? 2ull * ps.hash_entries[c] : (5ull * ps.hash_entries[c]) / 4 + 1;
                uint32_t cap = 16;
                while (cap < want) cap <<= 1;
                if (used + cap > A.hash_pool_entries) {
                    overflow = true;
                    break;
                }
                ps.hash_base[c] = (uint32_t)used;
                ps.hash_mask[c] = cap - 1;
                used += cap;
            }
        }
        A.hash_used[0] = overflow ? 0u : (uint32_t)used;
        A.hash_used[1] = overflow ? 1u : 0u;
        if (!overflow) return;
    }
    // overflow: degenerate tables that are never searched (every kernel checks hash_used[1]); the run reports it
    for (int p = 0; p < n_pairs; ++p)
        for (int c = 0; c < kNumClasses; ++c) {
            A.ps[p].hash_base[c] = 0;
            A.ps[p].hash_mask[c] = 0;
        }
}

__global__ void __launch_bounds__(256) k_hash_clear(DeviceArrays A) {
    const uint32_t used = A.hash_used[0];
    const uint4 z = make_uint4(0, 0, 0, 0);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < used; i += gridDim.x * blockDim.x)
        reinterpret_cast<uint4 *>(A.hash)[i] = z;
}

} // namespace mulls
