// Exact radius-bounded nearest neighbour on the multi-level hashed grid of one target class — the replacement of
// the kd-tree query of cregistration.hpp:1742-1745 (pcl::registration::CorrespondenceEstimation ->
// KdTreeFLANN::nearestKSearch, k = 1) — written as __host__ __device__ code: k_search (kernels_iterate.cuh) runs it
// on the device, tests/harness/search_host.cu instantiates the very same functions on the CPU, where the CPU suite
// checks them against a brute-force scan and the CPU restatement (tests/test_search_core.py). The product never runs the
// host instantiation.
//
// Result: the target j (index inside the Morton-sorted class slice) that minimises the total order
// (FLANN L2_Simple float distance, original index) among all targets with d2 <= r2_prune; the caller applies the
// reference's keep test in double.
//
// One query per thread, no cooperation between threads:
//   seed     a real candidate: the previous iteration's match, or (none / stale) a greedy descent from p's own cell
//   level    the smallest level l whose block guarantees coverage of the seed distance (cover_l below)
//   block    the 2x2x2 cells made of p's cell and, per axis, the neighbour on the side of the half-cell p lies in
//            (level 0: by the fractional position inside the cell). The block contains every target closer than
//            cover_l = 0.999 * h_l / 2 (level 0: 0.998 * h0 / 2 — the margins absorb the float rounding of the cell
//            assignment, <= 4096 * 2^-23 cells). Cells that can still beat the bound are walked one after the other
//   walk     depth first, nearest octant first: a cell holding more than leaf_count points is split — its entry
//            carries the mask of existing children, the children that can still beat the bound are pushed with their
//            box distance — and a small cell is examined where it is met (or, once the seeds are good, queued and
//            examined together with the block's other small cells in one go)
//            The top level of the full pyramid (2x2x2 cells) takes all 8 cells: the block is the whole grid
//   stop     best <= cover_l^2 (the best found is the global nearest) or cover_l^2 >= r2_prune; else next level
//   scan     a small cell's points four at a time: fused estimates of the squared distances, their minimum against the
//            best so far, and only then the exact FLANN distances with the tie rule (walk_scan_leaf)
//   bounds   optionally (WalkBounds) the search also returns a certificate: the squared radius inside which its answer
//            is the only target — what lets k_search keep a match in later iterations without searching
// The stack lives in thread-local arrays of 8-byte entries (local memory, L1-resident: measured faster than a
// shared-memory stack, and faster than two warp-cooperative / round-based forms that were tried — DESIGN.md section 5.1).
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>

#include "grid_key.cuh"

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#else
#error "compile with nvcc (host instantiation: nvcc -x cu, host code only)"
#endif

namespace mulls {

struct HashEntry { // 16 B, one 128-bit load per probe
    uint32_t key_lo, key_hi, start, count;
};

struct GridView {
    const HashEntry *table;
    uint32_t mask;
    const float4 *pos; // class slice
    const float4 *nrm; // class slice (w = original index, for tie-breaks)
    float ox, oy, oz, h0, inv_h0;
    int n_levels;
    int leaf_count; // cells with at most this many points are scanned, larger ones are split
    float level_slack2; // >= 1.002001: the start level's coverage must reach sqrt(level_slack2) x the seed distance
};

// ---- grid geometry of one pair (k_pair_setup; tests/harness/search_host.cu exports both rules to the CPU suite) ----
// level-0 cell size: h0_min, doubled until the extent plus two cells of margin on each side fits in 4096 - 4 cells
MULLS_HD float grid_h0(double ext, float h0_min) {
    float h0 = h0_min;
    while ((ext + 8.0 * h0) * 1.001 > (double)h0 * ((1 << kCoordBits) - 4)) h0 *= 2.0f;
    return h0;
}

// number of levels: the top level's guaranteed coverage 0.999 * h_top / 2 (nn_search_walk) must reach the largest search
// radius 2.5 * thre (filter_dis_times, cregistration.hpp:1707) of any iteration. solve_and_advance updates the threshold
// as thre <- max(thre / rate, thre_min) from thre_unit, so it grows when rate < 1 or thre_min > thre_unit; the largest
// value of iterations 0 .. max_iter - 1 is followed here in double (the float updates round by at most 64 half ulps,
// far inside the 1.0001 of rmax). A shrinking schedule gives thre_unit itself, bit for bit. Beyond the coverage of the
// full pyramid there is nothing left to add: its top level is the whole grid (nn_search_walk examines all 8 cells).
MULLS_HD int grid_levels(float h0, float thre_unit, float thre_min, float thre_rate, int max_iter) {
    float thre_max = thre_unit;
    double t = (double)thre_unit;
    for (int k = 1; k < max_iter; ++k) {
        t = t / (double)thre_rate;
        if (!(t > (double)thre_min)) t = (double)thre_min;
        if (t > (double)thre_max) thre_max = (float)t;
    }
    const float rmax = 2.5f * thre_max * 1.0001f;
    int L = 2; // level l's 2x2x2 block covers 0.999 * h0 * 2^(l-1)
    while (L < kMaxLevels && 0.999f * 0.5f * h0 * (float)(1 << (L - 1)) < rmax) ++L;
    return L;
}

struct NoStats {
    MULLS_HD void probe() {}
    MULLS_HD void eval(int) {}
    MULLS_HD void expand() {}
    MULLS_HD void level() {}
    MULLS_HD void seed_probe() {}
    MULLS_HD void seed_eval(int) {}
};

MULLS_HD uint4 ld_entry(const HashEntry *e) {
#ifdef __CUDA_ARCH__
    return __ldg(reinterpret_cast<const uint4 *>(e));
#else
    return *reinterpret_cast<const uint4 *>(e);
#endif
}
MULLS_HD float4 ld_point(const float4 *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}
MULLS_HD int f2i_bits(float f) {
#ifdef __CUDA_ARCH__
    return __float_as_int(f);
#else
    union {
        float f;
        int i;
    } u;
    u.f = f;
    return u.i;
#endif
}

// index of the lowest set bit (v != 0)
MULLS_HD int lowest_bit(uint32_t v) {
#ifdef __CUDA_ARCH__
    return __ffs((int)v) - 1;
#else
    return __builtin_ctz(v);
#endif
}

// finish a probe whose first slot was loaded by the caller: follow the chain (rare at load factor <= 0.5)
MULLS_HD bool probe_finish(const GridView &g, uint32_t slot, uint4 e, uint32_t klo, uint32_t khi, uint32_t &start,
                           uint32_t &count, uint32_t &cmask) {
    while (true) {
        if (e.x == klo && (e.y & kKeyHiMask) == khi) {
            start = e.z;
            count = e.w;
            cmask = (e.y >> 16) & 0xffu;
            return true;
        }
        if (e.x == 0u && e.y == 0u) return false;
        slot = (slot + 1) & g.mask;
        e = ld_entry(&g.table[slot]);
    }
}

MULLS_HD bool probe_key(const GridView &g, uint32_t klo, uint32_t khi, uint32_t &start, uint32_t &count, uint32_t &cmask) {
    const uint32_t slot = cell_hash(klo, khi) & g.mask;
    return probe_finish(g, slot, ld_entry(&g.table[slot]), klo, khi, start, count, cmask);
}
MULLS_HD bool probe_cell(const GridView &g, uint32_t x, uint32_t y, uint32_t z, int level, uint32_t &start, uint32_t &count,
                         uint32_t &cmask) {
    return probe_key(g, cell_key_lo(x, y, z), cell_key_hi(z, level), start, count, cmask);
}

// distance along one axis from p to the slab [lo - margin, hi + margin]
MULLS_HD float slab_dist(float lo, float hi, float p, float margin) {
    return fmaxf(0.0f, fmaxf((lo - margin) - p, p - (hi + margin)));
}

// a cell packed into 8 bytes: .x = key_lo (x | y<<12 | (z&0xff)<<24), .y = z>>8 | level<<4 | child mask<<8
MULLS_HD uint2 pack_cell(uint32_t x, uint32_t y, uint32_t z, int lv, uint32_t cmask) {
    return make_uint2(cell_key_lo(x, y, z), (z >> 8) | ((uint32_t)lv << 4) | (cmask << 8));
}

MULLS_HD float i2f_bits(uint32_t u) {
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    union {
        uint32_t u;
        float f;
    } c;
    c.u = u;
    return c.f;
#endif
}
// second key word of a cell (8 significant bits: z >> 8 | (level + 1) << 4) + the upper 24 bits of a non-negative float
MULLS_HD uint32_t pack_meta(uint32_t khi, float d2) { return (khi & 0xffu) | ((uint32_t)f2i_bits(d2) & 0xffffff00u); }
MULLS_HD float meta_d2(uint32_t packed) { return i2f_bits(packed & 0xffffff00u); }

// index of the highest set bit (v != 0)
MULLS_HD int highest_bit(uint32_t v) {
#ifdef __CUDA_ARCH__
    return 31 - __clz((int)v);
#else
    return 31 - __builtin_clz(v);
#endif
}

constexpr int kWalkStack = 48; // DFS entries: at most 7 stay behind per descended level
constexpr int kWalkQueue = 8;  // small cells of one block whose scan is deferred to the end of its traversal

// What a finished search knows beyond its answer (all squared distances from the query): `second` — the closest
// examined candidate other than the answer; `pruned` — the closest cell (box distance) that was left out because it
// could not beat the bound. With the coverage radius of the last block they bound from below the distance of EVERY
// target other than the answer: the certificate that lets a later iteration keep the match without searching
// (k_search: a query that has moved by delta keeps its match q if |p - q| + delta < that bound).
struct WalkBounds {
    float second = INFINITY, pruned = INFINITY;
    MULLS_HD void see(float d2) { second = fminf(second, d2); }
    MULLS_HD void prune(float d2) { pruned = fminf(pruned, d2); }
    MULLS_HD float radius2(float cover2) const { return fminf(fminf(second, pruned), cover2); }
};
// the same interface doing nothing: searches whose certificate nobody will read (the first iterations)
struct NoBounds {
    MULLS_HD void see(float) {}
    MULLS_HD void prune(float) {}
    MULLS_HD float radius2(float) const { return 0.0f; }
};

// one candidate under the total order (FLANN float distance, original index)
template <class Bounds>
MULLS_HD void walk_consider(const GridView &g, float d2, uint32_t jj, float &best_d2, int &best_j, Bounds &wb) {
    if (d2 < best_d2) {
        wb.see(best_d2); // (the displaced candidate; +inf while there was none)
        best_d2 = d2;
        best_j = (int)jj;
    } else if ((int)jj != best_j) {
        wb.see(d2);
        if (d2 == best_d2 && best_j >= 0) {
            const int oj = f2i_bits(ld_point(&g.nrm[jj]).w);
            const int ob = f2i_bits(ld_point(&g.nrm[best_j]).w);
            if (oj < ob) best_j = (int)jj;
        }
    }
}

// fused estimate of the squared distance: within 6e-7 relative of flann_l2 (both are a few roundings away from the real
// value) — only ever used to decide whether the exact distance has to be looked at
MULLS_HD float approx_l2(float px, float py, float pz, float qx, float qy, float qz) {
    const float dx = px - qx, dy = py - qy, dz = pz - qz;
#ifdef __CUDA_ARCH__
    return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, dx * dx));
#else
    return fmaf(dz, dz, fmaf(dy, dy, dx * dx));
#endif
}

// examine the points [start, start+count) of a small cell (count >= 1): FLANN distance, total order (d2, original index).
// Four candidates per trip (independent loads at fixed offsets from one address): the fused estimates are reduced to
// their minimum, and only a group whose minimum could reach the best so far is looked at exactly, point by point — with
// a real candidate as the seed that is the exception. The last group of a cell may read up to two points past the
// cell (their estimates are replaced by +inf): the position array carries kScanOverrun spare elements at its end.
constexpr int kScanOverrun = 4;
template <class Bounds>
MULLS_HD void walk_scan_leaf(const GridView &g, float px, float py, float pz, uint32_t start, uint32_t count, float &best_d2,
                             int &best_j, Bounds &wb) {
    const uint32_t end = start + count;
    uint32_t jj = start;
    for (; jj + 4 <= end; jj += 4) {
        const float4 *b = &g.pos[jj];
        const float4 q0 = ld_point(b), q1 = ld_point(b + 1), q2 = ld_point(b + 2), q3 = ld_point(b + 3);
        const float a0 = approx_l2(px, py, pz, q0.x, q0.y, q0.z), a1 = approx_l2(px, py, pz, q1.x, q1.y, q1.z);
        const float a2 = approx_l2(px, py, pz, q2.x, q2.y, q2.z), a3 = approx_l2(px, py, pz, q3.x, q3.y, q3.z);
        const float m = fminf(fminf(a0, a1), fminf(a2, a3));
        const float ml = m * 0.999999f; // below the exact float distance of every point of the group
        if (ml <= best_d2) {
            walk_consider(g, flann_l2(px, py, pz, q0.x, q0.y, q0.z), jj, best_d2, best_j, wb);
            walk_consider(g, flann_l2(px, py, pz, q1.x, q1.y, q1.z), jj + 1, best_d2, best_j, wb);
            walk_consider(g, flann_l2(px, py, pz, q2.x, q2.y, q2.z), jj + 2, best_d2, best_j, wb);
            walk_consider(g, flann_l2(px, py, pz, q3.x, q3.y, q3.z), jj + 3, best_d2, best_j, wb);
        } else {
            wb.see(ml);
        }
    }
    if (jj < end) { // 1..3 points left
        const float4 *b = &g.pos[jj];
        const float4 q0 = ld_point(b), q1 = ld_point(b + 1), q2 = ld_point(b + 2);
        const bool v1 = jj + 1 < end, v2 = jj + 2 < end;
        const float a0 = approx_l2(px, py, pz, q0.x, q0.y, q0.z);
        const float a1 = v1 ? approx_l2(px, py, pz, q1.x, q1.y, q1.z) : INFINITY;
        const float a2 = v2 ? approx_l2(px, py, pz, q2.x, q2.y, q2.z) : INFINITY;
        const float m = fminf(a0, fminf(a1, a2));
        const float ml = m * 0.999999f;
        if (ml <= best_d2) {
            walk_consider(g, flann_l2(px, py, pz, q0.x, q0.y, q0.z), jj, best_d2, best_j, wb);
            if (v1) walk_consider(g, flann_l2(px, py, pz, q1.x, q1.y, q1.z), jj + 1, best_d2, best_j, wb);
            if (v2) walk_consider(g, flann_l2(px, py, pz, q2.x, q2.y, q2.z), jj + 2, best_d2, best_j, wb);
        } else {
            wb.see(ml);
        }
    }
}

// No (usable) candidate yet: walk greedily from p's own cell (first level, from `l` upwards, at which it exists) down
// through the nearest existing child to a small cell and take its best point as the seed. A handful of probes, and
// the exact search that follows has a tight bound from its first cell on. Ties are settled by the exact search.
template <class Stats>
MULLS_HD void walk_greedy_seed(const GridView &g, float px, float py, float pz, int l, float &best_d2, int &best_j, Stats &st) {
    const int c0x = (int)floorf((px - g.ox) * g.inv_h0);
    const int c0y = (int)floorf((py - g.oy) * g.inv_h0);
    const int c0z = (int)floorf((pz - g.oz) * g.inv_h0);
    const int L = g.n_levels;
    l = (l < 1) ? 1 : ((l < L - 1) ? l : L - 1);
    for (int lr = l; lr < L && best_j < 0; ++lr) {
        const int ncell = 4096 >> lr;
        int cx = c0x >> lr, cy = c0y >> lr, cz = c0z >> lr;
        if (!(cx >= 0 && cy >= 0 && cz >= 0 && cx < ncell && cy < ncell && cz < ncell)) break;
        for (int lv = lr;; --lv) {
            uint32_t start, count, cmask;
            st.seed_probe();
            if (!probe_cell(g, (uint32_t)cx, (uint32_t)cy, (uint32_t)cz, lv, start, count, cmask)) break; // only possible at lv == lr
            if (count <= (uint32_t)g.leaf_count || lv == 0) {
                st.seed_eval((int)count);
                NoBounds unused; // (the exact search that follows examines this cell again)
                walk_scan_leaf(g, px, py, pz, start, count, best_d2, best_j, unused);
                break;
            }
            const float hl = g.h0 * (float)(1 << lv);
            const int ox = (px >= g.ox + ((float)cx + 0.5f) * hl) ? 1 : 0;
            const int oy = (py >= g.oy + ((float)cy + 0.5f) * hl) ? 1 : 0;
            const int oz = (pz >= g.oz + ((float)cz + 0.5f) * hl) ? 1 : 0;
            int ch = ox | (oy << 1) | (oz << 2);
            if (!((cmask >> ch) & 1u)) ch = cmask ? lowest_bit(cmask) : -1; // any existing child still yields a valid seed
            if (ch < 0) break;
            cx = 2 * cx + (ch & 1), cy = 2 * cy + ((ch >> 1) & 1), cz = 2 * cz + (ch >> 2);
        }
    }
}

// distance along one axis from p to the (slightly inflated) extent of cell x at a level with cell size H
MULLS_HD float walk_axis_dist(float o, float H, int x, float p, float margin) {
    const float lo = o + (float)x * H - margin, hi = o + (float)(x + 1) * H + margin;
    return fmaxf(0.0f, fmaxf(lo - p, p - hi));
}

// best_d2 / best_j come in seeded: (INFINITY, -1) or a real candidate. defer_scan: queue the small cells of a block
// and examine them together after its traversal (pays once the seeds are good).
// Returns the squared certificate radius: every target other than the answer is at least that far (squared) from p
// (Bounds = WalkBounds; with NoBounds nothing is tracked and 0 — no certificate — is returned).
template <class Bounds, class Stats>
MULLS_HD float nn_search_walk_b(const GridView &g, float px, float py, float pz, float r2_prune, int start_level, bool defer_scan,
                                float &best_d2, int &best_j, Stats &st) {
    Bounds wb = Bounds();
    const float fx = (px - g.ox) * g.inv_h0, fy = (py - g.oy) * g.inv_h0, fz = (pz - g.oz) * g.inv_h0;
    const float flx = floorf(fx), fly = floorf(fy), flz = floorf(fz);
    const int c0x = (int)flx, c0y = (int)fly, c0z = (int)flz;
    const int L = g.n_levels;
    const float margin = 1e-3f * g.h0; // covers the float rounding of the cell assignment
    // stack entry, 8 bytes: the first key word of the cell, and the second (its 8 significant bits) packed with the upper
    // 24 bits of the cell's box distance — truncating a positive float only lowers it, so pruning stays conservative
    uint32_t st_cell[kWalkStack], st_meta[kWalkStack];
    uint32_t q_start[kWalkQueue], q_count[kWalkQueue];
    int nq = 0;
    int l = (start_level < 1) ? 1 : ((start_level < L - 1) ? start_level : L - 1);
    if (best_j >= 0) { // seeded: the smallest level whose coverage reaches the seed (level 0: 0.998 * h0 / 2).
        // Only a starting point — the stop test below is what makes the result exact — so the level comes from the
        // exponent of (need / cover_1)^2 instead of a square root and a division: floor(log2 t) = floor(log2 t^2) >> 1
        const float c1 = 0.999f * 0.5f * g.h0, c0 = 0.998f * 0.5f * g.h0;
        const float t2 = (g.level_slack2 * best_d2) * (1.0f / (c1 * c1));
        if (t2 <= 1.0f) l = (g.level_slack2 * best_d2 <= c0 * c0) ? 0 : 1;
        else l = ((int)((f2i_bits(t2) >> 23) & 0xff) - 127 >> 1) + 1;
        l = (l < L - 1) ? l : L - 1;
    }
    for (;; ++l) {
        st.level();
        const float H = g.h0 * (float)(1 << l);
        const int ncell = (1 << kCoordBits) >> l;
        const bool whole = ncell == 2; // top of the full pyramid: its 8 cells ARE the grid, all of them are walked
        int xs[2], ys[2], zs[2];
        xs[0] = c0x >> l, ys[0] = c0y >> l, zs[0] = c0z >> l;
        if (whole) { // p's own cell first where p is inside the grid
            xs[0] = (xs[0] > 0) ? 1 : 0, ys[0] = (ys[0] > 0) ? 1 : 0, zs[0] = (zs[0] > 0) ? 1 : 0;
            xs[1] = xs[0] ^ 1, ys[1] = ys[0] ^ 1, zs[1] = zs[0] ^ 1;
        } else if (l == 0) { // side of the half-cell p lies in: by the fractional position inside the level-0 cell
            xs[1] = xs[0] + (((fx - flx) >= 0.5f) ? 1 : -1);
            ys[1] = ys[0] + (((fy - fly) >= 0.5f) ? 1 : -1);
            zs[1] = zs[0] + (((fz - flz) >= 0.5f) ? 1 : -1);
        } else {
            xs[1] = xs[0] + (((c0x >> (l - 1)) & 1) ? 1 : -1);
            ys[1] = ys[0] + (((c0y >> (l - 1)) & 1) ? 1 : -1);
            zs[1] = zs[0] + (((c0z >> (l - 1)) & 1) ? 1 : -1);
        }
        float ex[2], ey[2], ez[2];
        bool vx[2], vy[2], vz[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            vx[i] = xs[i] >= 0 && xs[i] < ncell;
            vy[i] = ys[i] >= 0 && ys[i] < ncell;
            vz[i] = zs[i] >= 0 && zs[i] < ncell;
        }
        // p lies inside its own cell (the margin covers the rounding of the cell assignment): only the three
        // neighbour slabs are at a distance — except on the whole grid, whose first cells are only the nearest ones
        ex[0] = ey[0] = ez[0] = 0.0f;
        if (whole) {
            ex[0] = walk_axis_dist(g.ox, H, xs[0], px, margin);
            ey[0] = walk_axis_dist(g.oy, H, ys[0], py, margin);
            ez[0] = walk_axis_dist(g.oz, H, zs[0], pz, margin);
            ex[0] *= ex[0], ey[0] *= ey[0], ez[0] *= ez[0];
        }
        ex[1] = walk_axis_dist(g.ox, H, xs[1], px, margin);
        ey[1] = walk_axis_dist(g.oy, H, ys[1], py, margin);
        ez[1] = walk_axis_dist(g.oz, H, zs[1], pz, margin);
        ex[1] *= ex[1], ey[1] *= ey[1], ez[1] *= ez[1];
        // live cells of the block as a bit mask, then one loop trip per LIVE cell
        uint32_t live = 0;
        {
            const float bound0 = fminf(best_d2, r2_prune) * 1.0001f + 1e-12f;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int i = k & 1, j = (k >> 1) & 1, m = k >> 2;
                const float dk = ex[i] + ey[j] + ez[m];
                if (vx[i] && vy[j] && vz[m]) {
                    if (dk <= bound0) live |= 1u << k;
                    else wb.prune(dk);
                }
            }
        }
#pragma unroll 1
        while (live) { // lowest bit first: k = 0 is p's own cell
            const int k = lowest_bit(live);
            live &= live - 1;
            const int i = k & 1, j = (k >> 1) & 1, m = k >> 2;
            int sp = 0;
            st_cell[0] = cell_key_lo((uint32_t)xs[i], (uint32_t)ys[j], (uint32_t)zs[m]);
            st_meta[0] = pack_meta(cell_key_hi((uint32_t)zs[m], l), ex[i] + ey[j] + ez[m]);
            sp = 1;
            while (sp > 0) {
                --sp;
                const uint32_t cell = st_cell[sp], packed = st_meta[sp];
                const float cell_d2 = meta_d2(packed);
                // a cell farther than the best so far (or than the radius) cannot change the result
                if (cell_d2 > fminf(best_d2, r2_prune) * 1.0001f + 1e-12f) {
                    wb.prune(cell_d2);
                    continue;
                }
                const uint32_t meta = packed & 0xffu;
                uint32_t start, count, cmask;
                st.probe();
                if (!probe_key(g, cell, meta, start, count, cmask)) continue;
                const int lv = (int)((meta >> 4) & 0xfu) - 1;
                if (count <= (uint32_t)g.leaf_count || lv == 0 || sp + 8 > kWalkStack) {
                    if (defer_scan && nq < kWalkQueue) { // examined together with the block's other small cells
                        q_start[nq] = start;
                        q_count[nq] = count;
                        ++nq;
                    } else {
                        st.eval((int)count);
                        walk_scan_leaf(g, px, py, pz, start, count, best_d2, best_j, wb);
                    }
                } else {
                    st.expand();
                    const int cx = (int)(cell & 0xfffu), cy = (int)((cell >> 12) & 0xfffu), cz = (int)((cell >> 24) | ((meta & 0xfu) << 8));
                    const float hc = 0.5f * g.h0 * (float)(1 << lv);
                    float ax[2], ay[2], az[2];
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        ax[b] = walk_axis_dist(g.ox, hc, 2 * cx + b, px, margin);
                        ay[b] = walk_axis_dist(g.oy, hc, 2 * cy + b, py, margin);
                        az[b] = walk_axis_dist(g.oz, hc, 2 * cz + b, pz, margin);
                        ax[b] *= ax[b], ay[b] *= ay[b], az[b] *= az[b];
                    }
                    // octant of p relative to the cell centre: the child with zero (or least) distance
                    const int near_child = (ax[1] < ax[0] ? 1 : 0) | (ay[1] < ay[0] ? 2 : 0) | (az[1] < az[0] ? 4 : 0);
                    const float bound = fminf(best_d2, r2_prune) * 1.0001f + 1e-12f;
                    // children that exist and can still beat the bound, as a bit mask ...
                    uint32_t pass = 0;
#pragma unroll
                    for (int ch = 0; ch < 8; ++ch) {
                        const float dc = ax[ch & 1] + ay[(ch >> 1) & 1] + az[ch >> 2];
                        if (dc <= bound) pass |= 1u << ch;
                        else if ((cmask >> ch) & 1u) wb.prune(dc);
                    }
                    pass &= cmask;
                    // ... re-indexed by c = ch ^ near_child (bit permutation by conditional swaps), so that the
                    // highest set bit is the farthest octant: pushed first, the nearest one last (popped first)
                    if (near_child & 1) pass = ((pass & 0x55u) << 1) | ((pass & 0xaau) >> 1);
                    if (near_child & 2) pass = ((pass & 0x33u) << 2) | ((pass & 0xccu) >> 2);
                    if (near_child & 4) pass = ((pass & 0x0fu) << 4) | ((pass & 0xf0u) >> 4);
                    while (pass) {
                        const int c = highest_bit(pass);
                        pass ^= 1u << c;
                        const int ch = c ^ near_child;
                        const uint32_t x2 = (uint32_t)(2 * cx + (ch & 1)), y2 = (uint32_t)(2 * cy + ((ch >> 1) & 1)), z2 = (uint32_t)(2 * cz + (ch >> 2));
                        st_cell[sp] = cell_key_lo(x2, y2, z2);
                        st_meta[sp] = pack_meta(cell_key_hi(z2, lv - 1), ax[ch & 1] + ay[(ch >> 1) & 1] + az[ch >> 2]);
                        ++sp;
                    }
                }
            }
        }
        // the queued small cells of this block
        for (int qi = 0; qi < nq; ++qi) {
            st.eval((int)q_count[qi]);
            walk_scan_leaf(g, px, py, pz, q_start[qi], q_count[qi], best_d2, best_j, wb);
        }
        nq = 0;
        // every closer target has been examined (the whole grid: every target has been examined or pruned)
        const float cover = whole ? INFINITY : (l == 0) ? 0.998f * 0.5f * g.h0 : 0.999f * 0.5f * H;
        const float cover2 = cover * cover;
        // every target outside the block is farther than `cover`; inside it, what was not examined is behind `pruned`.
        // Stopping at a top level below the full pyramid relies on grid_levels: its coverage reaches every radius the
        // pair searches with
        if (best_d2 <= cover2 || cover2 >= r2_prune || l == L - 1) // (global nearest found / whole radius examined / top)
            return wb.radius2(cover2);
    }
}
template <class Stats>
MULLS_HD float nn_search_walk(const GridView &g, float px, float py, float pz, float r2_prune, int start_level, bool defer_scan,
                              float &best_d2, int &best_j, Stats &st) {
    return nn_search_walk_b<WalkBounds>(g, px, py, pz, r2_prune, start_level, defer_scan, best_d2, best_j, st);
}

} // namespace mulls
