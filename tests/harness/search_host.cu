// TEST INFRASTRUCTURE. Instantiates the `__host__ __device__` search of mulls_b200/csrc/search_core.cuh on the CPU
// over a grid built here with the same keys, hash and entry layout as k_hash_build (kernels_ingest.cuh), so that
// the CPU suite can compare the product's search logic with a brute-force scan / the oracle without a GPU, and
// count its work (probes, candidate evaluations, expansions) per query. Built by tests/test_search_core.py with
// nvcc (host code only; no CUDA call is made). The product never executes this instantiation.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <vector>

#include "../../mulls_b200/csrc/search_core.cuh"

using namespace mulls;

namespace {

struct HostGrid {
    std::vector<HashEntry> table;
    std::vector<float4> pos, nrm;
    std::vector<uint32_t> inv; // original index -> sorted position
    GridView g;
    uint32_t n_cells = 0;
    uint64_t chain_sum = 0;
};

struct Counters {
    uint64_t probes = 0, evals = 0, expands = 0, levels = 0, seed_probes = 0, seed_evals = 0, max_evals_query = 0, cur_evals = 0;
    void probe() { probes++; }
    void eval(int n) { evals += n, cur_evals += n; }
    void expand() { expands++; }
    void level() { levels++; }
    void seed_probe() { seed_probes++; }
    void seed_eval(int n) { seed_evals += n; }
};

void insert(HostGrid &G, uint32_t x, uint32_t y, uint32_t z, int level, uint32_t start, uint32_t count, uint32_t cmask) {
    const uint32_t klo = cell_key_lo(x, y, z), khi = cell_key_hi(z, level);
    uint32_t slot = cell_hash(klo, khi) & G.g.mask;
    uint64_t chain = 1;
    while (G.table[slot].key_lo != 0u || G.table[slot].key_hi != 0u) slot = (slot + 1) & G.g.mask, ++chain;
    G.table[slot] = HashEntry{klo, khi | (cmask << 16), start, count};
    G.n_cells++;
    G.chain_sum += chain;
}

} // namespace

extern "C" {

// pts: n x 4 floats (x y z _). Grid geometry as k_pair_setup would choose it (sh_h0_for, sh_levels_for) is supplied by
// the caller.
void *sh_build(const float *pts, uint32_t n, float ox, float oy, float oz, float h0, int n_levels, int leaf_count) {
    HostGrid *G = new HostGrid();
    std::vector<uint64_t> key(n);
    const float inv_h0 = 1.0f / h0;
    for (uint32_t i = 0; i < n; ++i) {
        int cx = (int)floorf((pts[4 * i + 0] - ox) * inv_h0), cy = (int)floorf((pts[4 * i + 1] - oy) * inv_h0),
            cz = (int)floorf((pts[4 * i + 2] - oz) * inv_h0);
        cx = std::min(std::max(cx, 0), 4095), cy = std::min(std::max(cy, 0), 4095), cz = std::min(std::max(cz, 0), 4095);
        key[i] = morton36((uint32_t)cx, (uint32_t)cy, (uint32_t)cz);
    }
    std::vector<uint32_t> order(n);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
    G->pos.resize(n + kScanOverrun), G->nrm.resize(n), G->inv.resize(n);
    std::vector<uint64_t> sk(n);
    for (uint32_t s = 0; s < n; ++s) {
        const uint32_t i = order[s];
        G->pos[s] = make_float4(pts[4 * i], pts[4 * i + 1], pts[4 * i + 2], 0.f);
        float w;
        const int oi = (int)i;
        std::memcpy(&w, &oi, 4);
        G->nrm[s] = make_float4(0.f, 0.f, 1.f, w);
        G->inv[i] = s;
        sk[s] = key[i];
    }
    // cells of every level: runs of equal (code >> 3l)
    size_t cells = 0;
    for (int l = 0; l < n_levels; ++l)
        for (uint32_t s = 0; s < n; ++s)
            if (s == 0 || (sk[s] >> (3 * l)) != (sk[s - 1] >> (3 * l))) ++cells;
    uint32_t cap = 16;
    while (cap < 2 * cells) cap <<= 1;
    G->table.assign(cap, HashEntry{0, 0, 0, 0});
    G->g.table = nullptr;
    G->g.mask = cap - 1;
    for (int l = 0; l < n_levels; ++l) {
        uint32_t s = 0;
        while (s < n) {
            const uint64_t code = sk[s] >> (3 * l);
            uint32_t e = s;
            uint32_t cmask = 0;
            while (e < n && (sk[e] >> (3 * l)) == code) {
                if (l > 0) cmask |= 1u << ((sk[e] >> (3 * (l - 1))) & 7u);
                ++e;
            }
            insert(*G, compact12(code), compact12(code >> 1), compact12(code >> 2), l, s, e - s, cmask);
            s = e;
        }
    }
    G->g.table = G->table.data();
    G->g.pos = G->pos.data();
    G->g.nrm = G->nrm.data();
    G->g.ox = ox, G->g.oy = oy, G->g.oz = oz, G->g.h0 = h0, G->g.inv_h0 = inv_h0;
    G->g.n_levels = n_levels;
    G->g.leaf_count = leaf_count;
    G->g.level_slack2 = 1.002001f;
    if (const char *e = getenv("MULLS_LEVEL_SLACK")) { // (study switch: scripts/studies/skip_certificate_study.py)
        const float sl = (float)atof(e);
        if (sl >= 1.0f) G->g.level_slack2 = 1.002001f * sl * sl;
    }
    return G;
}

void sh_free(void *h) { delete (HostGrid *)h; }

void sh_grid_info(void *h, uint64_t *out /*[3]: cells, table capacity, sum of insert chain lengths*/) {
    HostGrid *G = (HostGrid *)h;
    out[0] = G->n_cells, out[1] = G->table.size(), out[2] = G->chain_sum;
}

// q: m x 3 floats. seed: original target index of a candidate or -1 (may be null). Results as ORIGINAL target indices.
// reseed_d2: a seeded query whose seed is farther than this also tries the greedy seed (negative: never) — the seeding
// rule of k_search. stats[10] on entry: 1 = queue the small cells of a block (k_search from iteration defer_from_iter on).
// cert (may be null): the squared certificate radius of every query (nn_search_walk's return value).
int sh_search_cert(void *h, const float *q, const int *seed, uint32_t m, float r2_prune, int start_level, float reseed_d2,
                   int *out_idx, float *out_d2, uint64_t *stats /*[12]*/, uint32_t *evals_per_query /*[m] or null*/, float *cert) {
    HostGrid *G = (HostGrid *)h;
    const GridView &g = G->g;
    Counters C;
    const bool defer = stats[10] != 0;
    for (uint32_t i = 0; i < m; ++i) {
        const float px = q[3 * i], py = q[3 * i + 1], pz = q[3 * i + 2];
        float best_d2 = INFINITY;
        int best_j = -1;
        if (seed && seed[i] >= 0) {
            best_j = (int)G->inv[seed[i]];
            const float4 t = g.pos[best_j];
            best_d2 = flann_l2(px, py, pz, t.x, t.y, t.z);
        }
        if (best_j < 0 || (reseed_d2 >= 0.0f && best_d2 > reseed_d2)) {
            float d2 = INFINITY;
            int j = -1;
            walk_greedy_seed(g, px, py, pz, start_level, d2, j, C);
            if (j >= 0 && d2 < best_d2) best_d2 = d2, best_j = j;
        }
        C.cur_evals = 0;
        const float c2 = nn_search_walk(g, px, py, pz, r2_prune, start_level, defer, best_d2, best_j, C);
        if (cert) cert[i] = c2;
        C.max_evals_query = std::max(C.max_evals_query, C.cur_evals);
        if (evals_per_query) evals_per_query[i] = (uint32_t)C.cur_evals;
        out_d2[i] = best_d2;
        if (best_j >= 0) {
            int oi;
            std::memcpy(&oi, &g.nrm[best_j].w, 4);
            out_idx[i] = oi;
        } else {
            out_idx[i] = -1;
        }
    }
    stats[0] = C.probes, stats[2] = C.evals, stats[3] = C.expands, stats[4] = C.levels;
    stats[6] = C.seed_probes, stats[7] = C.seed_evals, stats[8] = C.max_evals_query;
    return 0;
}

int sh_search(void *h, const float *q, const int *seed, uint32_t m, float r2_prune, int start_level, float reseed_d2,
              int *out_idx, float *out_d2, uint64_t *stats /*[12]*/, uint32_t *evals_per_query /*[m] or null*/) {
    return sh_search_cert(h, q, seed, m, r2_prune, start_level, reseed_d2, out_idx, out_d2, stats, evals_per_query, nullptr);
}

// the grid geometry rules of k_pair_setup (search_core.cuh)
int sh_levels_for(float h0, float thre_unit, float thre_min, float thre_rate, int max_iter) {
    return grid_levels(h0, thre_unit, thre_min, thre_rate, max_iter);
}
float sh_h0_for(double ext, float h0_min) { return grid_h0(ext, h0_min); }

uint32_t sh_morton_roundtrip(uint32_t v) { return compact12(spread12(v)) == (v & 0xfffu) && compact12(spread12(v) << 1 >> 1) == (v & 0xfffu); }

} // extern "C"
