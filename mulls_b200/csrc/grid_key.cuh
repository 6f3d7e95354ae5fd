// Keys and hashing of the multi-level grid over one target class (built by k_hash_build, searched by
// search_core.cuh, kernels_pca.cuh). A level-l cell is named by its integer coordinates at that level
// (x, y, z < 4096 >> l) — no Morton spreading on the search side; the Morton code only orders the points.
//   key_lo = x | y << 12 | (z & 0xff) << 24
//   key_hi = z >> 8 | (l + 1) << 4          (bits 16..23 of the stored word carry the mask of existing children)
// (0, 0) marks an empty slot: l + 1 >= 1 keeps every real key non-zero.
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define MULLS_HD __host__ __device__ __forceinline__
#else
#define MULLS_HD inline
#endif

namespace mulls {

constexpr uint32_t kKeyHiMask = 0xffffu;
constexpr int kMaxLevels = 12; // levels 0 .. 11: the top level has 2 x 2 x 2 cells, the whole grid
constexpr int kCoordBits = 12; // Morton bits per axis: 4096 level-0 cells

// FLANN L2_Simple<float> accumulation (result += diff*diff per axis, float) — the distance the reference's
// kd-tree returns to CorrespondenceEstimation (cregistration.hpp:1745). Non-fused: the library is built with
// -fmad=false, the CPU harness with -ffp-contract=off.
MULLS_HD float flann_l2(float px, float py, float pz, float qx, float qy, float qz) {
    const float dx = px - qx, dy = py - qy, dz = pz - qz;
    return (dx * dx + dy * dy) + dz * dz;
}

MULLS_HD uint32_t cell_key_lo(uint32_t x, uint32_t y, uint32_t z) { return x | (y << 12) | ((z & 0xffu) << 24); }
MULLS_HD uint32_t cell_key_hi(uint32_t z, int level) { return (z >> 8) | ((uint32_t)(level + 1) << 4); }

// 32-bit mix of the two key words (multiplicative + xor-shift; linear probing at load factor <= 0.5)
MULLS_HD uint32_t cell_hash(uint32_t klo, uint32_t khi) {
    uint32_t h = klo * 0x9E3779B1u;
    h ^= khi * 0x85EBCA77u;
    h ^= h >> 15;
    h *= 0x2C1B3C6Du;
    h ^= h >> 13;
    return h;
}

// 12-bit -> every third bit
MULLS_HD uint64_t spread12(uint32_t v) {
    uint64_t x = v & 0xfffu;
    x = (x | (x << 16)) & 0x0000ff0000ffull;
    x = (x | (x << 8)) & 0x00f00f00f00full;
    x = (x | (x << 4)) & 0x0c30c30c30c3ull;
    x = (x | (x << 2)) & 0x249249249249ull;
    return x;
}
MULLS_HD uint64_t morton36(uint32_t x, uint32_t y, uint32_t z) { return spread12(x) | (spread12(y) << 1) | (spread12(z) << 2); }

// every third bit of a 36-bit Morton code -> 12-bit coordinate
MULLS_HD uint32_t compact12(uint64_t m) {
    uint64_t x = m & 0x249249249249ull;
    x = (x | (x >> 2)) & 0x0c30c30c30c3ull;
    x = (x | (x >> 4)) & 0x00f00f00f00full;
    x = (x | (x >> 8)) & 0x0000ff0000ffull;
    x = (x | (x >> 16)) & 0x00000000ffffull;
    return (uint32_t)x & 0xfffu;
}

} // namespace mulls
