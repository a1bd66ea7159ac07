// tc_math.hpp -- host side of the tensor-core health check (tc_check.cuh): operand generation, the exact product,
// the row hash, and the packing of the operand pool into the canonical UMMA shared-memory layout.
//
// The C++ restatement of oracle/tc_check.py (the specification; tests/golden/tc_check_vectors.json pins it).  As with
// pattern_math.hpp, the expected values are computed here, on the host: the device under test is never asked for its
// own reference.
//
// Exactness: operands are integers in [-7, 7] (exact in bf16 and e4m3), so every partial sum of a K = 128 chain is an
// integer with |x| <= 128 * 49 = 6272 < 2^13 -- exact in fp32 in any summation order, and in any accumulator at least
// 14 bits wide.  A mismatch is a fault, never rounding.  Keep K * 49 < 2^13 if K or the value range changes.
#pragma once
#include <cstdint>
#include <cstring>
#include <vector>

#if defined(__CUDACC__)
#define B2DP_TC_HD __host__ __device__
#else
#define B2DP_TC_HD
#endif

namespace b2dp {
namespace tc {

constexpr int kM = 128, kN = 128, kK = 128;   // one tile: M x N accumulator, K-long chain
constexpr int kSets = 3;                      // A tiles and B tiles in the pool
constexpr int kComb = kSets * kSets;          // (A_i, B_j) combinations
constexpr int kVmax = 7;
constexpr uint32_t kGold = 0x9E3779B9u, kSalt2 = 0x7F4A7C15u, kSalt3 = 0x5BD1E995u;
static_assert(kK * kVmax * kVmax < (1 << 13), "partial sums must stay exact (see the header comment)");

inline uint32_t mix32(uint32_t x) {  // murmur3 fmix32: a bijection of 32-bit words
    x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
    return x;
}
// The row-hash term of column j; the row hash is the sum of the terms mod 2^64 (order-independent).
inline uint64_t hash_term(uint32_t bits, uint32_t j) {
    return ((uint64_t)mix32(bits ^ (j * kGold)) << 32) | mix32(bits ^ (j * kSalt2) ^ kSalt3);
}

inline uint32_t seed_for(int index) { return 0x7C5E0000u | (uint32_t)(index & 0xffff); }

// value of operand set `set_id` (A: 0..2, B: 3..5) at (row, k)
inline int operand(uint32_t seed, int set_id, int row, int k) {
    const uint32_t idx = (uint32_t)((set_id * kM + row) * kK + k);
    return (int)(mix32((idx * kGold) ^ seed) % (2 * kVmax + 1)) - kVmax;
}

inline uint16_t enc_bf16(int v) {  // exact for |v| < 256
    const float f = (float)v;
    uint32_t u;
    memcpy(&u, &f, 4);
    return (uint16_t)(u >> 16);
}
inline uint8_t enc_e4m3(int v) {  // exact for |v| <= 7 (bias 7, 3 mantissa bits)
    if (v == 0) return 0;
    const int x = v < 0 ? -v : v;
    int e = 0;
    while ((x >> (e + 1)) != 0) ++e;
    const uint8_t code = (uint8_t)(((e + 7) << 3) | (((x << 3) >> e) & 7));
    return v < 0 ? (uint8_t)(code | 0x80) : code;
}

// Exact C = A_a . B_b^T as fp32 bit patterns, row-major [128][128].
inline void exact_c_bits(uint32_t seed, int a_set, int b_set, uint32_t* c) {
    std::vector<int> a((size_t)kM * kK), b((size_t)kN * kK);
    for (int r = 0; r < kM; ++r)
        for (int k = 0; k < kK; ++k) { a[(size_t)r * kK + k] = operand(seed, a_set, r, k); b[(size_t)r * kK + k] = operand(seed, kSets + b_set, r, k); }
    for (int m = 0; m < kM; ++m)
        for (int n = 0; n < kN; ++n) {
            int s = 0;
            for (int k = 0; k < kK; ++k) s += a[(size_t)m * kK + k] * b[(size_t)n * kK + k];
            const float f = (float)s;
            memcpy(&c[(size_t)m * kN + n], &f, 4);
        }
}

// The 128 row hashes of combination (a_set, b_set).  Both kinds accumulate the same integers exactly, so the kind does
// not change them.
inline void row_hashes(uint32_t seed, int a_set, int b_set, uint64_t* out /*[128]*/) {
    std::vector<uint32_t> c((size_t)kM * kN);
    exact_c_bits(seed, a_set, b_set, c.data());
    for (int m = 0; m < kM; ++m) {
        uint64_t h = 0;
        for (int n = 0; n < kN; ++n) h += hash_term(c[(size_t)m * kN + n], (uint32_t)n);
        out[m] = h;
    }
}

// ---- canonical UMMA layout: K-major, no swizzle ------------------------------------------------------------------
// A "core matrix" is 8 rows x 16 bytes, stored as 128 contiguous bytes.  Core matrices adjacent in K are kLbo bytes
// apart (leading byte offset), 8-row groups are sbo(es) bytes apart (stride byte offset):
//     byte(row, kb) = (row / 8) * SBO + (kb / 16) * LBO + (row % 8) * 16 + kb % 16        kb = k * element size
// One MMA consumes 32 bytes of K (16 bf16 or 32 e4m3) = two core matrices, so step s starts 2 * LBO * s bytes in.
constexpr uint32_t kLbo = 128;
B2DP_TC_HD inline constexpr uint32_t sbo(int es) { return (uint32_t)(kK * es / 16) * 128u; }
B2DP_TC_HD inline constexpr uint32_t tile_bytes(int es) { return (uint32_t)(kM * kK * es); }
constexpr uint32_t kHashBytes = (uint32_t)kComb * kM * 8;
B2DP_TC_HD inline constexpr uint32_t pool_bytes(int es) { return 2u * kSets * tile_bytes(es) + kHashBytes; }
inline size_t umma_offset(int row, int kb, int es) {
    return (size_t)(row / 8) * sbo(es) + (size_t)(kb / 16) * kLbo + (size_t)(row % 8) * 16 + (size_t)(kb % 16);
}

// Shared-memory matrix descriptor without its start address (bits 0-13, added per operand on the device):
// LBO >> 4 at bits 16-29, SBO >> 4 at bits 32-45, version 1 at bits 46-47 (sm_100), base offset 0, layout 0 = no swizzle.
inline uint64_t smem_desc_base(int es) {
    return ((uint64_t)(kLbo >> 4) << 16) | ((uint64_t)(sbo(es) >> 4) << 32) | (1ull << 46);
}
// Instruction descriptor of tcgen05.mma kind::f16 (bf16) / kind::f8f6f4 (e4m3): fp32 D (bit 4), A/B format (bits 7-9,
// 10-12: bf16 = 1 under kind::f16, e4m3 = 0 under kind::f8f6f4), both K-major, N >> 3 at bits 17-22, M >> 4 at 24-28.
inline uint32_t instr_desc(int kind) {
    const uint32_t fmt = kind == 0 ? 1u : 0u;
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(kN >> 3) << 17) | ((uint32_t)(kM >> 4) << 24);
}

// The pool one launch of `kind` (0 bf16, 1 e4m3) loads into shared memory: A_0..A_2, B_0..B_2 in the UMMA layout, then
// the [kComb][128] row-hash table (combination a_set * kSets + b_set).
inline std::vector<uint8_t> pack_pool(uint32_t seed, int kind, const uint64_t* table /*[kComb*128]*/) {
    const int es = kind == 0 ? 2 : 1;
    std::vector<uint8_t> out(pool_bytes(es), 0);
    for (int s = 0; s < 2 * kSets; ++s) {
        uint8_t* t = out.data() + (size_t)s * tile_bytes(es);
        for (int r = 0; r < kM; ++r)
            for (int k = 0; k < kK; ++k) {
                const int v = operand(seed, s, r, k);
                if (es == 2) { const uint16_t e = enc_bf16(v); memcpy(t + umma_offset(r, 2 * k, es), &e, 2); }
                else t[umma_offset(r, k, es)] = enc_e4m3(v);
            }
    }
    memcpy(out.data() + 2u * kSets * tile_bytes(es), table, kHashBytes);
    return out;
}

inline std::vector<uint64_t> hash_table(uint32_t seed) {
    std::vector<uint64_t> t((size_t)kComb * kM);
    for (int c = 0; c < kComb; ++c) row_hashes(seed, c / kSets, c % kSets, t.data() + (size_t)c * kM);
    return t;
}

}  // namespace tc
}  // namespace b2dp
