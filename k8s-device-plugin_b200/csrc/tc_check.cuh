// tc_check.cuh — sm_100a tensor-core health check: every SM runs bit-exact tcgen05 GEMM tiles against host hashes.
//
// The HBM probe (hbm_probe.cuh) streams bytes and never touches a tensor core; a part with a bad tensor core or SM
// datapath returns wrong products without an ECC error or an Xid.  This kernel runs on one CTA per SM (dynamic shared
// memory above half of the SM's 227 KB, so two CTAs cannot share an SM) and checks what the tensor cores compute:
//
//   1. warp 0 allocates 256 TMEM columns (two fp32 accumulators of N = 128) and gives up the allocation permit;
//   2. one thread bulk-copies the operand pool (3 A + 3 B tiles, K-major, canonical UMMA layout packed by the host at
//      open, tc_math.hpp) and the [9][128] table of expected row hashes from HBM into shared memory, once per launch;
//   3. warp 0 lane 0 issues tile t as one M=128 N=128 K=128 chain of tcgen05.mma.cta_group::1 (the first MMA with
//      enable_input_d = 0) into accumulator t & 1 and commits it to full[t & 1]; tile t uses combination
//      (smid + check + t) mod 9, so every SM meets every (A_i, B_j) within 9 checks;
//   4. warps 1-4 (one accumulator row per thread) tcgen05.ld tile t while tile t+1 is being issued, release the
//      accumulator (empty[t & 1]), fold the row's 128 fp32 bit patterns into an order-independent 64-bit hash and
//      compare it with the host's hash for (combination, row);
//   5. per-SM counters (tiles, bad rows, first bad tile/row, CTAs) go to the device control block; the last CTA of the
//      launch that publishes copies them into pinned, device-mapped host memory, fences at system scope and then
//      writes the sequence number -- completion needs no driver call (as ProbeOut in hbm_probe.cuh).
//
// Exactness (tc_math.hpp): integer operands in [-7, 7], |partial sums| < 2^13, so fp32 results are exact in any order.
// Fault hook (data only): the CTA on SM `fault_sm` XORs `fault_mask` into row 0, column 0 of its first tile after
// tcgen05.ld -- a simulated wrong product for testing attribution; the GPU itself is never made to fault.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "hbm_probe.cuh"  // globaltimer_ns, smem_u32, mbarrier and bulk-copy helpers
#include "tc_math.hpp"

namespace b2dp {

constexpr int kTcThreads = 160;        // warp 0: TMEM allocation + MMA issue; warps 1-4: verification
constexpr uint32_t kTcTmemCols = 256;  // two fp32 accumulators, N = 128 columns each
constexpr int kTcMaxSm = 256;          // %smid range the records cover
// dynamic shared memory of both kinds: the bf16 pool + hashes + barriers; the e4m3 launch asks for the same so that it
// too runs one CTA per SM
constexpr size_t kTcSmem = tc::pool_bytes(2) + 64;
static_assert(kTcSmem > 232448 / 2 && kTcSmem <= 232448, "one CTA per SM: more than half of 227 KB, at most all of it");

struct TcSmRec {
    unsigned int tiles;      // tiles verified on this SM
    unsigned int bad_rows;   // rows whose hash did not match
    unsigned int first_bad;  // (tile << 8) | row of the first bad row, ~0u if none
    unsigned int ctas;       // CTAs that ran on this SM
};
// Device-resident control block (one per GPU).  The publishing CTA resets it for the next check.
struct TcCtl {
    TcSmRec rec[2][kTcMaxSm];  // [kind][smid]
    unsigned long long t_start_ns;
    unsigned int done[2];      // CTA completion tickets per kind
};
// Result block: pinned, device-mapped host memory.
struct TcOut {
    TcSmRec rec[2][kTcMaxSm];
    unsigned long long t_start_ns, t_end_ns;
    unsigned int nsmid, pad;
    unsigned long long seq;    // written last
};

struct TcParams {
    const uint8_t* pool;           // this kind's pool (tc::pack_pool)
    unsigned long long desc_base;  // smem descriptor without the start address (tc::smem_desc_base)
    uint32_t idesc;                // instruction descriptor (tc::instr_desc)
    uint32_t tiles;                // tiles per CTA
    uint32_t check;                // check number: the combination schedule's offset
    int fixed_comb;                // >= 0: every tile uses this combination (single-tile parity hook)
    int fault_sm;                  // -1: no injected fault
    uint32_t fault_mask;
    float* c_out;                  // single-tile hook: the raw accumulator [128][128] of tile 0, else nullptr
    TcCtl* ctl;
    TcOut* out;
    unsigned long long seq;
    int publish;                   // the last CTA of this launch publishes both kinds' records and `seq`
};

// ---- tcgen05 wrappers --------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int KIND>
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (KIND == 0)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                     :: "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    else
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                     "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
                     :: "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 :: "r"(smem_u32(bar)) : "memory");
}
// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ uint32_t tc_mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
    return x;
}

// KIND 0: kind::f16 with bf16 operands; KIND 1: kind::f8f6f4 with e4m3 operands.  fp32 accumulators for both.
template <int KIND>
__global__ void __launch_bounds__(kTcThreads, 1) tc_check(TcParams p) {
    constexpr int ES = KIND == 0 ? 2 : 1;
    constexpr uint32_t TILE = tc::tile_bytes(ES);
    constexpr uint32_t OPS = 2u * tc::kSets * TILE;
    constexpr int KSTEPS = tc::kK * ES / 32;  // one MMA consumes 32 bytes of K
    extern __shared__ __align__(1024) uint8_t smem[];
    const uint64_t* hashes = reinterpret_cast<const uint64_t*>(smem + OPS);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OPS + tc::kHashBytes);  // [0] pool, [1,2] full, [3,4] empty
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
    __shared__ unsigned int s_ticket;

    const unsigned long long t0 = globaltimer_ns();
    uint32_t smid, nsmid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    asm volatile("mov.u32 %0, %%nsmid;" : "=r"(nsmid));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1); mbar_init(&bars[2], 1);
        mbar_init(&bars[3], 128); mbar_init(&bars[4], 128);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async_smem();
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(tmem_slot)), "r"(kTcTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (threadIdx.x == 0) {
        mbar_expect_tx(&bars[0], OPS + tc::kHashBytes);
        for (int s = 0; s < 2 * tc::kSets; ++s) bulk_g2s(smem + (size_t)s * TILE, p.pool + (size_t)s * TILE, TILE, &bars[0]);
        bulk_g2s(smem + OPS, p.pool + OPS, tc::kHashBytes, &bars[0]);
    }
    mbar_wait(&bars[0], 0);

    auto comb_of = [&](uint32_t t) -> int {
        return p.fixed_comb >= 0 ? p.fixed_comb : (int)((smid + p.check + t) % (uint32_t)tc::kComb);
    };
    unsigned int bad = 0, first = ~0u;
    if (warp == 0) {
        if (lane == 0) {
            const uint32_t base = smem_u32(smem);
            for (uint32_t t = 0; t < p.tiles; ++t) {
                const uint32_t buf = t & 1;
                if (t >= 2) mbar_wait(&bars[3 + buf], ((t >> 1) - 1) & 1);  // verifiers have read tile t-2
                tc_fence_after();
                const int c = comb_of(t);
                const uint32_t a_addr = base + (uint32_t)(c / tc::kSets) * TILE;
                const uint32_t b_addr = base + (uint32_t)(tc::kSets + c % tc::kSets) * TILE;
#pragma unroll
                for (int k = 0; k < KSTEPS; ++k) {
                    const uint64_t ad = p.desc_base | (uint64_t)(((a_addr + k * 2 * tc::kLbo) >> 4) & 0x3FFF);
                    const uint64_t bd = p.desc_base | (uint64_t)(((b_addr + k * 2 * tc::kLbo) >> 4) & 0x3FFF);
                    tc_mma<KIND>(tmem + buf * (uint32_t)tc::kN, ad, bd, p.idesc, k > 0 ? 1u : 0u);
                }
                tc_commit(&bars[1 + buf]);
            }
        }
        __syncwarp();
    } else {
        const uint32_t quarter = (uint32_t)(warp & 3);  // a warp reads TMEM lanes 32 * (warp id % 4) ..
        const uint32_t row = quarter * 32 + (uint32_t)lane;
        const uint32_t lane_addr = tmem + ((quarter * 32) << 16);
        for (uint32_t t = 0; t < p.tiles; ++t) {
            const uint32_t buf = t & 1;
            mbar_wait(&bars[1 + buf], (t >> 1) & 1);
            tc_fence_after();
            uint64_t h = 0;
#pragma unroll
            for (int ch = 0; ch < tc::kN / 32; ++ch) {
                uint32_t v[32];
                tc_ld32(lane_addr + buf * (uint32_t)tc::kN + ch * 32, v);
                if (ch == tc::kN / 32 - 1) {  // the accumulator is in registers: MMA may overwrite it
                    tc_fence_before();
                    mbar_arrive(&bars[3 + buf]);
                }
                if (ch == 0 && t == 0 && row == 0 && (int)smid == p.fault_sm) v[0] ^= p.fault_mask;
                if (p.c_out && t == 0) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) p.c_out[row * tc::kN + ch * 32 + j] = __uint_as_float(v[j]);
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const uint32_t col = (uint32_t)(ch * 32 + j);
                    h += ((uint64_t)tc_mix32(v[j] ^ (col * tc::kGold)) << 32) |
                         tc_mix32(v[j] ^ (col * tc::kSalt2) ^ tc::kSalt3);
                }
            }
            if (h != hashes[comb_of(t) * tc::kM + row]) {
                ++bad;
                if (first == ~0u) first = (t << 8) | row;
            }
        }
        bad = __reduce_add_sync(0xffffffffu, bad);
        first = __reduce_min_sync(0xffffffffu, first);
        if (lane == 0 && bad) {
            atomicAdd(&p.ctl->rec[KIND][smid & (kTcMaxSm - 1)].bad_rows, bad);
            atomicMin(&p.ctl->rec[KIND][smid & (kTcMaxSm - 1)].first_bad, first);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(kTcTmemCols) : "memory");
    }
    if (threadIdx.x == 0) {
        atomicAdd(&p.ctl->rec[KIND][smid & (kTcMaxSm - 1)].tiles, p.tiles);
        atomicAdd(&p.ctl->rec[KIND][smid & (kTcMaxSm - 1)].ctas, 1u);
        atomicMin(&p.ctl->t_start_ns, t0);
        __threadfence();
        s_ticket = atomicAdd(&p.ctl->done[KIND], 1u);
    }
    __syncthreads();
    if (!p.publish || s_ticket != gridDim.x - 1) return;
    // the last CTA of the publishing launch: every CTA of both kinds has added its counters (the other kind's launch
    // finished earlier on the same stream)
    __threadfence();
    volatile TcSmRec* src = &p.ctl->rec[0][0];
    TcSmRec* dst = &p.out->rec[0][0];
    for (int i = threadIdx.x; i < 2 * kTcMaxSm; i += kTcThreads) {
        TcSmRec r;
        r.tiles = src[i].tiles; r.bad_rows = src[i].bad_rows; r.first_bad = src[i].first_bad; r.ctas = src[i].ctas;
        dst[i] = r;
        src[i].tiles = 0; src[i].bad_rows = 0; src[i].first_bad = ~0u; src[i].ctas = 0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long ts = atomicMin(&p.ctl->t_start_ns, ~0ull);
        p.ctl->t_start_ns = ~0ull;
        p.ctl->done[0] = 0; p.ctl->done[1] = 0;
        __threadfence();
        p.out->t_start_ns = ts;
        p.out->t_end_ns = globaltimer_ns();
        p.out->nsmid = nsmid;
        __threadfence_system();
        *((volatile unsigned long long*)&p.out->seq) = p.seq;
    }
}

}  // namespace b2dp
