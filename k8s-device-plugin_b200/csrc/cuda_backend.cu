// cuda_backend.cu -- the `cuda:` backend: real B200s.
//
// One worker thread per GPU owns that GPU's primary context, stream, events, pinned result
// block and the two probe buffers; callers (cgo threads, ctypes, gRPC handlers) never touch
// a CUDA "current device".  The heartbeat probe enqueues one pass on every GPU's stream before
// waiting on any (so the N kernels run concurrently), either from the calling thread with event
// polling (default, lowest latency) or through the per-GPU workers (B2DP_PROBE_VIA_WORKERS); a
// device that does not finish before the deadline yields B2DP_E_TIMEOUT / Unhealthy for that
// device only and is collected later by its worker.
//
// Replaces: the node-level text check `simpleHealthCheck` (plugin.go:161-206), the exporter
// round trip `getGPUHealth` (exporter/health.go:42-82) and the kfd link `type` read
// (allocator/device.go:143-149).  Enumeration replaces GetAMDGPUs (amdgpu.go:149-268) with
// CUDA/NVML/sysfs queries; the record layout and id formats are the reference's.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <pthread.h>
#include <sched.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <deque>
#include <functional>
#include <thread>

#include "gosem.hpp"
#include "hbm_probe.cuh"
#include "internal.hpp"
#include "nvml_dyn.hpp"
#include "pattern_math.hpp"
#include "tc_check.cuh"
#include "units_backend.hpp"

namespace b2dp {

// ---- kernel shapes chosen from profiles/r01_sweep1_kernel_variants.csv --------------------
constexpr int kTmaCW = 4;           // verifier warps
constexpr int kTmaTileVec = 1024;   // 16 KiB tiles
constexpr int kTmaStages = 3;
constexpr int kTmaCtasPerSm = 2;    // 2 x 3 x 16 KiB = 96 KiB staged per SM
constexpr size_t kTmaSmem = (size_t)kTmaStages * kTmaTileVec * 16 + 2 * kTmaStages * 8;
constexpr int kRegThreads = 512, kRegUnroll = 2, kRegCtasPerSm = 2;
constexpr unsigned long long kFloorMinBytes = 128ull << 20;  // a ring slot above the 126 MB L2: the pass measures HBM, not the cache

// bit b of (uint32(i) * K) summed over i < n_words, for the closed-form checksum
__global__ void pattern_bit_counts(unsigned long long n_words, unsigned long long* counts /*[32]*/) {
    unsigned int c[32];  // per-thread iterations stay far below 2^32 for any buffer that fits in HBM
#pragma unroll
    for (int b = 0; b < 32; ++b) c[b] = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += stride) {
        const uint32_t m = (uint32_t)i * kPatternMul;
#pragma unroll
        for (int b = 0; b < 32; ++b) c[b] += (m >> b) & 1u;
    }
#pragma unroll
    for (int b = 0; b < 32; ++b) {
        unsigned long long v = c[b];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&counts[b], v);
    }
}

struct Completion {
    std::mutex mu;
    std::condition_variable cv;
    bool done = false;
    void signal() { { std::lock_guard<std::mutex> g(mu); done = true; } cv.notify_all(); }
    bool wait_until(std::chrono::steady_clock::time_point tp) {
        std::unique_lock<std::mutex> l(mu);
        return cv.wait_until(l, tp, [&] { return done; });
    }
    void wait() { std::unique_lock<std::mutex> l(mu); cv.wait(l, [&] { return done; }); }
};

struct Gpu {
    int ordinal = 0;
    Device dev;                 // the enumerate record
    std::string name, pci_device_id, vbios, family;
    std::string uuid;                     // "GPU-xxxxxxxx-xxxx-xxxx-xxxx-xxxxxxxxxxxx" (cudaDeviceProp.uuid == nvmlDeviceGetUUID)
    int nvml_index = -1;                  // nvmlDeviceGetIndex: what a bare integer in NVIDIA_VISIBLE_DEVICES / a CDI name means
    std::string inforom_image, inforom_oem, inforom_ecc, inforom_power, gsp_fw;
    int64_t vram = 0, sms = 0;
    bool mig_capable = false;
    float gbs_cal = 0.f;                  // best of the calibration passes at open (this device)
    int slow_streak = 0;                  // consecutive passes below the floor (slow_passes= debounce)
    // prearm=1: the NEXT pass is enqueued in advance behind a stream wait on a host-mapped doorbell; a heartbeat then
    // only stores to the doorbell (no launch on the critical path -- after seconds of idle a launch costs ~35 us)
    bool armed = false;
    unsigned long long armed_seq = 0;
    uint32_t armed_seed = 0;
    volatile unsigned int* bell_h = nullptr;
    unsigned long long bell_d = 0;
    cudaEvent_t done_ev = nullptr;        // recorded between pass k and the armed pass k+1: "pass k finished"
    std::atomic<float> gbs_ref{0.f};      // the ceiling the GB/s floor is a fraction of (peer group max, ref_gbs=, or b2dp_probe_set_ref)
    std::array<unsigned long long, 32> bc{};  // host closed-form bit counts for n_vec*4 words (pattern_math.hpp)
    void* nvh = nullptr;                  // NVML device handle (optional)
    unsigned long long ecc_base = 0;      // uncorrected volatile ECC count when the context was opened
    bool have_ecc = false;
    bool xid_registered = false;
    std::atomic<unsigned long long> xid_fault{0};  // first critical Xid seen on this device (sticky, like a real fault)
    int last_healthy = 1;
    // worker
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::deque<std::function<void()>> q;
    bool quit = false;
    // state owned by the worker thread
    std::vector<uint4*> buf;            // ring of cfg.slots buffers: pass k reads buf[cur], writes buf[next()]
    unsigned long long n_vec = 0;       // 16-byte vectors per slot on THIS GPU (cfg.bytes / 16 unless HBM was short at open)
    bool small_ring = false;            // slots had to be smaller than requested: passes carry no GB/s floor
    bool broken = false;                // per-GPU setup failed at open: listed, never probed, always Unhealthy
    std::string broken_reason;
    ProbeCtl* ctl = nullptr;
    ProbeOut *out_h = nullptr, *out_d = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    uint32_t seed = 0;
    int cur = 0;
    int next() const { return (cur + 1) % (int)buf.size(); }
    unsigned long long seq = 0;
    std::atomic<bool> inflight{false};  // a timed-out pass is still owned by the worker
    std::vector<char> peer_enabled;
    int seed_idx = 0;                   // the index the per-device seeds derive from
    // tensor-core check (tc_check.cuh); set up at open with compute=1, else on first use
    bool tc_ready = false;
    uint32_t tc_seed = 0;
    uint8_t* tc_pool[2] = {nullptr, nullptr};  // per kind: operand tiles (UMMA layout) + row-hash table
    TcCtl* tc_ctl = nullptr;
    TcOut *tc_out_h = nullptr, *tc_out_d = nullptr;
    float* tc_c = nullptr;              // b2dp_compute_tile's accumulator
    cudaEvent_t tc_e0 = nullptr, tc_e1 = nullptr;
    unsigned long long tc_seq = 0;
    uint32_t tc_check_no = 0;           // advances the combination schedule
    int tc_fault_sm = -1;               // b2dp_compute_inject_fault: one-shot
    uint32_t tc_fault_mask = 0;
};

// launchers=2: a second launcher thread enqueues the passes of the GPUs on the OTHER NUMA node while the caller
// enqueues its own half, so the last GPU starts ~half as late.  The helper spins for `spin_us` after a fan-out (and after
// cuda_prearm(), which the library's own ListAndWatch loop calls just before a tick is due) and sleeps on a condition
// variable otherwise; woken from sleep it still does the right thing, only later.
struct ProbeJobResult;
struct Launcher {
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::atomic<unsigned long long> cmd{0}, done{0};
    std::atomic<bool> sleeping{false}, quit{false}, arm{false};
    std::vector<size_t> idx;  // gpu indices this thread launches on
    // the job (written by the caller before cmd is bumped, read by the helper after it sees the new cmd)
    std::vector<std::shared_ptr<ProbeJobResult>>* res = nullptr;
    std::vector<char>* state = nullptr;
    uint32_t variant = 0;
};

class CudaBackend {
public:
    CudaConfig cfg;
    std::vector<std::unique_ptr<Gpu>> gpus;  // sorted by dev.id
    Nvml nvml;
    std::string driver_version, driver_src_version;
    std::mutex probe_mu;  // one fan-out at a time
    std::mutex bc_mu;
    std::unique_ptr<UnitsBackend> units;             // probe=helpers / probe=off / MIG: the NVML-driven half (units_backend.hpp)
    std::vector<std::unique_ptr<std::atomic<unsigned long long>>> unit_xid;  // xid=1 in units mode: one sticky latch per unit
    void* libcuda = nullptr;                         // prearm=1: cuStreamWaitValue32 from the driver API (cudart is linked statically)
    int (*wait32)(void* stream, unsigned long long addr, unsigned value, unsigned flags) = nullptr;
    std::unique_ptr<Launcher> launcher;              // launchers=2
    std::vector<size_t> caller_idx;                  // the GPUs the calling thread enqueues (all of them without a launcher)
    cpu_set_t caller_cpus;                           // pin=1: CPUs local to the caller's GPUs
    bool have_caller_cpus = false;
    void* xid_set = nullptr;                         // NVML event set (xid=1), waited on by xid_thread only
    std::thread xid_thread;
    std::atomic<bool> xid_quit{false};
    std::mutex xid_cb_mu;
    std::function<void()> on_health_event;           // e.g. "run a heartbeat now on every ListAndWatch stream"
    void fire_health_event() {
        std::function<void()> fn;
        { std::lock_guard<std::mutex> l(xid_cb_mu); fn = on_health_event; }
        if (fn) fn();
    }
    std::map<unsigned long long, std::array<unsigned long long, 32>> bitcounts;
};

static std::string cuda_err(const char* what, cudaError_t e) {
    return std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
}

static void worker_loop(Gpu* g) {
    cudaSetDevice(g->ordinal);
    for (;;) {
        std::function<void()> fn;
        {
            std::unique_lock<std::mutex> l(g->mu);
            g->cv.wait(l, [&] { return g->quit || !g->q.empty(); });
            if (g->q.empty()) return;  // quit
            fn = std::move(g->q.front());
            g->q.pop_front();
        }
        fn();
    }
}

// Run fn on g's worker; returns the completion to wait on.
static std::shared_ptr<Completion> post(Gpu* g, std::function<void()> fn) {
    auto c = std::make_shared<Completion>();
    {
        std::lock_guard<std::mutex> l(g->mu);
        g->q.push_back([fn = std::move(fn), c] { fn(); c->signal(); });
    }
    g->cv.notify_one();
    return c;
}
template <class F>
static void run_sync(Gpu* g, F&& fn) { post(g, std::forward<F>(fn))->wait(); }

// Closed-form checksum of a clean buffer: computed on the HOST (pattern_math.hpp) -- a health probe must not ask the
// device under test for its own reference value.  Cached per size; the per-GPU ring size is cached in Gpu::bc.
static const std::array<unsigned long long, 32>& host_bitcounts(CudaBackend* be, unsigned long long n_words) {
    std::lock_guard<std::mutex> l(be->bc_mu);
    auto it = be->bitcounts.find(n_words);
    if (it == be->bitcounts.end()) it = be->bitcounts.emplace(n_words, pattern_bit_counts_host(n_words)).first;
    return it->second;  // std::map nodes are stable
}

static std::string read_trim(const std::string& p) {
    std::string d;
    if (!go::read_file(p, d)) return "";
    return go::trim_space(d);
}

// ---- the probe fan-out -----------------------------------------------------------------------
struct ProbeJobResult {
    cudaError_t ce = cudaSuccess;
    ProbeOut out{};
    float ms = 0;
    uint32_t seed = 0;
    unsigned long long seq = 0;
    bool seq_ok = false;
    unsigned long long n_vec = 0;   // vectors this pass covers (shrunk on a busy GPU)
    bool advance = true;            // false: verify-only prefix pass, buffers/seed stay as they are
    bool timed = false;             // bracket the kernel with CUDA events (B2DP_PROBE_EVENT_TIMING)
    int grid = 0;                   // CTAs to launch (0 = the tuned shape); diagnostic hook, see b2dp_probe_opts.grid_ctas
};

static void launch_probe(Gpu* g, unsigned long long n_vec, uint32_t variant, uint32_t seed, uint32_t delta,
                         const uint4* src, uint4* dst, unsigned long long seq, int grid = 0) {
    if (variant == B2DP_PROBE_VARIANT_R128)
        hbm_probe_r128<kRegThreads, kRegUnroll><<<grid > 0 ? grid : (int)g->sms * kRegCtasPerSm, kRegThreads, 0, g->stream>>>(
            src, dst, n_vec, seed, delta, g->ctl, g->out_d, seq);
    else
        hbm_probe_tma<kTmaCW, kTmaTileVec, kTmaStages>
            <<<grid > 0 ? grid : (int)g->sms * kTmaCtasPerSm, (kTmaCW + 1) * 32, kTmaSmem, g->stream>>>(
                src, dst, n_vec, seed, delta, g->ctl, g->out_d, seq);
}

// Enqueue one pass on g's stream (caller must have made g's device current).
static void probe_issue(Gpu* g, ProbeJobResult* r, uint32_t variant) {
    const uint32_t seed = g->seed, next = seed * 1664525u + 1013904223u;
    const unsigned long long n_vec = r->n_vec ? r->n_vec : g->n_vec;
    r->n_vec = n_vec;
    r->seed = seed;
    r->seq = ++g->seq;
    if (r->timed) cudaEventRecord(g->e0, g->stream);
    launch_probe(g, n_vec, variant, seed, r->advance ? seed ^ next : 0u, g->buf[g->cur], g->buf[g->next()], r->seq, r->grid);
    r->ce = cudaGetLastError();
    if (r->timed) cudaEventRecord(g->e1, g->stream);
}

// ---- prearm=1 ---------------------------------------------------------------------------------------------------------
// While pass k runs, pass k+1 is enqueued behind `cuStreamWaitValue32(doorbell == seq)`: a stream wait occupies no SM.
// The next heartbeat rings the doorbell (one host store per GPU) instead of launching: measured on B200
// (tools/doorbell_probe.cu, profiles/r02_doorbell_vs_launch.csv) start-of-work latency is 6 vs 8 us back to back and
// 13 vs 34 us after 2 s of idle -- the production shape, a heartbeat every few seconds.  An armed pass that is not
// wanted (fault repair, peek/poke/reset, P2P, a pass with other options, close) is FLUSHED: rung, waited for, its
// result ignored, the ring state not advanced -- it read and re-keyed exactly what the next ordinary pass will.
// Off by default: a pending stream wait stalls every OTHER piece of work this process submits to the same GPU (other
// streams, a second context -- measured; other processes keep their latency), so it belongs in a process whose only GPU
// user is this library.
static inline void probe_ring(Gpu* g, unsigned long long seq) { __atomic_store_n(g->bell_h, (unsigned int)seq, __ATOMIC_RELEASE); }

static void probe_arm(CudaBackend* be, Gpu* g) {  // g's device is current; pass k has just been enqueued on g->stream
    if (!be->wait32 || g->armed) return;
    const uint32_t seed = g->seed * 1664525u + 1013904223u, next = seed * 1664525u + 1013904223u;  // the state AFTER pass k
    const int M = (int)g->buf.size(), src = (g->cur + 1) % M, dst = (g->cur + 2) % M;
    cudaEventRecord(g->done_ev, g->stream);
    const unsigned long long seq = g->seq + 1;
    if (be->wait32((void*)g->stream, g->bell_d, (unsigned int)seq, 1u /*CU_STREAM_WAIT_VALUE_EQ*/) != 0) return;
    g->seq = seq;
    launch_probe(g, g->n_vec, 0u, seed, seed ^ next, g->buf[src], g->buf[dst], seq);
    if (cudaGetLastError() != cudaSuccess) { probe_ring(g, seq); return; }  // release the wait; nothing follows it
    g->armed = true;
    g->armed_seq = seq;
    g->armed_seed = seed;
}

static void probe_flush(Gpu* g) {  // discard the armed pass (see above); needs no current device
    if (!g->armed) return;
    probe_ring(g, g->armed_seq);
    cudaStreamSynchronize(g->stream);
    g->armed = false;
}

// The last CTA publishes the result block and, after a system-scope fence, the launch's sequence
// number into pinned host memory (hbm_probe.cuh finish()): seeing the number means every CTA's
// stores and the whole block are done -- completion without a driver call.
static inline bool probe_published(const Gpu* g, const ProbeJobResult* r) {
    return *(volatile const unsigned long long*)&g->out_h->seq == r->seq;
}

// After the pass completed: read the published result, advance the seed / ping-pong state.
static void probe_collect(Gpu* g, ProbeJobResult* r) {
    const unsigned long long n_vec = g->n_vec;  // repairs re-fill the whole slot
    cudaError_t e = r->ce;
    if (e == cudaSuccess && r->timed) {
        e = cudaEventSynchronize(g->e1);  // the result is already published; the event follows within ~1 us
        if (e == cudaSuccess) e = cudaEventElapsedTime(&r->ms, g->e0, g->e1);
    }
    r->ce = e;
    if (e != cudaSuccess) return;
    std::atomic_thread_fence(std::memory_order_acquire);       // the sequence number was read first (probe_published)
    memcpy(&r->out, (const void*)g->out_h, sizeof(ProbeOut));  // the block is complete once its sequence number shows
    r->seq_ok = r->out.seq == r->seq;
    if (!r->advance) {
        if (r->out.mismatches != 0 || !r->seq_ok) {  // repair the source buffer in place
            cudaSetDevice(g->ordinal);
            probe_flush(g);
            hbm_fill<256><<<(int)g->sms * 8, 256, 0, g->stream>>>(g->buf[g->cur], n_vec, g->seed);
            cudaStreamSynchronize(g->stream);
        }
        return;
    }
    g->seed = g->seed * 1664525u + 1013904223u;
    g->cur = g->next();
    if (r->out.mismatches != 0 || !r->seq_ok) {
        // report once, then start the next pass from a clean pattern: a transient flip is
        // reported exactly once, a stuck cell shows up again on the next pass
        cudaSetDevice(g->ordinal);
        probe_flush(g);  // the armed pass would read the buffer about to be repaired: discard it first
        hbm_fill<256><<<(int)g->sms * 8, 256, 0, g->stream>>>(g->buf[g->cur], n_vec, g->seed);
        cudaStreamSynchronize(g->stream);
    }
}

// ---- tensor-core check (tc_check.cuh) ---------------------------------------------------------------------------------
// Runs on g's worker: the operand pools and the expected row hashes are computed on the HOST (tc_math.hpp) and copied
// once; the device under test never computes its own reference.
static cudaError_t tc_setup(Gpu* g) {
    if (g->tc_ready) return cudaSuccess;
    cudaError_t e;
    g->tc_seed = tc::seed_for(g->seed_idx);
    const std::vector<uint64_t> table = tc::hash_table(g->tc_seed);
    for (int kind = 0; kind < 2; ++kind) {
        const std::vector<uint8_t> pool = tc::pack_pool(g->tc_seed, kind, table.data());
        if ((e = cudaMalloc(&g->tc_pool[kind], pool.size())) != cudaSuccess) return e;
        if ((e = cudaMemcpy(g->tc_pool[kind], pool.data(), pool.size(), cudaMemcpyHostToDevice)) != cudaSuccess) return e;
    }
    auto ctl = std::make_unique<TcCtl>();
    memset(ctl.get(), 0, sizeof(TcCtl));
    for (auto& kind : ctl->rec) for (auto& r : kind) r.first_bad = ~0u;
    ctl->t_start_ns = ~0ull;
    if ((e = cudaMalloc(&g->tc_ctl, sizeof(TcCtl))) != cudaSuccess) return e;
    if ((e = cudaMemcpy(g->tc_ctl, ctl.get(), sizeof(TcCtl), cudaMemcpyHostToDevice)) != cudaSuccess) return e;
    if ((e = cudaHostAlloc(&g->tc_out_h, sizeof(TcOut), cudaHostAllocMapped)) != cudaSuccess) return e;
    memset(g->tc_out_h, 0, sizeof(TcOut));
    if ((e = cudaHostGetDevicePointer(&g->tc_out_d, g->tc_out_h, 0)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&g->tc_c, sizeof(float) * tc::kM * tc::kN)) != cudaSuccess) return e;
    if ((e = cudaEventCreate(&g->tc_e0)) != cudaSuccess) return e;
    if ((e = cudaEventCreate(&g->tc_e1)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(tc_check<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmem)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(tc_check<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmem)) != cudaSuccess) return e;
    g->tc_ready = true;
    return cudaSuccess;
}

static void tc_free(Gpu* g) {
    for (uint8_t*& p : g->tc_pool) { if (p) cudaFree(p); p = nullptr; }
    if (g->tc_ctl) cudaFree(g->tc_ctl);
    if (g->tc_out_h) cudaFreeHost(g->tc_out_h);
    if (g->tc_c) cudaFree(g->tc_c);
    if (g->tc_e0) cudaEventDestroy(g->tc_e0);
    if (g->tc_e1) cudaEventDestroy(g->tc_e1);
    g->tc_ctl = nullptr; g->tc_out_h = nullptr; g->tc_c = nullptr; g->tc_e0 = g->tc_e1 = nullptr;
    g->tc_ready = false;
}

struct TcJob {
    cudaError_t ce = cudaSuccess;
    unsigned long long seq = 0;
    uint32_t tiles = 0;
    bool timed = false;
    float ms = 0;
};

static TcParams tc_params(Gpu* g, int kind, uint32_t tiles) {
    TcParams p{};
    p.pool = g->tc_pool[kind];
    p.desc_base = tc::smem_desc_base(kind == 0 ? 2 : 1);
    p.idesc = tc::instr_desc(kind);
    p.tiles = tiles;
    p.check = g->tc_check_no;
    p.fixed_comb = -1;
    p.fault_sm = -1;
    p.ctl = g->tc_ctl;
    p.out = g->tc_out_d;
    return p;
}

// Enqueue one check (bf16 then e4m3, one CTA per SM each) on g's stream; g's device is current.  The e4m3 launch
// publishes both kinds' records and the sequence number.
static void tc_issue(Gpu* g, TcJob* r) {
    r->seq = ++g->tc_seq;
    TcParams p = tc_params(g, 0, r->tiles);
    p.seq = r->seq;
    p.fault_sm = g->tc_fault_sm;
    p.fault_mask = g->tc_fault_mask;
    g->tc_fault_sm = -1;
    g->tc_fault_mask = 0;
    if (r->timed) cudaEventRecord(g->tc_e0, g->stream);
    tc_check<0><<<(int)g->sms, kTcThreads, kTcSmem, g->stream>>>(p);
    p = tc_params(g, 1, r->tiles);
    p.seq = r->seq;
    p.publish = 1;
    tc_check<1><<<(int)g->sms, kTcThreads, kTcSmem, g->stream>>>(p);
    r->ce = cudaGetLastError();
    if (r->timed) cudaEventRecord(g->tc_e1, g->stream);
    ++g->tc_check_no;
}

static inline bool tc_published(const Gpu* g, const TcJob* r) {
    return *(volatile const unsigned long long*)&g->tc_out_h->seq == r->seq;
}

// Fold the published block into the ABI result.
static void tc_result(Gpu* g, TcJob* r, b2dp_compute_result& o) {
    o.seed = g->tc_seed;
    o.sms = (int32_t)g->sms;
    o.first_bad_sm = o.first_bad_kind = o.first_bad_tile = o.first_bad_row = -1;
    cudaError_t e = r->ce;
    if (e == cudaSuccess && r->timed) {
        e = cudaEventSynchronize(g->tc_e1);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&r->ms, g->tc_e0, g->tc_e1);
    }
    if (e != cudaSuccess) { o.err = B2DP_E_CUDA; o.healthy = 0; return; }
    std::atomic_thread_fence(std::memory_order_acquire);
    TcOut out;
    memcpy(&out, (const void*)g->tc_out_h, sizeof out);
    if (out.seq != r->seq) { o.err = B2DP_E_CUDA; o.healthy = 0; return; }
    for (int s = 0; s < kTcMaxSm; ++s) {
        const TcSmRec& a = out.rec[0][s];
        const TcSmRec& b = out.rec[1][s];
        o.tiles += (uint64_t)a.tiles + b.tiles;
        o.bad_rows += (uint64_t)a.bad_rows + b.bad_rows;
        if (a.ctas && b.ctas) { o.covered_mask[s / 32] |= 1u << (s % 32); ++o.sms_covered; }
        if (a.bad_rows || b.bad_rows) {
            o.bad_sm_mask[s / 32] |= 1u << (s % 32);
            if (o.sms_failed++ == 0) {
                const int k = a.bad_rows ? 0 : 1;
                const unsigned fb = out.rec[k][s].first_bad;
                o.first_bad_sm = s; o.first_bad_kind = k; o.first_bad_tile = (int32_t)(fb >> 8); o.first_bad_row = (int32_t)(fb & 0xff);
            }
        }
    }
    o.ms_device = (float)((double)(out.t_end_ns - out.t_start_ns) * 1e-6);
    o.ms_event = r->timed ? r->ms : 0.f;
    const float ms = r->timed ? r->ms : o.ms_device;
    o.tflops = ms > 0 ? (float)((double)tc::kM * tc::kN * tc::kK * 2.0 * (double)o.tiles / ((double)ms * 1e-3) * 1e-12) : 0.f;
    o.healthy = o.bad_rows == 0 ? 1 : 0;
}

static void tc_log(const Gpu* g, const b2dp_compute_result& o) {
    if (o.err == B2DP_E_TIMEOUT) logf(2, "%s: tensor-core check missed its deadline", g->dev.id.c_str());
    else if (o.err != B2DP_OK) logf(2, "%s: tensor-core check failed to run or publish", g->dev.id.c_str());
    else if (!o.healthy)
        logf(2, "%s: tensor-core check failed on SM %d (%s, tile %d, row %d), %llu rows bad", g->dev.id.c_str(), o.first_bad_sm,
             o.first_bad_kind == 0 ? "bf16" : "e4m3", o.first_bad_tile, o.first_bad_row, (unsigned long long)o.bad_rows);
    if (o.err == B2DP_OK && o.sms_covered < o.sms)
        logf(1, "%s: tensor-core check covered %d of %d SMs (the others ran no CTA; not a verdict)", g->dev.id.c_str(), o.sms_covered, o.sms);
}

// Launch the check on every GPU in `idx` (all before waiting on any), then poll the pinned result blocks until
// `deadline`.  A device that misses it is B2DP_E_TIMEOUT; its worker collects the launches later (inflight).
// The caller holds probe_mu; out has one entry per GPU of the backend.
static void tc_fanout(CudaBackend* be, const std::vector<size_t>& idx, uint32_t tiles, bool timed,
                      std::chrono::steady_clock::time_point deadline, std::vector<b2dp_compute_result>& out) {
    int prev_dev = -1;
    cudaGetDevice(&prev_dev);
    std::vector<std::shared_ptr<TcJob>> jobs(be->gpus.size());
    std::vector<size_t> pending;
    for (size_t i : idx) {
        Gpu* g = be->gpus[i].get();
        b2dp_compute_result& o = out[i];
        cudaSetDevice(g->ordinal);
        cudaError_t e = tc_setup(g);
        if (e != cudaSuccess) { o.err = B2DP_E_CUDA; o.healthy = 0; logf(2, "%s: tensor-core check setup: %s", g->dev.id.c_str(), cudaGetErrorName(e)); continue; }
        jobs[i] = std::make_shared<TcJob>();
        jobs[i]->tiles = tiles;
        jobs[i]->timed = timed;
        tc_issue(g, jobs[i].get());
        pending.push_back(i);
    }
    unsigned spins = 0;
    while (!pending.empty()) {
        for (size_t k = 0; k < pending.size();) {
            const size_t i = pending[k];
            Gpu* g = be->gpus[i].get();
            TcJob* r = jobs[i].get();
            if (r->ce == cudaSuccess && !tc_published(g, r)) {
                if ((spins & 0x3ff) != 0x3ff) { ++k; continue; }
                const cudaError_t q = cudaStreamQuery(g->stream);  // a kernel that faulted never publishes
                if (q == cudaErrorNotReady) { ++k; continue; }
                if (q != cudaSuccess) r->ce = q;
            }
            if (r->timed || r->ce != cudaSuccess) cudaSetDevice(g->ordinal);
            tc_result(g, r, out[i]);
            pending[k] = pending.back();
            pending.pop_back();
        }
        if (!pending.empty() && (++spins & 0x3ff) == 0 && std::chrono::steady_clock::now() > deadline) break;
    }
    for (size_t i : pending) {
        Gpu* g = be->gpus[i].get();
        out[i].err = B2DP_E_TIMEOUT;
        out[i].healthy = 0;
        g->inflight.store(true);
        post(g, [g] { cudaStreamSynchronize(g->stream); g->inflight.store(false); });
    }
    if (prev_dev >= 0) cudaSetDevice(prev_dev);
}

// "0-31,64-95" -> cpu_set_t
static bool parse_cpulist(const std::string& text, cpu_set_t* set) {
    CPU_ZERO(set);
    bool any = false;
    size_t pos = 0;
    while (pos < text.size()) {
        size_t e = text.find(',', pos);
        if (e == std::string::npos) e = text.size();
        const std::string item = text.substr(pos, e - pos);
        pos = e + 1;
        if (item.empty()) continue;
        const size_t dash = item.find('-');
        const int lo = atoi(item.c_str()), hi = dash == std::string::npos ? lo : atoi(item.c_str() + dash + 1);
        for (int c = lo; c <= hi && c < CPU_SETSIZE; ++c) { if (c >= 0) { CPU_SET(c, set); any = true; } }
    }
    return any;
}

static void launcher_loop(CudaBackend* be, Launcher* L, int spin_us) {
    unsigned long long seen = 0;
    auto spin_until = std::chrono::steady_clock::now();
    for (;;) {
        // wait for the next command: spin inside the window, sleep outside it
        for (;;) {
            if (L->quit.load(std::memory_order_acquire)) return;
            if (L->cmd.load(std::memory_order_acquire) != seen) break;
            if (L->arm.exchange(false)) spin_until = std::chrono::steady_clock::now() + std::chrono::microseconds(4 * spin_us);
            if (std::chrono::steady_clock::now() < spin_until) {
#if defined(__x86_64__)
                __builtin_ia32_pause();
#endif
                continue;
            }
            std::unique_lock<std::mutex> l(L->mu);
            L->sleeping.store(true);
            L->cv.wait(l, [&] { return L->quit.load() || L->arm.load() || L->cmd.load() != seen; });
            L->sleeping.store(false);
        }
        seen = L->cmd.load(std::memory_order_acquire);
        for (size_t i : L->idx) {
            Gpu* g = be->gpus[i].get();
            if ((*L->state)[i] != 0) continue;
            if (g->inflight.load()) { (*L->state)[i] = 2; continue; }
            cudaSetDevice(g->ordinal);
            probe_issue(g, (*L->res)[i].get(), L->variant);
        }
        L->done.store(seen, std::memory_order_release);
        spin_until = std::chrono::steady_clock::now() + std::chrono::microseconds(spin_us);
    }
}

// The library's ListAndWatch loop calls this shortly before a tick is due: the helper launcher leaves its condition
// variable and spins, so the fan-out that follows finds it hot.
void cuda_prearm(CudaBackend* be) {
    Launcher* L = be->launcher.get();
    if (!L) return;
    L->arm.store(true);
    if (L->sleeping.load()) { std::lock_guard<std::mutex> l(L->mu); L->cv.notify_one(); }
}

static void xid_listener(CudaBackend* be);

int cuda_backend_open(const CudaConfig& cfg, CudaBackend** out, std::string& err) {
    auto be = std::make_unique<CudaBackend>();
    be->cfg = cfg;
    be->nvml.load();
    // MIG: CUDA shows a process ONE compute instance (and then no other GPU), so a node with any MIG-enabled GPU is
    // enumerated through NVML and probed by one helper process per unit; this process never creates a CUDA context.
    int mode = cfg.probe_mode;
    if (mode == 0 && cfg.mig_auto && be->nvml.ok && be->nvml.device_count && be->nvml.handle_by_index && be->nvml.mig_mode) {
        unsigned cnt = 0;
        if (be->nvml.device_count(&cnt) == 0)
            for (unsigned i = 0; i < cnt; ++i) {
                void* h = nullptr;
                unsigned cur = 0, pend = 0;
                if (be->nvml.handle_by_index(i, &h) == 0 && be->nvml.mig_mode(h, &cur, &pend) == 0 && cur == 1) mode = 1;
            }
    }
    if (mode != 0) {
        int rc = units_open(cfg, be->nvml, mode == 1, &be->units, err);
        if (rc != B2DP_OK) return rc;
        {
            int n_mig = 0;
            for (auto& u : be->units->units) n_mig += u.mig_slot >= 0;
            logf(0, "NVML enumeration: %zu unit(s), %d MIG instance(s), probe=%s%s", be->units->units.size(), n_mig, mode == 1 ? "helpers" : "off",
                 cfg.probe_mode == 0 ? " (forced by MIG: CUDA shows a process one compute instance)" : "");
        }
        if (be->nvml.driver_version) {
            char buf[96] = {0};
            if (be->nvml.driver_version(buf, sizeof buf) == 0) be->driver_version = buf;
        }
        if (be->driver_version.empty()) be->driver_version = read_trim(go::join(cfg.sysroot, "sys/module/nvidia/version"));
        be->driver_src_version = read_trim(go::join(cfg.sysroot, "sys/module/nvidia/srcversion"));
        for (size_t i = 0; i < be->units->units.size(); ++i) be->unit_xid.push_back(std::make_unique<std::atomic<unsigned long long>>(0));
        // xid=1 needs no CUDA: NVML delivers critical Xid events to this process for the physical GPUs the units live on
        if (cfg.check_xid && be->nvml.event_set_create && be->nvml.register_events && be->nvml.event_wait &&
            be->nvml.event_set_create(&be->xid_set) == 0) {
            std::vector<void*> seen;
            for (auto& u : be->units->units)
                if (u.nvh && std::find(seen.begin(), seen.end(), u.nvh) == seen.end()) {
                    seen.push_back(u.nvh);
                    be->nvml.register_events(u.nvh, 0x8ull /*nvmlEventTypeXidCriticalError*/, be->xid_set);
                }
            be->xid_thread = std::thread(xid_listener, be.get());
        }
        *out = be.release();
        return B2DP_OK;
    }
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count == 0) {
        err = ce != cudaSuccess ? cuda_err("cudaGetDeviceCount", ce) : "no CUDA devices";
        return B2DP_E_NOGPU;
    }
    std::vector<int> ords = cfg.devices;
    if (ords.empty()) for (int i = 0; i < count; ++i) ords.push_back(i);
    for (int o : ords) if (o < 0 || o >= count) { err = "device ordinal out of range"; return B2DP_E_INVAL; }
    for (size_t a = 0; a < ords.size(); ++a)
        for (size_t b = a + 1; b < ords.size(); ++b)
            if (ords[a] == ords[b]) { err = "device ordinal listed twice"; return B2DP_E_INVAL; }

    if (be->nvml.ok && be->nvml.driver_version) {
        char buf[96] = {0};
        if (be->nvml.driver_version(buf, sizeof buf) == 0) be->driver_version = buf;
    }
    if (be->driver_version.empty()) be->driver_version = read_trim("/sys/module/nvidia/version");
    be->driver_src_version = read_trim("/sys/module/nvidia/srcversion");

    // CPU topology nodes precede GPU nodes in a kfd tree; count NUMA nodes (>= 1)
    int n_cpu = 0;
    for (auto& p : go::glob_prefixed(go::join(cfg.sysroot, "sys/devices/system/node"), "node"))
        if (p.size() > 4 && go::is_digit(p.back())) ++n_cpu;
    if (n_cpu < 1) n_cpu = 1;

    for (int o : ords) {
        auto g = std::make_unique<Gpu>();
        g->ordinal = o;
        cudaDeviceProp prop;
        if ((ce = cudaGetDeviceProperties(&prop, o)) != cudaSuccess) { err = cuda_err("cudaGetDeviceProperties", ce); return B2DP_E_CUDA; }
        char bdf[32];
        snprintf(bdf, sizeof bdf, "%04x:%02x:%02x.0", prop.pciDomainID, prop.pciBusID, prop.pciDeviceID);
        g->dev.id = bdf;  // same shape as the reference's PCI dir names (amdgpu.go:154-155)
        char devid[32];
        snprintf(devid, sizeof devid, "%04x:%02x:%02x:0", prop.pciDomainID, prop.pciBusID, prop.pciDeviceID);  // amdgpu.go:141
        g->dev.dev_id = devid;
        g->name = prop.name;
        {
            const unsigned char* u = reinterpret_cast<const unsigned char*>(prop.uuid.bytes);
            char ub[48];
            snprintf(ub, sizeof ub, "GPU-%02x%02x%02x%02x-%02x%02x-%02x%02x-%02x%02x-%02x%02x%02x%02x%02x%02x", u[0], u[1], u[2],
                     u[3], u[4], u[5], u[6], u[7], u[8], u[9], u[10], u[11], u[12], u[13], u[14], u[15]);
            g->uuid = ub;
        }
        g->vram = (int64_t)prop.totalGlobalMem;
        g->sms = prop.multiProcessorCount;
        g->family = prop.major == 10 || prop.major == 12 ? "Blackwell" : prop.major == 9 ? "Hopper"
                    : prop.major == 8 ? (prop.minor == 9 ? "Ada" : "Ampere") : "sm_" + std::to_string(prop.major * 10 + prop.minor);
        const std::string pci_dir = go::join(cfg.sysroot, std::string("sys/bus/pci/devices/") + bdf);
        g->pci_device_id = read_trim(pci_dir + "/device");
        if (g->pci_device_id.empty()) g->pci_device_id = "0x0000";
        std::string numa = read_trim(pci_dir + "/numa_node");
        int64_t nv = 0;
        g->dev.numa = (!numa.empty() && go::atoi(numa, &nv) == go::NumErr::none) ? (int)nv : 0;
        // /dev/nvidia<minor>
        g->dev.card = o;
        bool have_minor = false;
        if (be->nvml.ok && be->nvml.handle_by_bus_id && be->nvml.minor_number) {
            void* h = nullptr;
            char busid[32];
            snprintf(busid, sizeof busid, "%08x:%02x:%02x.0", prop.pciDomainID, prop.pciBusID, prop.pciDeviceID);
            if (be->nvml.handle_by_bus_id(busid, &h) == 0) {
                g->nvh = h;
                if (be->nvml.ecc_total && be->nvml.ecc_total(h, 1 /*UNCORRECTED*/, 0 /*VOLATILE*/, &g->ecc_base) == 0)
                    g->have_ecc = true;
                unsigned mn = 0;
                if (be->nvml.minor_number(h, &mn) == 0) { g->dev.card = (int)mn; have_minor = true; }
                char vb[96] = {0};
                if (be->nvml.vbios && be->nvml.vbios(h, vb, sizeof vb) == 0) g->vbios = vb;
                unsigned ni = 0;
                if (be->nvml.index_of && be->nvml.index_of(h, &ni) == 0) g->nvml_index = (int)ni;
                if (be->nvml.uuid_of && be->nvml.uuid_of(h, vb, sizeof vb) == 0 && vb[0]) g->uuid = vb;
                // firmware label sources (the analogue of libdrm's per-block firmware versions, amdgpu.go:392-437)
                if (be->nvml.inforom_image && be->nvml.inforom_image(h, vb, sizeof vb) == 0) g->inforom_image = vb;
                if (be->nvml.inforom_object) {
                    if (be->nvml.inforom_object(h, 0, vb, sizeof vb) == 0) g->inforom_oem = vb;
                    if (be->nvml.inforom_object(h, 1, vb, sizeof vb) == 0) g->inforom_ecc = vb;
                    if (be->nvml.inforom_object(h, 2, vb, sizeof vb) == 0) g->inforom_power = vb;
                }
                if (be->nvml.gsp_firmware && be->nvml.gsp_firmware(h, vb) == 0) g->gsp_fw = vb;  // NVML_GSP_FIRMWARE_VERSION_BUF_SIZE = 64
                unsigned cur = 0, pend = 0;
                if (be->nvml.mig_mode && be->nvml.mig_mode(h, &cur, &pend) == 0) g->mig_capable = true;
            }
        }
        if (!have_minor) {
            std::string info;
            if (go::read_file(std::string("/proc/driver/nvidia/gpus/") + bdf + "/information", info)) {
                size_t p = info.find("Device Minor:");
                if (p != std::string::npos) g->dev.card = atoi(info.c_str() + p + 13);
            }
        }
        be->gpus.push_back(std::move(g));
    }
    std::sort(be->gpus.begin(), be->gpus.end(), [](const auto& a, const auto& b) { return a->dev.id < b->dev.id; });
    for (size_t i = 0; i < be->gpus.size(); ++i) {
        be->gpus[i]->dev.render_d = 128 + (int)i;
        be->gpus[i]->dev.node_id = n_cpu + (int)i;
        be->gpus[i]->peer_enabled.assign(be->gpus.size(), 0);
    }

    // xid=1: one NVML event set for the node, every GPU registered for critical Xid events
    if (cfg.check_xid && be->nvml.ok && be->nvml.event_set_create && be->nvml.register_events && be->nvml.event_wait &&
        be->nvml.event_set_create(&be->xid_set) == 0) {
        for (auto& gp : be->gpus)
            if (gp->nvh && be->nvml.register_events(gp->nvh, 0x8ull /*nvmlEventTypeXidCriticalError*/, be->xid_set) == 0)
                gp->xid_registered = true;
        be->xid_thread = std::thread(xid_listener, be.get());
    }

    // start workers and allocate per-GPU state on them
    for (auto& gp : be->gpus) gp->th = std::thread(worker_loop, gp.get());
    std::vector<std::shared_ptr<Completion>> cs;
    std::vector<cudaError_t> errs(be->gpus.size(), cudaSuccess);
    std::vector<const char*> where(be->gpus.size(), "");
    for (size_t i = 0; i < be->gpus.size(); ++i) {
        Gpu* g = be->gpus[i].get();
        const unsigned long long bytes = cfg.bytes, n_vec = cfg.bytes / 16;
        const int idx = (int)i;
        const int calib = cfg.calib;
        const int seed_idx = cfg.seed_index >= 0 ? cfg.seed_index + idx : idx;  // a helper's one device stands for unit seed_index
        g->buf.assign((size_t)cfg.slots, nullptr);
        (void)n_vec;
        const bool compute = cfg.compute;
        cs.push_back(post(g, [g, bytes, idx, calib, seed_idx, compute, &errs, &where] {
            cudaError_t e;
#define TRY(x) if ((e = (x)) != cudaSuccess) { errs[idx] = e; where[idx] = #x; return; }
            TRY(cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
            TRY(cudaEventCreate(&g->e0));
            TRY(cudaEventCreate(&g->e1));
            // HBM may be short when the daemon restarts under running pods: rather than fail (and take the node's
            // GPUs away from the kubelet) halve the slot size until the ring fits, down to 1 MiB
            unsigned long long slot = bytes;
            for (;;) {
                e = cudaSuccess;
                for (auto& b : g->buf) if ((e = cudaMalloc(&b, slot)) != cudaSuccess) break;
                if (e == cudaSuccess) break;
                cudaGetLastError();
                for (auto& b : g->buf) { if (b) cudaFree(b); b = nullptr; }
                if (e != cudaErrorMemoryAllocation || slot <= (1ull << 20)) { errs[idx] = e; where[idx] = "cudaMalloc(probe ring)"; return; }
                slot = (slot / 2) & ~15ull;
            }
            g->n_vec = slot / 16;
            g->small_ring = slot < bytes;
            TRY(cudaMalloc(&g->ctl, sizeof(ProbeCtl)));
            ProbeCtl init{};
            init.first_bad = ~0ull; init.t_start_ns = ~0ull;
            TRY(cudaMemcpy(g->ctl, &init, sizeof init, cudaMemcpyHostToDevice));
            TRY(cudaHostAlloc(&g->out_h, sizeof(ProbeOut), cudaHostAllocMapped));
            memset(g->out_h, 0, sizeof(ProbeOut));
            TRY(cudaHostGetDevicePointer(&g->out_d, g->out_h, 0));
            {   // doorbell for prearm=1 (allocated always: 64 bytes)
                void* bell = nullptr;
                void* bell_dev = nullptr;
                TRY(cudaHostAlloc(&bell, 64, cudaHostAllocMapped));
                memset(bell, 0, 64);
                TRY(cudaHostGetDevicePointer(&bell_dev, bell, 0));
                g->bell_h = static_cast<volatile unsigned int*>(bell);
                g->bell_d = (unsigned long long)(uintptr_t)bell_dev;
                TRY(cudaEventCreateWithFlags(&g->done_ev, cudaEventDisableTiming));
            }
            TRY(cudaFuncSetAttribute(hbm_probe_tma<kTmaCW, kTmaTileVec, kTmaStages>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTmaSmem));
            TRY(cudaFuncSetAttribute(hbm_probe_tma<kTmaCW, kTmaTileVec, kTmaStages>,
                                     cudaFuncAttributePreferredSharedMemoryCarveout, 100));
            g->seed = 0x5EED0000u | (uint32_t)(seed_idx & 0xffff);  // SURVEY 8(d) config 2
            g->seed_idx = seed_idx;
            if (compute) { if ((e = tc_setup(g)) != cudaSuccess) { errs[idx] = e; where[idx] = "tensor-core check setup"; return; } }
            g->cur = 0;
            hbm_fill<256><<<(int)g->sms * 8, 256, 0, g->stream>>>(g->buf[0], g->n_vec, g->seed);
            TRY(cudaGetLastError());
            TRY(cudaStreamSynchronize(g->stream));
            // Integer self-test of THIS GPU against the host: the pattern's bit counts, computed by the SMs, must equal
            // the host's closed form (which is what every later verdict is judged against).
            g->bc = pattern_bit_counts_host(g->n_vec * 4);
            {
                unsigned long long* d = nullptr;
                std::array<unsigned long long, 32> dev_counts{};
                TRY(cudaMalloc(&d, sizeof dev_counts));
                TRY(cudaMemsetAsync(d, 0, sizeof dev_counts, g->stream));
                pattern_bit_counts<<<(int)g->sms * 4, 256, 0, g->stream>>>(g->n_vec * 4, d);
                TRY(cudaGetLastError());
                TRY(cudaMemcpyAsync(dev_counts.data(), d, sizeof dev_counts, cudaMemcpyDeviceToHost, g->stream));
                TRY(cudaStreamSynchronize(g->stream));
                cudaFree(d);
                if (dev_counts != g->bc) { errs[idx] = cudaErrorUnknown; where[idx] = "integer self-test (pattern bit counts != host closed form)"; return; }
            }
            // Calibration: best of `calib` warm, non-advancing passes (read slot 0, write slot 1 un-re-keyed; seed and
            // ring position stay where they are) = what this device streams when healthy and idle.
            for (int k = 0; k < (calib > 0 ? calib + 1 : 0); ++k) {
                ProbeJobResult r;
                r.advance = false;
                r.timed = true;
                probe_issue(g, &r, 0u);
                if (r.ce == cudaSuccess) r.ce = cudaStreamSynchronize(g->stream);
                probe_collect(g, &r);
                TRY(r.ce);
                // the verdict's clock is the in-kernel span (first CTA start .. result published): it is there on every
                // pass, event-timed or not
                const double span_ms = (double)(r.out.t_end_ns - r.out.t_start_ns) * 1e-6;
                if (k == 0 || span_ms <= 0) continue;  // first pass warms clocks, TLBs and the instruction cache
                const float gbs = (float)(2.0 * (double)g->n_vec * 16.0 / span_ms * 1e-6);
                if (gbs > g->gbs_cal) g->gbs_cal = gbs;
            }
#undef TRY
        }));
    }
    for (auto& c : cs) c->wait();
    // One GPU that cannot be set up (fallen off the bus, exclusive-process mode held by a tenant, no memory at
    // all) must not take the node's other GPUs away from the kubelet: it stays in the device list and is
    // reported Unhealthy on every heartbeat.  Only a node with no usable GPU fails to open.
    size_t n_broken = 0;
    for (size_t i = 0; i < errs.size(); ++i) {
        const bool forced = std::find(cfg.break_devices.begin(), cfg.break_devices.end(), (int)i) != cfg.break_devices.end();
        if (errs[i] == cudaSuccess && !forced) continue;
        Gpu* g = be->gpus[i].get();
        g->broken = true;
        g->broken_reason = forced ? "setup failure injected (break=)" : cuda_err(where[i], errs[i]);
        g->last_healthy = 0;
        logf(2, "%s could not be set up and will be reported Unhealthy: %s", g->dev.id.c_str(), g->broken_reason.c_str());
        err = g->broken_reason + " on " + g->dev.id;
        ++n_broken;
    }
    if (n_broken == be->gpus.size()) {
        CudaBackend* raw = be.release();
        cuda_backend_close(raw);
        return B2DP_E_CUDA;
    }
    // The ceiling a device's GB/s floor is a fraction of: ref_gbs= if given, else the best calibration of any
    // device of the same product with the same ring size -- a part that is already slow when the daemon starts is
    // judged against its siblings, not against itself.
    for (auto& g : be->gpus) {
        if (g->broken) continue;
        float ref = cfg.ref_gbs;
        if (ref <= 0)
            for (auto& o : be->gpus)
                if (!o->broken && o->name == g->name && o->n_vec == g->n_vec) ref = std::max(ref, o->gbs_cal);
        g->gbs_ref.store(ref);
        logf(0, "%s %s ring %d x %llu MiB%s, calibrated %.0f GB/s, ceiling %.0f GB/s, floor %.0f GB/s", g->dev.id.c_str(), g->name.c_str(),
             (int)g->buf.size(), (unsigned long long)(g->n_vec * 16 >> 20), g->small_ring ? " (shrunk: HBM was short)" : "", g->gbs_cal, ref,
             cfg.min_gbs > 0 ? cfg.min_gbs : cfg.min_frac * ref);
    }
    if (cfg.prearm && cfg.compute) logf(1, "prearm=1 is off with compute=1: a check queued behind an armed pass would wait for the next heartbeat");
    if (cfg.prearm && cfg.launchers < 2 && !cfg.compute) {
        be->libcuda = dlopen("libcuda.so.1", RTLD_NOW | RTLD_LOCAL);
        if (be->libcuda) {
            void* f = dlsym(be->libcuda, "cuStreamWaitValue32_v2");
            if (!f) f = dlsym(be->libcuda, "cuStreamWaitValue32");
            be->wait32 = reinterpret_cast<int (*)(void*, unsigned long long, unsigned, unsigned)>(f);
        }
        if (!be->wait32) logf(1, "prearm=1: cuStreamWaitValue32 is not available; passes are launched at each heartbeat");
    }
    // launchers=2: split the GPUs by NUMA node (GPU 0's node stays with the caller; one NUMA node: split in halves)
    for (size_t i = 0; i < be->gpus.size(); ++i) be->caller_idx.push_back(i);
    if (cfg.launchers >= 2 && be->gpus.size() >= 2) {
        auto L = std::make_unique<Launcher>();
        be->caller_idx.clear();
        const int numa0 = be->gpus[0]->dev.numa;
        for (size_t i = 0; i < be->gpus.size(); ++i)
            (be->gpus[i]->dev.numa == numa0 ? be->caller_idx : L->idx).push_back(i);
        if (L->idx.empty()) {
            be->caller_idx.clear();
            for (size_t i = 0; i < be->gpus.size(); ++i) (i < (be->gpus.size() + 1) / 2 ? be->caller_idx : L->idx).push_back(i);
        }
        Launcher* raw = L.get();
        CudaBackend* bp = be.get();
        raw->th = std::thread(launcher_loop, bp, raw, cfg.spin_us);
        cpu_set_t set;  // keep the helper on the CPUs next to its GPUs
        if (parse_cpulist(read_trim(go::join(cfg.sysroot, "sys/bus/pci/devices/" + be->gpus[raw->idx[0]]->dev.id + "/local_cpulist")), &set))
            pthread_setaffinity_np(raw->th.native_handle(), sizeof set, &set);
        be->launcher = std::move(L);
    }
    if (cfg.pin_caller)
        be->have_caller_cpus = parse_cpulist(
            read_trim(go::join(cfg.sysroot, "sys/bus/pci/devices/" + be->gpus[be->caller_idx[0]]->dev.id + "/local_cpulist")), &be->caller_cpus);
    *out = be.release();
    return B2DP_OK;
}

void cuda_backend_close(CudaBackend* be) {
    if (!be) return;
    if (be->units) {
        be->xid_quit = true;
        if (be->xid_thread.joinable()) be->xid_thread.join();
        { std::lock_guard<std::mutex> l(be->xid_cb_mu); be->on_health_event = nullptr; }
        units_close(be->units.get());
        if (be->xid_set && be->nvml.event_set_free) be->nvml.event_set_free(be->xid_set);
        delete be;
        return;
    }
    be->xid_quit = true;
    if (be->xid_thread.joinable()) be->xid_thread.join();
    { std::lock_guard<std::mutex> l(be->xid_cb_mu); be->on_health_event = nullptr; }
    if (be->launcher) {
        be->launcher->quit.store(true);
        { std::lock_guard<std::mutex> l(be->launcher->mu); be->launcher->cv.notify_all(); }
        if (be->launcher->th.joinable()) be->launcher->th.join();
    }
    for (auto& gp : be->gpus) {
        Gpu* g = gp.get();
        if (!g->th.joinable()) continue;
        post(g, [g] {
            probe_flush(g);
            if (g->stream) cudaStreamSynchronize(g->stream);
            if (g->bell_h) cudaFreeHost(const_cast<unsigned int*>(g->bell_h));
            if (g->done_ev) cudaEventDestroy(g->done_ev);
            for (uint4* b : g->buf) if (b) cudaFree(b);
            if (g->ctl) cudaFree(g->ctl);
            if (g->out_h) cudaFreeHost(g->out_h);
            if (g->e0) cudaEventDestroy(g->e0);
            if (g->e1) cudaEventDestroy(g->e1);
            tc_free(g);
            if (g->stream) cudaStreamDestroy(g->stream);
        })->wait();
        { std::lock_guard<std::mutex> l(g->mu); g->quit = true; }
        g->cv.notify_all();
        g->th.join();
    }
    if (be->xid_set && be->nvml.event_set_free) be->nvml.event_set_free(be->xid_set);
    if (be->libcuda) dlclose(be->libcuda);
    delete be;
}

int cuda_device_count(CudaBackend* be) { return be->units ? (int)be->units->units.size() : (int)be->gpus.size(); }
float cuda_min_gbs(CudaBackend* be) { return be->cfg.min_gbs; }
void cuda_set_health_event_callback(CudaBackend* be, std::function<void()> fn) {
    std::lock_guard<std::mutex> l(be->xid_cb_mu);
    be->on_health_event = std::move(fn);
}

int cuda_enumerate(CudaBackend* be, std::vector<Device>& out, std::string&) {
    out.clear();
    if (be->units) { for (auto& u : be->units->units) out.push_back(u.dev); return B2DP_OK; }
    for (auto& g : be->gpus) out.push_back(g->dev);
    return B2DP_OK;
}

int cuda_node_health(CudaBackend* be) {
    // the analogue of "a GPU node exists in the kfd topology" (plugin.go:198-201):
    // the driver still answers and reports the devices this context was opened on
    if (be->units) {  // no CUDA in this process: NVML must still count the physical GPUs the units live on
        unsigned cnt = 0;
        return be->nvml.device_count && be->nvml.device_count(&cnt) == 0 && cnt > 0 && !be->units->units.empty() ? 1 : 0;
    }
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) return 0;
    return count >= (int)be->gpus.size() && !be->gpus.empty() ? 1 : 0;
}

void cuda_label_source(CudaBackend* be, LabelSource& src) {
    src.native = true;
    src.driver_version = be->driver_version;
    src.driver_src_version = be->driver_src_version;
    if (be->units) {
        bool migc = !be->units->units.empty();
        for (auto& u : be->units->units) {
            src.family.push_back(u.family);
            src.product_name.push_back(u.name);
            src.device_id.push_back(u.pci_device_id);
            src.vbios.push_back(u.vbios);
            src.firmware.push_back(u.firmware);
            src.vram_bytes.push_back(u.vram);
            src.sm_count.push_back(u.sms);
            migc = migc && u.mig_capable;
        }
        src.part_supported[0] = src.part_supported[1] = migc;
        return;
    }
    bool mig = !be->gpus.empty();
    for (auto& g : be->gpus) {
        src.family.push_back(g->family);
        src.product_name.push_back(g->name);
        src.device_id.push_back(g->pci_device_id);
        src.vbios.push_back(g->vbios);
        // per-block firmware versions, the key scheme of main.go:116-144 ("<block>.fw.<version>")
        std::vector<std::pair<std::string, std::string>> fw;
        if (!g->vbios.empty()) fw.push_back({"vbios", g->vbios});
        if (!g->inforom_image.empty()) fw.push_back({"inforom-img", g->inforom_image});
        if (!g->inforom_oem.empty()) fw.push_back({"inforom-oem", g->inforom_oem});
        if (!g->inforom_ecc.empty()) fw.push_back({"inforom-ecc", g->inforom_ecc});
        if (!g->inforom_power.empty()) fw.push_back({"inforom-pwr", g->inforom_power});
        if (!g->gsp_fw.empty()) fw.push_back({"gsp", g->gsp_fw});
        src.firmware.push_back(std::move(fw));
        src.vram_bytes.push_back(g->vram);
        src.sm_count.push_back(g->sms);
        mig = mig && g->mig_capable;
    }
    src.part_supported[0] = src.part_supported[1] = mig;
}

// Xids that report an application's own fault (bad kernel, MMU fault of a user context, preemption,
// user-stopped) rather than a broken device -- the list NVIDIA's own device plugin ignores.
static bool xid_is_application_error(unsigned long long xid) {
    switch (xid) { case 13: case 31: case 43: case 45: case 68: case 109: return true; default: return false; }
}

static void latch_xid(Gpu* g, unsigned long long xid) {
    unsigned long long none = 0;
    if (!xid_is_application_error(xid)) g->xid_fault.compare_exchange_strong(none, xid ? xid : 999);
}

// xid=1: the only thread that waits on the NVML event set.  A device-level Xid is latched on its device and
// reported at once (on_health_event), not at the next pulse.
static void xid_listener(CudaBackend* be) {
    Nvml::EventData d{};
    while (!be->xid_quit.load()) {
        const int rc = be->nvml.event_wait(be->xid_set, &d, 200);  // ms; NVML_ERROR_TIMEOUT (10) when idle
        if (rc != 0) {
            if (rc != 10) std::this_thread::sleep_for(std::chrono::milliseconds(200));  // a failing set must not spin
            continue;
        }
        if (d.type != 0x8ull) continue;  // nvmlEventTypeXidCriticalError
        bool hit = false;
        for (auto& g : be->gpus)
            if (g->nvh == d.device && !xid_is_application_error(d.data)) { latch_xid(g.get(), d.data); hit = true; }
        if (be->units && !xid_is_application_error(d.data))
            for (size_t i = 0; i < be->units->units.size(); ++i) {
                const Unit& u = be->units->units[i];
                // a MIG-attributed Xid names its GPU instance; 0xFFFFFFFF = the whole GPU (every instance on it)
                if (u.nvh != d.device || (u.mig_slot >= 0 && d.gi != 0xffffffffu && d.gi != u.gi)) continue;
                unsigned long long none = 0;
                be->unit_xid[i]->compare_exchange_strong(none, d.data ? d.data : 999);
                hit = true;
            }
        if (hit) { logf(2, "critical Xid %llu reported by NVML: device(s) latched Unhealthy", d.data); be->fire_health_event(); }
    }
}

int cuda_probe(CudaBackend* be, const b2dp_probe_opts* opts, std::vector<b2dp_probe_result>& out, std::string& err) {
    std::lock_guard<std::mutex> pl(be->probe_mu);
    if (be->units) {
        if (!be->units->helpers) { err = "probe=off: this context enumerates only"; return B2DP_E_UNSUPPORTED; }
        const int rc = units_probe(be->units.get(), opts, out, err);
        if (rc == B2DP_OK && be->cfg.check_xid)
            for (size_t i = 0; i < out.size() && i < be->unit_xid.size(); ++i)
                if (be->unit_xid[i]->load()) { out[i].flags |= B2DP_RES_XID; out[i].healthy = 0; be->units->units[i].last_healthy = 0; }
        return rc;
    }
    int rc = B2DP_OK;
    const uint32_t variant = opts ? (opts->flags & B2DP_PROBE_VARIANT_MASK) : 0;
    const bool via_workers = opts && (opts->flags & B2DP_PROBE_VIA_WORKERS);
    const bool timed = opts && (opts->flags & B2DP_PROBE_EVENT_TIMING);
    const uint32_t timeout_ms = opts && opts->timeout_ms ? opts->timeout_ms : 5000;  // health.go:37
    // GB/s floor: an absolute one if the call or the context names it (min_gbs), else min_frac (default 0.8,
    // BASELINE.json's ">= 80 % of HBM peak") of the device's calibrated ceiling
    const float abs_floor = opts && opts->min_gbs > 0 ? opts->min_gbs : be->cfg.min_gbs;
    const int grid = opts ? (int)std::min<uint32_t>(opts->grid_ctas, 1u << 16) : 0;  // diagnostic hook, bounded
    const size_t n = be->gpus.size();
    std::vector<std::shared_ptr<ProbeJobResult>> res(n);
    std::vector<std::shared_ptr<Completion>> cs(n);
    std::vector<char> state(n, 0);  // 0 pending, 1 done, 2 timed out / busy
    std::vector<char> rung_any(n, 0);  // prearm=1: this pass was already enqueued and only had its doorbell rung
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(timeout_ms);
    for (size_t i = 0; i < n; ++i) { res[i] = std::make_shared<ProbeJobResult>(); res[i]->timed = timed; res[i]->grid = grid; }
    for (size_t i = 0; i < n; ++i) if (be->gpus[i]->broken) state[i] = 4;  // never launched on
    // busy policy (tenant workloads): a 2 GiB-traffic probe steals bandwidth from a pod that owns the
    // GPU; `busy=skip` keeps the last verdict, `busy=shrink` verifies a small prefix without re-keying
    std::vector<uint32_t> rflags(n, 0);
    if (be->cfg.busy_policy != 0 && be->nvml.ok && be->nvml.running_procs) {
        for (size_t i = 0; i < n; ++i) {
            Gpu* g = be->gpus[i].get();
            if (!g->nvh || state[i] != 0) continue;
            unsigned cnt = 0;
            const int nrc = be->nvml.running_procs(g->nvh, &cnt, nullptr);  // count only (INSUFFICIENT_SIZE = 7)
            if ((nrc != 0 && nrc != 7) || cnt <= 1) continue;              // this process holds one context itself
            if (be->cfg.busy_policy == 1) { state[i] = 3; rflags[i] = B2DP_RES_SKIPPED_BUSY; }
            else {
                unsigned long long sv = be->cfg.shrink_bytes / 16;
                res[i]->n_vec = sv < g->n_vec ? (sv ? sv : 1) : g->n_vec;
                res[i]->advance = false;
                rflags[i] = B2DP_RES_SHRUNK;
            }
        }
    }

    if (via_workers) {
        // fully isolated path: each GPU's own thread launches and waits; a wedged driver call can
        // only ever block that worker
        for (size_t i = 0; i < n; ++i) {  // launch everywhere before waiting anywhere
            Gpu* g = be->gpus[i].get();
            auto r = res[i];
            if (state[i] != 0) continue;
            if (g->inflight.load()) { state[i] = 2; continue; }
            g->inflight.store(true);  // until collected: a pass that misses the deadline still owns seed/ring state
            cs[i] = post(g, [g, r, variant] {
                probe_flush(g);
                probe_issue(g, r.get(), variant);
                if (r->ce == cudaSuccess) r->ce = cudaStreamSynchronize(g->stream);
                probe_collect(g, r.get());
                g->inflight.store(false);
            });
        }
        for (size_t i = 0; i < n; ++i)
            if (state[i] == 0) state[i] = cs[i]->wait_until(deadline) ? 1 : 2;
    } else {
        // low-latency path (default): the calling thread enqueues on every GPU's stream, then polls
        // the completion events; no thread hand-offs on the critical path.  A device that misses
        // the deadline is handed to its worker to be collected whenever it finishes.  The caller's
        // current CUDA device is restored before returning.
        int prev_dev = -1;
        cudaGetDevice(&prev_dev);
        if (be->have_caller_cpus) {  // pin=1: keep the enqueue + poll thread on the CPUs next to its GPUs (once per thread)
            static thread_local const CudaBackend* pinned_for = nullptr;
            if (pinned_for != be) { pthread_setaffinity_np(pthread_self(), sizeof be->caller_cpus, &be->caller_cpus); pinned_for = be; }
        }
        Launcher* L = be->launcher.get();
        unsigned long long cmd = 0;
        if (L) {  // hand the other NUMA node's GPUs to the helper, then enqueue our own
            L->res = &res; L->state = &state; L->variant = variant;
            cmd = L->cmd.fetch_add(1) + 1;  // seq_cst: ordered against the `sleeping` load below (store/load pair on both sides)
            if (L->sleeping.load()) { std::lock_guard<std::mutex> l(L->mu); L->cv.notify_one(); }
        }
        // prearm=1: a pass with the default options may be the one that is already enqueued behind its doorbell
        const bool can_arm = be->wait32 && !be->cfg.compute && variant == B2DP_PROBE_VARIANT_TMA && !timed && grid == 0 && be->cfg.busy_policy == 0;
        std::vector<char> arm_ok(n, 0);  // decided before any pass is issued (issuing fills in r->n_vec)
        for (size_t i = 0; i < n; ++i) arm_ok[i] = can_arm && res[i]->n_vec == 0 && res[i]->advance;
        auto armable = [&](size_t i) { return arm_ok[i] != 0; };
        std::vector<char> rung(n, 0);
        for (size_t i : be->caller_idx) {  // doorbells first: one host store each, every armed GPU starts within microseconds
            Gpu* g = be->gpus[i].get();
            if (state[i] != 0 || !g->armed || !armable(i) || g->inflight.load()) continue;
            ProbeJobResult* r = res[i].get();
            r->n_vec = g->n_vec; r->seed = g->armed_seed; r->seq = g->armed_seq; r->ce = cudaSuccess;
            probe_ring(g, g->armed_seq);
            g->armed = false;
            rung[i] = rung_any[i] = 1;
        }
        for (size_t i : be->caller_idx) {
            Gpu* g = be->gpus[i].get();
            if (state[i] != 0 || rung[i]) continue;
            if (g->inflight.load()) { state[i] = 2; continue; }
            cudaSetDevice(g->ordinal);
            probe_flush(g);  // an armed pass that does not fit this call's options is discarded
            probe_issue(g, res[i].get(), variant);
        }
        if (L) while (L->done.load(std::memory_order_acquire) != cmd) {
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
        // while the passes run: enqueue the NEXT one behind its doorbell (overlapped with ~0.33 ms of GPU work)
        if (can_arm)
            for (size_t i : be->caller_idx) {
                Gpu* g = be->gpus[i].get();
                if (state[i] != 0 || !armable(i) || res[i]->ce != cudaSuccess) continue;
                cudaSetDevice(g->ordinal);
                probe_arm(be, g);
            }
        size_t pending = 0;
        for (size_t i = 0; i < n; ++i) pending += state[i] == 0;
        unsigned spins = 0;
        while (pending) {
            for (size_t i = 0; i < n; ++i) {
                if (state[i] != 0) continue;
                Gpu* g = be->gpus[i].get();
                if (res[i]->ce == cudaSuccess && !probe_published(g, res[i].get())) {
                    // not there yet; now and then ask the driver too, so that a faulted kernel (which
                    // never publishes) is reported at once instead of at the deadline
                    if ((spins & 0x3ff) != 0x3ff) continue;
                    const cudaError_t q = cudaStreamQuery(g->stream);
                    if (q == cudaErrorNotReady) continue;
                    if (q != cudaSuccess) res[i]->ce = q;
                }
                probe_collect(g, res[i].get());  // no driver call unless event-timed or a repair is due
                state[i] = 1;
                --pending;
            }
            if (pending && (++spins & 0x3ff) == 0 && std::chrono::steady_clock::now() > deadline) break;
        }
        for (size_t i = 0; i < n; ++i) {
            if (state[i] != 0) continue;
            state[i] = 2;
            Gpu* g = be->gpus[i].get();
            auto r = res[i];
            g->inflight.store(true);
            post(g, [g, r] {
                // with a pass armed behind this one, "this pass is done" is the event recorded between the two
                if (r->ce == cudaSuccess) r->ce = g->armed ? cudaEventSynchronize(g->done_ev) : cudaStreamSynchronize(g->stream);
                probe_collect(g, r.get());
                probe_flush(g);
                g->inflight.store(false);
            });
        }
        if (prev_dev >= 0) cudaSetDevice(prev_dev);
    }

    out.assign(n, b2dp_probe_result{});
    for (size_t i = 0; i < n; ++i) {
        b2dp_probe_result& o = out[i];
        o.device = (int)i;
        o.bytes = 2ull * be->gpus[i]->n_vec * 16;
        o.first_bad_word = ~0ull;
        o.flags = rflags[i] | (be->gpus[i]->small_ring ? B2DP_RES_SMALL_RING : 0u) | (!via_workers && rung_any[i] ? B2DP_RES_PREARMED : 0u);
        if (state[i] == 2) { o.err = B2DP_E_TIMEOUT; o.healthy = 0; be->gpus[i]->last_healthy = 0; continue; }
        if (state[i] == 3) { o.bytes = 0; o.healthy = be->gpus[i]->last_healthy; continue; }  // skipped: last verdict stands
        if (state[i] == 4) { o.bytes = 0; o.err = B2DP_E_CUDA; o.healthy = 0; err = be->gpus[i]->broken_reason + " on " + be->gpus[i]->dev.id; continue; }
        const ProbeJobResult& r = *res[i];
        o.seed = r.seed;
        if (r.ce != cudaSuccess) {
            o.err = B2DP_E_CUDA; o.healthy = 0;
            be->gpus[i]->last_healthy = 0;
            err = cuda_err("probe", r.ce) + " on " + be->gpus[i]->dev.id;
            continue;
        }
        Gpu* g = be->gpus[i].get();
        o.expected_checksum = expected_checksum_from_counts(
            r.n_vec == g->n_vec ? g->bc : host_bitcounts(be, r.n_vec * 4), r.n_vec * 4, r.seed);  // host closed form
        o.bytes = 2ull * r.n_vec * 16;
        o.checksum = r.out.checksum;
        o.mismatches = r.out.mismatches;
        o.first_bad_word = r.out.first_bad;
        o.ms_event = r.ms;  // 0 unless B2DP_PROBE_EVENT_TIMING
        o.ms_device = (float)((double)(r.out.t_end_ns - r.out.t_start_ns) * 1e-6);
        const float ms_for_rate = r.timed ? r.ms : o.ms_device;
        o.gbs = ms_for_rate > 0 ? (float)((double)o.bytes / (double)ms_for_rate * 1e-6) : 0.f;
        // the verdict's rate: bytes over the in-kernel span, the same clock the ceiling was calibrated with (o.gbs is
        // the event-timed figure when B2DP_PROBE_EVENT_TIMING asks for the roofline's clock)
        const float gbs_span = o.ms_device > 0 ? (float)((double)o.bytes / (double)o.ms_device * 1e-6) : 0.f;
        o.gbs_ref = g->gbs_ref.load();
        o.frac = o.gbs_ref > 0 ? gbs_span / o.gbs_ref : 0.f;
        // verdict (oracle/probe.py probe_healthy).  No GB/s floor for a pass that shares the GPU with a tenant by
        // design (shrunk / small ring); the fractional floor needs a ring that streams from HBM (> the 126 MB L2).
        float floor = 0.f;
        if (!(o.flags & (B2DP_RES_SHRUNK | B2DP_RES_SMALL_RING))) {
            if (abs_floor > 0) floor = abs_floor;
            else if (o.bytes / 2 >= kFloorMinBytes && o.gbs_ref > 0) floor = be->cfg.min_frac * o.gbs_ref;
            else o.flags |= B2DP_RES_NO_FLOOR;
        }
        o.min_gbs_applied = floor;
        bool fast_enough = gbs_span >= floor;
        if (fast_enough) g->slow_streak = 0;
        else {
            o.flags |= B2DP_RES_SLOW;
            // slow_passes=K: only the K-th consecutive slow pass is a verdict (a one-heartbeat dip is flagged, not failed);
            // integrity faults are never debounced
            if (++g->slow_streak < be->cfg.slow_passes) fast_enough = true;
            // Slow path only: a pass that shared HBM bandwidth with another process on the GPU says nothing about the
            // part.  NVML counts the compute processes; this one holds one context itself.
            unsigned cnt = 0;
            if (be->nvml.ok && be->nvml.running_procs && g->nvh) {
                const int nrc = be->nvml.running_procs(g->nvh, &cnt, nullptr);  // count only (INSUFFICIENT_SIZE = 7)
                if ((nrc == 0 || nrc == 7) && cnt > 1) { o.flags |= B2DP_RES_CONTENDED; fast_enough = true; }
            }
        }
        o.healthy = (r.seq_ok && o.mismatches == 0 && o.checksum == o.expected_checksum && fast_enough) ? 1 : 0;
        if (be->cfg.check_ecc && be->gpus[i]->have_ecc) {  // opt-in: an NVML query per device per pass
            unsigned long long now = 0;
            if (be->nvml.ecc_total(be->gpus[i]->nvh, 1, 0, &now) == 0 && now > be->gpus[i]->ecc_base) {
                o.flags |= B2DP_RES_ECC;
                o.healthy = 0;
            }
            // HBM row remapping: a failed remap means the bad row stays in use (the part is due for replacement)
            unsigned corr = 0, unc = 0, pending = 0, failed = 0;
            if (be->nvml.remapped_rows && be->nvml.remapped_rows(be->gpus[i]->nvh, &corr, &unc, &pending, &failed) == 0 && failed) {
                o.flags |= B2DP_RES_ECC;
                o.healthy = 0;
            }
        }
        be->gpus[i]->last_healthy = o.healthy;
    }
    if (be->cfg.compute) {  // compute=1: the tensor-core check on every GPU whose pass ran, under the same deadline
        std::vector<size_t> idx;
        for (size_t i = 0; i < n; ++i) if (state[i] == 1 && !be->gpus[i]->inflight.load()) idx.push_back(i);
        std::vector<b2dp_compute_result> cr(n, b2dp_compute_result{});
        tc_fanout(be, idx, B2DP_COMPUTE_DEFAULT_TILES, false, deadline, cr);
        for (size_t i : idx) {
            if (cr[i].err == B2DP_OK && cr[i].healthy) continue;
            tc_log(be->gpus[i].get(), cr[i]);
            out[i].flags |= B2DP_RES_COMPUTE;
            out[i].healthy = 0;
            be->gpus[i]->last_healthy = 0;
        }
    }
    if (be->cfg.check_xid) {  // opt-in: a critical Xid since open fails the device whatever the pass said
        for (size_t i = 0; i < n; ++i)
            if (be->gpus[i]->xid_fault.load()) {
                out[i].flags |= B2DP_RES_XID;
                out[i].healthy = 0;
                be->gpus[i]->last_healthy = 0;
            }
    }
    return B2DP_OK;
}

static Gpu* gpu_at(CudaBackend* be, int device, std::string& err) {
    if (device < 0 || device >= (int)be->gpus.size()) { err = "device index out of range"; return nullptr; }
    if (be->gpus[device]->broken) { err = "device was not set up: " + be->gpus[device]->broken_reason; return nullptr; }
    return be->gpus[device].get();
}

// helpers mode: forward a single-unit operation to the unit's child
static int units_forward(CudaBackend* be, int device, HelperReq q, std::string& err, std::vector<uint32_t>* payload = nullptr) {
    UnitsBackend* ub = be->units.get();
    if (!ub->helpers) { err = "probe=off: this context enumerates only"; return B2DP_E_UNSUPPORTED; }
    if (device < 0 || device >= (int)ub->units.size()) { err = "device index out of range"; return B2DP_E_INVAL; }
    Unit& u = ub->units[device];
    if (u.broken) { err = "device was not set up: " + u.broken_reason; return B2DP_E_INVAL; }
    HelperRsp r{};
    int rc = units_call(u, q, &r, 30000, payload);
    if (rc == B2DP_OK && r.rc != B2DP_OK) { rc = r.rc; err = r.text; }
    else if (rc != B2DP_OK) {
        // the stream is out of step (a late answer may carry a payload): drop this child, the next heartbeat restarts it
        err = "probe helper did not answer";
        units_kill(u);
        u.broken = true;
        u.broken_reason = "probe helper unresponsive";
    }
    return rc;
}

int cuda_inject_fault(CudaBackend* be, int device, uint64_t word, uint32_t mask, std::string& err) {
    if (be->units && word == ~0ull) {  // synthetic critical Xid, as in the in-process mode below
        if (device < 0 || device >= (int)be->unit_xid.size()) { err = "device index out of range"; return B2DP_E_INVAL; }
        if (be->cfg.check_xid && !xid_is_application_error(mask)) {
            unsigned long long none = 0;
            be->unit_xid[device]->compare_exchange_strong(none, mask ? mask : 999);
            be->fire_health_event();
        }
        return B2DP_OK;
    }
    if (be->units) {
        std::lock_guard<std::mutex> pl(be->probe_mu);
        HelperReq q{};
        q.op = HOP_INJECT; q.a = word; q.b = mask;
        return units_forward(be, device, q, err);
    }
    if (word == ~0ull) {  // synthetic critical-Xid event `mask`, handled like one delivered by NVML (xid=1)
        Gpu* g = gpu_at(be, device, err);
        if (!g) return B2DP_E_INVAL;
        // like xid_listener: no backend lock is held while the context's callback runs (it takes the context lock,
        // and Start()/labels/export take that lock before probe_mu)
        if (be->cfg.check_xid && !xid_is_application_error(mask)) {
            latch_xid(g, mask);
            be->fire_health_event();
        }
        return B2DP_OK;
    }
    std::lock_guard<std::mutex> pl(be->probe_mu);
    Gpu* g = gpu_at(be, device, err);
    if (!g) return B2DP_E_INVAL;
    if (word >= g->n_vec * 4) { err = "word index out of range"; return B2DP_E_INVAL; }
    cudaError_t ce = cudaSuccess;
    run_sync(g, [&] {
        probe_flush(g);
        hbm_poke<<<1, 1, 0, g->stream>>>(reinterpret_cast<uint32_t*>(g->buf[g->cur]), word, mask);
        ce = cudaStreamSynchronize(g->stream);
    });
    if (ce != cudaSuccess) { err = cuda_err("hbm_poke", ce); return B2DP_E_CUDA; }
    return B2DP_OK;
}

int cuda_probe_reset(CudaBackend* be, int device, std::string& err) {
    std::lock_guard<std::mutex> pl(be->probe_mu);
    if (be->units) {
        for (int i = 0; i < (int)be->units->units.size(); ++i) {
            if (device >= 0 && device != i) continue;
            be->unit_xid[i]->store(0);  // operator acknowledgement
            if (be->units->units[i].broken || !be->units->helpers) continue;
            HelperReq q{};
            q.op = HOP_RESET;
            int rc = units_forward(be, i, q, err);
            if (rc != B2DP_OK) return rc;
        }
        return device >= (int)be->units->units.size() ? B2DP_E_INVAL : B2DP_OK;
    }
    for (int i = 0; i < (int)be->gpus.size(); ++i) {
        if (device >= 0 && device != i) continue;
        Gpu* g = be->gpus[i].get();
        if (g->broken) continue;
        g->xid_fault.store(0);  // operator acknowledgement: a latched Xid is cleared together with the buffers
        cudaError_t ce = cudaSuccess;
        run_sync(g, [&] {
            probe_flush(g);
            hbm_fill<256><<<(int)g->sms * 8, 256, 0, g->stream>>>(g->buf[g->cur], g->n_vec, g->seed);
            ce = cudaStreamSynchronize(g->stream);
        });
        if (ce != cudaSuccess) { err = cuda_err("hbm_fill", ce); return B2DP_E_CUDA; }
    }
    if (device >= (int)be->gpus.size()) { err = "device index out of range"; return B2DP_E_INVAL; }
    return B2DP_OK;
}

int cuda_probe_peek(CudaBackend* be, int device, uint64_t word, uint32_t* out, uint64_t n, std::string& err) {
    std::lock_guard<std::mutex> pl(be->probe_mu);
    if (be->units) {
        for (uint64_t done = 0; done < n;) {  // 1 Mi words per exchange
            const uint64_t chunk = std::min<uint64_t>(n - done, 1u << 20);
            HelperReq q{};
            q.op = HOP_PEEK; q.a = word + done; q.b = chunk;
            std::vector<uint32_t> payload;
            int rc = units_forward(be, device, q, err, &payload);
            if (rc != B2DP_OK) return rc;
            memcpy(out + done, payload.data(), (size_t)chunk * 4);
            done += chunk;
        }
        return B2DP_OK;
    }
    Gpu* g = gpu_at(be, device, err);
    if (!g) return B2DP_E_INVAL;
    if (word + n > g->n_vec * 4) { err = "range out of bounds"; return B2DP_E_INVAL; }
    cudaError_t ce = cudaSuccess;
    run_sync(g, [&] {
        probe_flush(g);
        ce = cudaMemcpyAsync(out, reinterpret_cast<const uint32_t*>(g->buf[g->cur]) + word, n * 4, cudaMemcpyDeviceToHost,
                             g->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(g->stream);
    });
    if (ce != cudaSuccess) { err = cuda_err("peek", ce); return B2DP_E_CUDA; }
    return B2DP_OK;
}

// What the NVIDIA container runtime / a CDI spec calls the device `id` names: the GPU UUID (default, unambiguous)
// or the NVML index.  NOT the /dev/nvidia minor: minors and NVML indices differ on HGX boards.
std::string cuda_runtime_id(CudaBackend* be, const std::string& id, bool by_index) {
    if (be->units) {
        for (auto& u : be->units->units)
            if (u.dev.id == id) {
                if (!by_index || u.nvml_index < 0) return u.uuid;
                // NVIDIA_VISIBLE_DEVICES index syntax: "<gpu>" or "<gpu>:<mig device index>"
                return u.mig_slot >= 0 ? std::to_string(u.nvml_index) + ":" + std::to_string(u.mig_slot) : std::to_string(u.nvml_index);
            }
        return "";
    }
    for (auto& g : be->gpus)
        if (g->dev.id == id) {
            if (by_index && g->nvml_index >= 0) return std::to_string(g->nvml_index);
            return g->uuid;
        }
    return "";
}

int cuda_set_ref(CudaBackend* be, int device, float gbs_ref, std::string& err) {
    if (be->units) {
        std::lock_guard<std::mutex> pl(be->probe_mu);
        if (device >= (int)be->units->units.size()) { err = "device index out of range"; return B2DP_E_INVAL; }
        for (int i = 0; i < (int)be->units->units.size(); ++i) {
            if ((device >= 0 && device != i) || be->units->units[i].broken) continue;
            Unit& u = be->units->units[i];
            u.gbs_ref = gbs_ref > 0 ? gbs_ref : u.gbs_cal;
            HelperReq q{};
            q.op = HOP_SETREF;
            memcpy(&q.a, &u.gbs_ref, sizeof(float));
            int rc = units_forward(be, i, q, err);
            if (rc != B2DP_OK) return rc;
        }
        return B2DP_OK;
    }
    if (device >= (int)be->gpus.size()) { err = "device index out of range"; return B2DP_E_INVAL; }
    for (int i = 0; i < (int)be->gpus.size(); ++i) {
        if (device >= 0 && device != i) continue;
        Gpu* g = be->gpus[i].get();
        g->gbs_ref.store(gbs_ref > 0 ? gbs_ref : g->gbs_cal);  // <= 0: back to this device's own calibration
    }
    return B2DP_OK;
}

int cuda_describe(CudaBackend* be, int device, b2dp_probe_info* o, std::string& err) {
    if (device < 0 || device >= cuda_device_count(be)) { err = "device index out of range"; return B2DP_E_INVAL; }
    if (be->units) {
        std::lock_guard<std::mutex> pl(be->probe_mu);  // a fan-out may be restarting this unit's helper
        const Unit& u = be->units->units[device];
        o->slot_bytes = u.slot_bytes; o->total_memory = (uint64_t)u.vram; o->sm_count = (int32_t)u.sms; o->slots = be->cfg.slots;
        o->gbs_cal = u.gbs_cal; o->gbs_ref = u.gbs_ref; o->usable = u.broken ? 0 : 1; o->via_helper = be->units->helpers ? 1 : 0;
        copy_str(o->uuid, sizeof o->uuid, u.uuid);
        copy_str(o->name, sizeof o->name, u.name);
        return B2DP_OK;
    }
    const Gpu* g = be->gpus[device].get();
    o->slot_bytes = g->n_vec * 16; o->total_memory = (uint64_t)g->vram; o->sm_count = (int32_t)g->sms; o->slots = (int32_t)g->buf.size();
    o->gbs_cal = g->gbs_cal; o->gbs_ref = g->gbs_ref.load(); o->usable = g->broken ? 0 : 1; o->via_helper = 0;
    copy_str(o->uuid, sizeof o->uuid, g->uuid);
    copy_str(o->name, sizeof o->name, g->name);
    return B2DP_OK;
}

int cuda_compute_check(CudaBackend* be, const b2dp_compute_opts* opts, std::vector<b2dp_compute_result>& out, std::string& err) {
    std::lock_guard<std::mutex> pl(be->probe_mu);
    if (be->units) { err = "the tensor-core check with per-SM detail runs in-process only (probe=inproc on whole GPUs)"; return B2DP_E_UNSUPPORTED; }
    const uint32_t tiles = opts && opts->tiles ? opts->tiles : B2DP_COMPUTE_DEFAULT_TILES;
    if (tiles > B2DP_COMPUTE_MAX_TILES) { err = "tiles must be at most 65536"; return B2DP_E_INVAL; }
    const uint32_t timeout_ms = opts && opts->timeout_ms ? opts->timeout_ms : 5000;
    const bool timed = opts && (opts->flags & B2DP_COMPUTE_EVENT_TIMING);
    const size_t n = be->gpus.size();
    out.assign(n, b2dp_compute_result{});
    std::vector<size_t> idx;
    for (size_t i = 0; i < n; ++i) {
        Gpu* g = be->gpus[i].get();
        out[i].device = (int)i;
        out[i].sms = (int32_t)g->sms;
        out[i].first_bad_sm = out[i].first_bad_kind = out[i].first_bad_tile = out[i].first_bad_row = -1;
        if (g->broken) { out[i].err = B2DP_E_CUDA; err = g->broken_reason + " on " + g->dev.id; continue; }
        if (g->inflight.load()) { out[i].err = B2DP_E_TIMEOUT; continue; }  // an earlier pass or check is still running
        if (g->armed) run_sync(g, [g] { probe_flush(g); });  // a check queued behind an armed stream wait would stall
        idx.push_back(i);
    }
    tc_fanout(be, idx, tiles, timed, std::chrono::steady_clock::now() + std::chrono::milliseconds(timeout_ms), out);
    for (size_t i : idx) {
        out[i].device = (int)i;
        if (out[i].err != B2DP_OK || !out[i].healthy || out[i].sms_covered < out[i].sms) tc_log(be->gpus[i].get(), out[i]);
    }
    return B2DP_OK;
}

int cuda_compute_tile(CudaBackend* be, int device, int kind, int a_set, int b_set, float* c, std::string& err) {
    std::lock_guard<std::mutex> pl(be->probe_mu);
    if (be->units) { err = "in-process only (probe=inproc on whole GPUs)"; return B2DP_E_UNSUPPORTED; }
    Gpu* g = gpu_at(be, device, err);
    if (!g) return B2DP_E_INVAL;
    if (g->inflight.load()) { err = "an earlier pass is still running on this device"; return B2DP_E_TIMEOUT; }
    cudaError_t ce = cudaSuccess;
    bool published = false;
    run_sync(g, [&] {
        probe_flush(g);
        if ((ce = tc_setup(g)) != cudaSuccess) return;
        TcParams p = tc_params(g, kind, 1);
        p.fixed_comb = a_set * tc::kSets + b_set;
        p.c_out = g->tc_c;
        p.seq = ++g->tc_seq;
        p.publish = 1;
        if (kind == 0) tc_check<0><<<1, kTcThreads, kTcSmem, g->stream>>>(p);
        else tc_check<1><<<1, kTcThreads, kTcSmem, g->stream>>>(p);
        if ((ce = cudaGetLastError()) != cudaSuccess) return;
        if ((ce = cudaMemcpyAsync(c, g->tc_c, sizeof(float) * tc::kM * tc::kN, cudaMemcpyDeviceToHost, g->stream)) != cudaSuccess) return;
        ce = cudaStreamSynchronize(g->stream);
        published = g->tc_out_h->seq == p.seq;
    });
    if (ce != cudaSuccess) { err = cuda_err("tc_check", ce); return B2DP_E_CUDA; }
    if (!published) { err = "the tile did not publish its sequence number"; return B2DP_E_CUDA; }
    return B2DP_OK;
}

int cuda_compute_inject_fault(CudaBackend* be, int device, int sm, uint32_t mask, std::string& err) {
    std::lock_guard<std::mutex> pl(be->probe_mu);
    if (be->units) { err = "in-process only (probe=inproc on whole GPUs)"; return B2DP_E_UNSUPPORTED; }
    Gpu* g = gpu_at(be, device, err);
    if (!g) return B2DP_E_INVAL;
    g->tc_fault_sm = sm;
    g->tc_fault_mask = mask;
    return B2DP_OK;
}

bool cuda_device_paths(CudaBackend* be, const std::string& id, std::vector<std::string>& out) {
    if (be->units) {
        for (auto& u : be->units->units)
            if (u.dev.id == id) {
                out.push_back("/dev/nvidia" + std::to_string(u.parent_minor));
                if (u.mig_slot >= 0) {  // a MIG instance needs its GPU-instance and compute-instance capability nodes too
                    if (u.cap_gi >= 0) out.push_back("/dev/nvidia-caps/nvidia-cap" + std::to_string(u.cap_gi));
                    if (u.cap_ci >= 0) out.push_back("/dev/nvidia-caps/nvidia-cap" + std::to_string(u.cap_ci));
                }
                return true;
            }
        return false;
    }
    for (auto& g : be->gpus)
        if (g->dev.id == id) { out.push_back("/dev/nvidia" + std::to_string(g->dev.card)); return true; }
    return false;
}

// ---- P2P matrix ------------------------------------------------------------------------------
constexpr float kNvlinkRefGbs = 770.f, kNvlinkClassFraction = 0.25f;  // oracle/probe.py

int cuda_p2p_matrix(CudaBackend* be, const b2dp_p2p_opts* opts, float* gbs, int32_t* link_type, uint64_t* mism, int n,
                    std::string& err) {
    std::lock_guard<std::mutex> pl(be->probe_mu);
    if (be->units) {
        // no CUDA context here and no P2P between MIG instances: the link classes are DECLARED from NVML (gbs = 0)
        if (n != (int)be->units->units.size()) { err = "n must equal the device count"; return B2DP_E_INVAL; }
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) {
                gbs[(size_t)i * n + j] = 0; mism[(size_t)i * n + j] = 0;
                link_type[(size_t)i * n + j] = i == j ? 0 : units_link_type(be->nvml, be->units->units[i], be->units->units[j]);
            }
        return B2DP_OK;
    }
    if (n != (int)be->gpus.size()) { err = "n must equal the device count"; return B2DP_E_INVAL; }
    unsigned long long bytes = opts && opts->bytes ? opts->bytes : be->cfg.p2p_bytes;
    for (auto& g : be->gpus) if (!g->broken) bytes = std::min<unsigned long long>(bytes, g->n_vec * 16);  // the smallest ring slot bounds a pass
    bytes &= ~15ull;
    const unsigned long long n_vec = bytes / 16;
    const int iters = opts && opts->iters ? (int)opts->iters : 2;
    for (int i = 0; i < n * n; ++i) { gbs[i] = 0; link_type[i] = 0; mism[i] = 0; }
    // a probe pass that missed its deadline still owns its GPU's seed/ring state: let the workers drain; an armed
    // pass (prearm=1) is discarded, the matrix uses every stream and the spare buffers
    for (auto& g : be->gpus)
        if (!g->broken && g->th.joinable()) { Gpu* gp = g.get(); run_sync(gp, [gp] { probe_flush(gp); }); }
    const std::array<unsigned long long, 32>& bc = host_bitcounts(be, n_vec * 4);  // host closed form

    // peer capability + enable (on the reader's worker)
    std::vector<char> can((size_t)n * n, 0);
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            if (i == j) continue;
            int c = 0;
            if (be->gpus[i]->broken || be->gpus[j]->broken) continue;
            cudaDeviceCanAccessPeer(&c, be->gpus[i]->ordinal, be->gpus[j]->ordinal);
            can[(size_t)i * n + j] = (char)c;
            if (c && !be->gpus[i]->peer_enabled[j]) {
                Gpu* g = be->gpus[i].get();
                const int peer = be->gpus[j]->ordinal;
                cudaError_t ce = cudaSuccess;
                run_sync(g, [&] {
                    ce = cudaDeviceEnablePeerAccess(peer, 0);
                    if (ce == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); ce = cudaSuccess; }
                });
                if (ce != cudaSuccess) can[(size_t)i * n + j] = 0;
                else g->peer_enabled[j] = 1;
            }
        }

    struct PairRes { cudaError_t ce = cudaSuccess; float best_ms = 1e30f; ProbeOut out{}; bool ran = false; };
    auto run_pair = [&](int i, int j, PairRes* pr) {
        // GPU i reads GPU j's current pattern buffer into its own spare buffer
        Gpu* g = be->gpus[i].get();
        Gpu* peer = be->gpus[j].get();
        const uint4* src = peer->buf[peer->cur];
        const uint32_t seed = peer->seed;
        return post(g, [g, src, seed, n_vec, iters, pr] {
            pr->ran = true;
            for (int it = 0; it < iters + 1; ++it) {  // first iteration is a warm-up
                const unsigned long long seq = ++g->seq;
                cudaEventRecord(g->e0, g->stream);
                // the same smem-staged kernel as the health probe, with a peer-mapped source: the bulk
                // copies cross NVLink, verification happens on the receiving GPU
                hbm_probe_tma<kTmaCW, kTmaTileVec, kTmaStages>
                    <<<(int)g->sms * kTmaCtasPerSm, (kTmaCW + 1) * 32, kTmaSmem, g->stream>>>(
                        src, g->buf[g->next()], n_vec, seed, 0u, g->ctl, g->out_d, seq);
                cudaError_t e = cudaGetLastError();
                cudaEventRecord(g->e1, g->stream);
                if (e == cudaSuccess) e = cudaEventSynchronize(g->e1);
                float ms = 0;
                if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, g->e0, g->e1);
                if (e != cudaSuccess) { pr->ce = e; return; }
                memcpy(&pr->out, (const void*)g->out_h, sizeof(ProbeOut));
                if (it > 0 && ms < pr->best_ms) pr->best_ms = ms;
            }
        });
    };

    // N-1 rounds of disjoint matchings (circle method).  Default: one direction of every pair per
    // half-round (a pull's read requests travel against the other direction's data, so running
    // both directions at once measures ~635 GB/s per direction instead of the link's ~745 --
    // profiles/r01_p2p_sweep_2gpu.csv); B2DP_P2P_BIDIR runs both directions together (full-duplex stress).
    const bool bidir = opts && (opts->flags & B2DP_P2P_BIDIR);
    const int m = n % 2 ? n + 1 : n;
    for (int hr = 0; hr < 2 * (m - 1) && n > 1; ++hr) {
        const int r = hr / 2, half = hr % 2;
        if (bidir && half) continue;
        std::vector<std::pair<int, int>> pairs;
        auto add = [&](int a, int b) { if (a < n && b < n) pairs.push_back({a, b}); };  // >= n: bye
        add(m - 1, r);
        for (int k = 1; k < m / 2; ++k) add((r + k) % (m - 1), (r - k + (m - 1)) % (m - 1));
        std::vector<std::unique_ptr<PairRes>> prs;
        std::vector<std::shared_ptr<Completion>> cs;
        std::vector<std::pair<int, int>> dirs;
        for (auto& p : pairs)
            for (int d = 0; d < 2; ++d) {
                if (!bidir && d != half) continue;
                const int i = d ? p.second : p.first, j = d ? p.first : p.second;
                if (!can[(size_t)i * n + j]) continue;
                prs.push_back(std::make_unique<PairRes>());
                dirs.push_back({i, j});
                cs.push_back(run_pair(i, j, prs.back().get()));
            }
        for (auto& c : cs) c->wait();
        for (size_t k = 0; k < dirs.size(); ++k) {
            const int i = dirs[k].first, j = dirs[k].second;
            const PairRes& pr = *prs[k];
            if (pr.ce != cudaSuccess) { err = cuda_err("p2p_probe", pr.ce); return B2DP_E_CUDA; }
            const float g_ = (float)((double)bytes / (double)pr.best_ms * 1e-6);
            gbs[(size_t)i * n + j] = g_;
            uint64_t bad = pr.out.mismatches;
            if (pr.out.checksum != expected_checksum_from_counts(bc, n_vec * 4, be->gpus[j]->seed)) bad = bad ? bad : 1;
            mism[(size_t)i * n + j] = bad;
        }
    }
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            if (i == j) continue;
            // oracle/probe.py classify_link
            link_type[(size_t)i * n + j] = !can[(size_t)i * n + j] ? 0
                : gbs[(size_t)i * n + j] >= kNvlinkClassFraction * kNvlinkRefGbs ? 11 : 2;
        }
    return B2DP_OK;
}

}  // namespace b2dp
