// ctx.cpp -- context object, backend dispatch and the context-level C ABI
// (enumerate / health / ListAndWatch / Allocate / GetPreferredAllocation / labels / export).
#include <sys/stat.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cstdarg>
#include <climits>
#include <condition_variable>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "gosem.hpp"
#include "internal.hpp"
#include "pattern_math.hpp"
#include "pbwire.hpp"

using namespace b2dp;

namespace {
const char kHealthy[] = "Healthy";      // v1beta1/constants.go:21
const char kUnhealthy[] = "Unhealthy";  // v1beta1/constants.go:23
thread_local std::string t_last_error;

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}
}  // namespace

struct b2dp_ctx {
    enum Kind { KFD, CUDA } kind = KFD;
    std::string sysroot;        // kfd: plays "/"; cuda: where numa_node is looked up
    CudaBackend* cuda = nullptr;
    std::mutex mu;              // guards policy / allocator_init_error / links
    std::shared_ptr<BestEffortPolicy> policy;  // shared: a restart must not free it under a running Allocate
    bool started = false, allocator_init_error = false;
    std::vector<Link> links;    // cuda: measured link list (node ids), filled by the p2p matrix
    bool have_links = false;
    std::vector<float> p2p_gbs; // last matrix, n x n
    std::vector<Device> stream_devs;  // the device list of the current ListAndWatch stream
    bool have_stream_devs = false;
    std::string cdi_kind;             // cuda: optional CDI kind ("nvidia.com/gpu"): Allocate also names CDI devices
    bool ids_by_index = false;        // cuda: id_strategy=index -- NVML indices instead of UUIDs in NVIDIA_VISIBLE_DEVICES / CDI names
    std::string owned_tmp_root;       // synthetic: backend -- the generated tree, removed at close
    std::vector<b2dp_watch*> watches;  // running b2dp_watch loops (guarded by mu): a latched Xid beats them all at once
};

static int fail(int code, const std::string& msg) { t_last_error = msg; return code; }

namespace b2dp {
CudaBackend* ctx_cuda_backend(b2dp_ctx* c) { return c && c->kind == b2dp_ctx::CUDA ? c->cuda : nullptr; }
int ctx_fail(int code, const std::string& msg) { return fail(code, msg); }
}  // namespace b2dp

static int enumerate_ctx(b2dp_ctx* c, std::vector<Device>& devs) {
    std::string err;
    int rc = c->kind == b2dp_ctx::KFD ? kfd_enumerate(c->sysroot, devs, err) : cuda_enumerate(c->cuda, devs, err);
    if (rc != B2DP_OK) t_last_error = err;
    return rc;
}

// ---- diagnostics -------------------------------------------------------------------------------------------------------
namespace {
std::mutex g_log_mu;
b2dp_log_cb g_log_cb = nullptr;
void* g_log_user = nullptr;
std::atomic<bool> g_log_on{false};
}  // namespace
namespace b2dp {
bool log_enabled() { return g_log_on.load(std::memory_order_relaxed); }
void logf(int level, const char* fmt, ...) {
    if (!log_enabled()) return;
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    std::lock_guard<std::mutex> l(g_log_mu);  // serialises callbacks; the callback must not re-enter the library
    if (g_log_cb) g_log_cb(g_log_user, level, buf);
}
}  // namespace b2dp
extern "C" void b2dp_set_log_callback(b2dp_log_cb cb, void* user) {
    std::lock_guard<std::mutex> l(g_log_mu);
    g_log_cb = cb;
    g_log_user = user;
    g_log_on.store(cb != nullptr);
}

extern "C" const char* b2dp_strerror(int code) {
    switch (code) {
        case B2DP_OK: return "ok";
        case B2DP_E_INVAL: return "invalid argument";
        case B2DP_E_NOSPC: return "output capacity too small";
        case B2DP_E_IO: return "i/o error";
        case B2DP_E_NOTFOUND: return "Topology property not found.";
        case B2DP_E_SYNTAX: return "invalid syntax";
        case B2DP_E_RANGE: return "value out of range";
        case B2DP_E_NODRIVER: return "amdgpu driver unavailable. exiting with exit code 2.";
        case B2DP_E_NOGPU: return "no usable CUDA device";
        case B2DP_E_CUDA: return "CUDA error";
        case B2DP_E_TIMEOUT: return "probe deadline expired";
        case B2DP_E_UNSUPPORTED: return "not supported by this backend";
        case B2DP_E_PANIC: return "the reference would panic on this input";
        case B2DP_E_NOMEM: return "out of memory";
        case B2DP_E_HETEROGENEOUS:
            return "Partitions of different styles across GPUs in a node is not supported with single strategy. "
                   "Please start device plugin with mixed strategy";
        case B2DP_E_ALLOC_SIZE: return "allocation size can not be negative";
        case B2DP_E_ALLOC_AVAILABLE: return "available devices count less than allocation size";
        case B2DP_E_ALLOC_REQUIRED: return "must_include devices size is more than allocation size";
        case B2DP_E_ALLOC_REQ_AVAILABLE: return "must_include length should be less than or equal to avilable device size";
        case B2DP_E_ALLOC_INIT: return "Init method must be called before Allocate";
        case B2DP_E_ALLOC_NOCANDIDATE: return "No candidate subset found with matching criteria";
        case B2DP_E_ALLOC_EMPTY_DEVICES: return "Devices list is empty. Unable to calculate pair wise weights";
        case B2DP_E_ALLOC_NO_WEIGHTS: return "Besteffort Policy init failed to initialize p2pWeights";
        case B2DP_E_ALLOC_SUBSET_SIZE: return "subset size should be positive integer";
        case B2DP_E_ALLOC_SUBSET_AVAIL: return "subset size is more than available devices";
    }
    return "unknown error";
}
extern "C" int b2dp_abi_version(void) { return B2DP_ABI_VERSION; }

// ---- open / close ------------------------------------------------------------------------
static bool mkdirs(const std::string& p);
static bool write_file(const std::string& path, const std::string& data);
static bool write_synthetic_tree(const std::string& root, int n_gpus, int partitions, int n_cpu_nodes,
                                 const std::string& compute, const std::string& memory);
static void remove_tree(const std::string& root);

static bool parse_kv(const std::string& body, std::map<std::string, std::string>& kv) {
    size_t pos = 0;
    while (pos < body.size()) {
        size_t e = body.find(',', pos);
        if (e == std::string::npos) e = body.size();
        std::string item = body.substr(pos, e - pos);
        pos = e + 1;
        if (item.empty()) continue;
        size_t eq = item.find('=');
        if (eq == std::string::npos) return false;
        kv[item.substr(0, eq)] = item.substr(eq + 1);
    }
    return true;
}

extern "C" int b2dp_open(const char* uri, b2dp_ctx** out) {
    if (!uri || !out) return B2DP_E_INVAL;
    *out = nullptr;
    const std::string u = uri;
    if (u.compare(0, 4, "kfd:") == 0) {
        auto* c = new b2dp_ctx();
        c->kind = b2dp_ctx::KFD;
        c->sysroot = u.substr(4);
        if (c->sysroot.empty()) c->sysroot = "/";
        if (!go::exists(go::join(c->sysroot, "sys/module/amdgpu/drivers/"))) {  // amdgpu.go:150-152
            delete c;
            return fail(B2DP_E_NODRIVER, "amdgpu driver unavailable under " + u.substr(4));
        }
        *out = c;
        return B2DP_OK;
    }
    if (u.compare(0, 10, "synthetic:") == 0) {
        // "synthetic:<N>[,mig=<k>][,compute=<name>][,memory=<name>][,cpus=<c>]": a generated kfd-shaped tree of an
        // N x B200 NVSwitch node (every pair linked with type 11, GPUs split over two NUMA nodes, optionally k
        // partitions per GPU, the MIG/CPX-style layout) opened through the kfd: reader -- CPU only, no probe.
        std::string body = u.substr(10);
        const size_t comma = body.find(',');
        const int n_gpus = atoi(body.substr(0, comma).c_str());
        std::map<std::string, std::string> kv;
        if (comma != std::string::npos && !parse_kv(body.substr(comma + 1), kv)) return fail(B2DP_E_INVAL, "bad synthetic: uri");
        int mig = 1, cpus = 2;
        std::string compute, memory;
        for (auto& p : kv) {
            if (p.first == "mig") mig = atoi(p.second.c_str());
            else if (p.first == "compute") compute = p.second;
            else if (p.first == "memory") memory = p.second;
            else if (p.first == "cpus") cpus = atoi(p.second.c_str());
            else return fail(B2DP_E_INVAL, "unknown synthetic: option " + p.first);
        }
        if (n_gpus < 1 || n_gpus > 64 || mig < 1 || mig > 8 || cpus < 0 || cpus > 16) return fail(B2DP_E_INVAL, "synthetic: wants 1..64 GPUs, mig 1..8");
        // partitions are only listed when their parent GPU reports BOTH partition types (amdgpu.go:240-249)
        if (mig > 1 && compute.empty()) compute = "mig" + std::to_string(mig);
        if (mig > 1 && memory.empty()) memory = "nps1";
        char tmpl[64];
        snprintf(tmpl, sizeof tmpl, "%s/b2dp_syn_XXXXXX", go::is_dir("/dev/shm") ? "/dev/shm" : "/tmp");
        if (!mkdtemp(tmpl)) return fail(B2DP_E_IO, std::string("mkdtemp: ") + strerror(errno));
        if (!write_synthetic_tree(tmpl, n_gpus, mig, cpus, compute, memory)) { remove_tree(tmpl); return fail(B2DP_E_IO, "writing the synthetic tree failed"); }
        auto* c = new b2dp_ctx();
        c->kind = b2dp_ctx::KFD;
        c->sysroot = tmpl;
        c->owned_tmp_root = tmpl;
        *out = c;
        return B2DP_OK;
    }
    if (u.compare(0, 5, "nvml:") == 0) return b2dp_open(("cuda:probe=off" + (u.size() > 5 ? "," + u.substr(5) : std::string())).c_str(), out);  // SURVEY 8(b)'s name for it
    if (u.compare(0, 5, "cuda:") == 0) {
        std::map<std::string, std::string> kv;
        if (!parse_kv(u.substr(5), kv)) return fail(B2DP_E_INVAL, "bad cuda: uri");
        CudaConfig cfg;
        std::string cdi_kind;
        bool ids_by_index = false;
        for (auto& p : kv) {
            if (p.first == "cdi") { cdi_kind = p.second; continue; }
            if (p.first == "id_strategy") {
                if (p.second == "index") ids_by_index = true;
                else if (p.second != "uuid") return fail(B2DP_E_INVAL, "id_strategy= wants uuid|index");
                continue;
            }
            if (p.first == "devices") {
                size_t pos = 0;
                while (pos <= p.second.size()) {
                    size_t e = p.second.find('+', pos);
                    if (e == std::string::npos) e = p.second.size();
                    if (e > pos) cfg.devices.push_back(atoi(p.second.substr(pos, e - pos).c_str()));
                    pos = e + 1;
                }
            } else if (p.first == "bytes") cfg.bytes = strtoull(p.second.c_str(), nullptr, 0);
            else if (p.first == "slots") cfg.slots = atoi(p.second.c_str());
            else if (p.first == "p2p_bytes") cfg.p2p_bytes = strtoull(p.second.c_str(), nullptr, 0);
            else if (p.first == "min_gbs") cfg.min_gbs = (float)atof(p.second.c_str());
            else if (p.first == "min_frac") cfg.min_frac = (float)atof(p.second.c_str());
            else if (p.first == "ref_gbs") cfg.ref_gbs = (float)atof(p.second.c_str());
            else if (p.first == "calib") cfg.calib = atoi(p.second.c_str());
            else if (p.first == "slow_passes") cfg.slow_passes = atoi(p.second.c_str());
            else if (p.first == "prearm") cfg.prearm = p.second != "0";
            else if (p.first == "probe") {
                if (p.second == "inproc") cfg.probe_mode = 0;
                else if (p.second == "helpers") cfg.probe_mode = 1;
                else if (p.second == "off") cfg.probe_mode = 2;
                else return fail(B2DP_E_INVAL, "probe= wants inproc|helpers|off");
            } else if (p.first == "mig") {
                if (p.second == "auto") cfg.mig_auto = true;
                else if (p.second == "off") cfg.mig_auto = false;
                else return fail(B2DP_E_INVAL, "mig= wants auto|off");
            } else if (p.first == "mig_bytes") cfg.mig_bytes = strtoull(p.second.c_str(), nullptr, 0);
            else if (p.first == "seed_index") cfg.seed_index = atoi(p.second.c_str());
            else if (p.first == "launchers") cfg.launchers = atoi(p.second.c_str());
            else if (p.first == "spin_us") cfg.spin_us = atoi(p.second.c_str());
            else if (p.first == "pin") cfg.pin_caller = p.second != "0";
            else if (p.first == "sysroot") cfg.sysroot = p.second;
            else if (p.first == "busy") {
                if (p.second == "probe") cfg.busy_policy = 0;
                else if (p.second == "skip") cfg.busy_policy = 1;
                else if (p.second == "shrink") cfg.busy_policy = 2;
                else return fail(B2DP_E_INVAL, "busy= wants probe|skip|shrink");
            } else if (p.first == "shrink_bytes") cfg.shrink_bytes = strtoull(p.second.c_str(), nullptr, 0);
            else if (p.first == "ecc") cfg.check_ecc = p.second != "0";
            else if (p.first == "xid") cfg.check_xid = p.second != "0";
            else if (p.first == "compute") {
                if (p.second == "0") cfg.compute = false;
                else if (p.second == "1") cfg.compute = true;
                else return fail(B2DP_E_INVAL, "compute= wants 0|1");
            }
            else if (p.first == "break") {
                size_t pos = 0;
                while (pos <= p.second.size()) {
                    size_t e = p.second.find('+', pos);
                    if (e == std::string::npos) e = p.second.size();
                    if (e > pos) cfg.break_devices.push_back(atoi(p.second.substr(pos, e - pos).c_str()));
                    pos = e + 1;
                }
            }
            else return fail(B2DP_E_INVAL, "unknown cuda: option " + p.first);
        }
        if (!kv.count("prearm")) { const char* e = getenv("B2DP_PREARM"); if (e && *e) cfg.prearm = *e != '0'; }  // site / test-wide default
        if (cfg.bytes < 4096 || cfg.bytes % 16) return fail(B2DP_E_INVAL, "bytes must be a multiple of 16, >= 4096");
        if (cfg.mig_bytes < 4096 || cfg.mig_bytes % 16) return fail(B2DP_E_INVAL, "mig_bytes must be a multiple of 16, >= 4096");
        // what every helper process inherits: the verdict-related options (the ring geometry is set per unit)
        for (const char* k : {"min_gbs", "min_frac", "ref_gbs", "calib", "slow_passes", "prearm", "busy", "shrink_bytes", "ecc", "compute"}) {
            auto it = kv.find(k);
            if (it != kv.end()) cfg.passthrough += std::string(",") + k + "=" + it->second;
        }
        if (cfg.slots < 2 || cfg.slots > 4096) return fail(B2DP_E_INVAL, "slots must be in [2, 4096]");
        if (!(cfg.min_frac >= 0.f && cfg.min_frac <= 1.f)) return fail(B2DP_E_INVAL, "min_frac must be in [0, 1]");
        if (cfg.calib < 0 || cfg.calib > 64) return fail(B2DP_E_INVAL, "calib must be in [0, 64]");
        if (cfg.slow_passes < 1 || cfg.slow_passes > 1000) return fail(B2DP_E_INVAL, "slow_passes must be in [1, 1000]");
        if (cfg.launchers < 1 || cfg.launchers > 2) return fail(B2DP_E_INVAL, "launchers must be 1 or 2");
        if (cfg.spin_us < 0 || cfg.spin_us > 100000) return fail(B2DP_E_INVAL, "spin_us must be in [0, 100000]");
        std::string err;
        CudaBackend* be = nullptr;
        int rc = cuda_backend_open(cfg, &be, err);
        if (rc != B2DP_OK) return fail(rc, err);
        auto* c = new b2dp_ctx();
        c->kind = b2dp_ctx::CUDA;
        c->sysroot = cfg.sysroot;
        c->cuda = be;
        c->cdi_kind = cdi_kind;
        c->ids_by_index = ids_by_index;
        // xid=1: a device-level Xid is pushed to the kubelet at once -- every running ListAndWatch loop of this
        // context runs a heartbeat cycle now instead of at the next pulse (the reference only learns at a pulse)
        cuda_set_health_event_callback(be, [c] {
            std::lock_guard<std::mutex> g(c->mu);
            for (b2dp_watch* w : c->watches) b2dp_watch_beat(w);
        });
        *out = c;
        return B2DP_OK;
    }
    return fail(B2DP_E_INVAL, "unknown backend uri (want kfd:<sysroot>, synthetic:<N>[,mig=<k>] or cuda:[opts])");
}

extern "C" void b2dp_close(b2dp_ctx* c) {
    if (!c) return;
    if (c->cuda) cuda_backend_close(c->cuda);
    if (!c->owned_tmp_root.empty()) remove_tree(c->owned_tmp_root);
    delete c;
}

extern "C" const char* b2dp_last_error(b2dp_ctx*) { return t_last_error.c_str(); }

// ---- enumerate & friends -----------------------------------------------------------------
extern "C" int b2dp_enumerate(b2dp_ctx* c, b2dp_device* out, int cap, int* n) {
    if (!c || !n || cap < 0) return B2DP_E_INVAL;
    std::vector<Device> devs;
    int rc = enumerate_ctx(c, devs);
    if (rc != B2DP_OK) return rc;
    *n = (int)devs.size();
    if (*n > cap) return B2DP_E_NOSPC;
    if (*n && !out) return B2DP_E_INVAL;
    for (int i = 0; i < *n; ++i) to_abi(devs[i], &out[i]);
    return B2DP_OK;
}

extern "C" int b2dp_partition_histogram(b2dp_ctx* c, b2dp_kv_count* out, int cap, int* n) {
    if (!c || !n || cap < 0) return B2DP_E_INVAL;
    std::vector<Device> devs;
    int rc = enumerate_ctx(c, devs);
    if (rc != B2DP_OK) return rc;
    auto h = partition_histogram(devs);
    *n = (int)h.size();
    if (*n > cap) return B2DP_E_NOSPC;
    if (*n && !out) return B2DP_E_INVAL;
    int i = 0;
    for (auto& kv : h) { memset(&out[i], 0, sizeof out[i]); copy_str(out[i].key, 64, kv.first); out[i].count = kv.second; ++i; }
    return B2DP_OK;
}

extern "C" int b2dp_is_homogeneous(b2dp_ctx* c, int32_t* homogeneous) {
    if (!c || !homogeneous) return B2DP_E_INVAL;
    std::vector<Device> devs;
    int rc = enumerate_ctx(c, devs);
    if (rc != B2DP_OK) return rc;
    *homogeneous = partition_histogram(devs).size() <= 1 ? 1 : 0;
    return B2DP_OK;
}

static void label_source(b2dp_ctx* c, LabelSource& src) {
    src.sysroot = c->sysroot;
    if (c->kind == b2dp_ctx::CUDA) cuda_label_source(c->cuda, src);
}

extern "C" int b2dp_partition_supported(b2dp_ctx* c, int which, int32_t* supported) {
    if (!c || !supported || which < 0 || which > 1) return B2DP_E_INVAL;
    if (c->kind == b2dp_ctx::KFD) *supported = kfd_partition_supported(c->sysroot, which) ? 1 : 0;
    else { LabelSource s; label_source(c, s); *supported = s.part_supported[which] ? 1 : 0; }
    return B2DP_OK;
}

extern "C" int b2dp_resource_list(b2dp_ctx* c, const char* strategy, char (*names)[64], int cap, int* n) {
    if (!c || !n || cap < 0) return B2DP_E_INVAL;
    std::vector<Device> devs;
    int rc = enumerate_ctx(c, devs);
    if (rc != B2DP_OK) return rc;
    std::vector<std::string> res;
    rc = resource_list(devs, strategy, res);
    if (rc != B2DP_OK) return rc;
    *n = (int)res.size();
    if (*n > cap) return B2DP_E_NOSPC;
    if (*n && !names) return B2DP_E_INVAL;
    for (int i = 0; i < *n; ++i) copy_str(names[i], 64, res[i]);
    return B2DP_OK;
}

static bool node_health(b2dp_ctx* c) {
    if (c->kind == b2dp_ctx::KFD) return kfd_simple_health_check(go::join(c->sysroot, "sys/class/kfd/kfd"));
    return cuda_node_health(c->cuda) == 1;
}

extern "C" int b2dp_node_health(b2dp_ctx* c, int32_t* healthy) {
    if (!c || !healthy) return B2DP_E_INVAL;
    *healthy = node_health(c) ? 1 : 0;
    return B2DP_OK;
}

// ---- probe -------------------------------------------------------------------------------
extern "C" int b2dp_probe_health(b2dp_ctx* c, const b2dp_probe_opts* opts, b2dp_probe_result* out, int cap, int* n) {
    if (!c || !n || cap < 0) return B2DP_E_INVAL;
    if (c->kind != b2dp_ctx::CUDA)
        return fail(B2DP_E_UNSUPPORTED, "the GPU health probe needs the cuda: backend (there is no CPU fallback)");
    std::vector<b2dp_probe_result> res;
    std::string err;
    int rc = cuda_probe(c->cuda, opts, res, err);
    if (rc != B2DP_OK) return fail(rc, err);
    *n = (int)res.size();
    if (*n > cap) return B2DP_E_NOSPC;
    if (*n && !out) return B2DP_E_INVAL;
    memcpy(out, res.data(), res.size() * sizeof(b2dp_probe_result));
    return B2DP_OK;
}
extern "C" int b2dp_probe_inject_fault(b2dp_ctx* c, int device, uint64_t word_index, uint32_t mask) {
    if (!c) return B2DP_E_INVAL;
    if (c->kind != b2dp_ctx::CUDA) return fail(B2DP_E_UNSUPPORTED, "cuda: backend only");
    std::string err;
    int rc = cuda_inject_fault(c->cuda, device, word_index, mask, err);
    return rc == B2DP_OK ? rc : fail(rc, err);
}
extern "C" int b2dp_probe_reset(b2dp_ctx* c, int device) {
    if (!c) return B2DP_E_INVAL;
    if (c->kind != b2dp_ctx::CUDA) return fail(B2DP_E_UNSUPPORTED, "cuda: backend only");
    std::string err;
    int rc = cuda_probe_reset(c->cuda, device, err);
    return rc == B2DP_OK ? rc : fail(rc, err);
}
extern "C" int b2dp_probe_set_ref(b2dp_ctx* c, int device, float gbs_ref) {
    if (!c) return B2DP_E_INVAL;
    if (c->kind != b2dp_ctx::CUDA) return fail(B2DP_E_UNSUPPORTED, "cuda: backend only");
    std::string err;
    int rc = cuda_set_ref(c->cuda, device, gbs_ref, err);
    return rc == B2DP_OK ? rc : fail(rc, err);
}
extern "C" int b2dp_probe_describe(b2dp_ctx* c, int device, b2dp_probe_info* out) {
    if (!c || !out) return B2DP_E_INVAL;
    if (c->kind != b2dp_ctx::CUDA) return fail(B2DP_E_UNSUPPORTED, "cuda: backend only");
    std::string err;
    memset(out, 0, sizeof *out);
    int rc = cuda_describe(c->cuda, device, out, err);
    return rc == B2DP_OK ? rc : fail(rc, err);
}
extern "C" int b2dp_expected_checksum(uint64_t n_words, uint32_t seed, uint64_t* checksum) {
    if (!checksum) return B2DP_E_INVAL;
    *checksum = expected_checksum_host(n_words, seed);
    return B2DP_OK;
}
extern "C" int b2dp_probe_peek(b2dp_ctx* c, int device, uint64_t word_index, uint32_t* out, uint64_t n_words) {
    if (!c || (!out && n_words)) return B2DP_E_INVAL;
    if (c->kind != b2dp_ctx::CUDA) return fail(B2DP_E_UNSUPPORTED, "cuda: backend only");
    std::string err;
    int rc = cuda_probe_peek(c->cuda, device, word_index, out, n_words, err);
    return rc == B2DP_OK ? rc : fail(rc, err);
}

extern "C" int b2dp_merge_health(const char (*ids)[64], int n, int32_t default_healthy, int have_source,
                                 const char (*src_ids)[64], const int32_t* src_health, int m, int32_t* out) {
    if (n < 0 || m < 0 || (n && (!ids || !out)) || (have_source && m && (!src_ids || !src_health))) return B2DP_E_INVAL;
    // health.go:86-106; hMap built at health.go:74-80 (later entries overwrite earlier ones)
    std::map<std::string, int> hmap;
    if (have_source)
        for (int j = 0; j < m; ++j) hmap[src_ids[j]] = src_health[j] ? 1 : 0;
    for (int i = 0; i < n; ++i) {
        if (!have_source) { out[i] = default_healthy ? 1 : 0; continue; }
        auto it = hmap.find(ids[i]);
        out[i] = it != hmap.end() ? it->second : (default_healthy ? 1 : 0);
    }
    return B2DP_OK;
}

// ---- ListAndWatch ------------------------------------------------------------------------
extern "C" int b2dp_list_and_watch(b2dp_ctx* c, const char* resource, const b2dp_cycle_opts* opts, uint8_t* buf,
                                   size_t cap, size_t* len, b2dp_cycle_stats* stats) {
    if (!c || !len) return B2DP_E_INVAL;
    const double t0 = now_ms();
    b2dp_cycle_stats st{};
    const uint32_t flags = opts ? opts->flags : B2DP_LW_INITIAL;
    const bool heartbeat = (flags & B2DP_LW_HEARTBEAT) != 0;
    *len = 0;

    // plugin.go:231-237: GetAMDGPUs + IsHomogeneous at stream start (the reference enumerates
    // twice; one enumeration serves both here).  The device list is built ONCE per stream
    // (plugin.go:235-299) and only re-sent with new health on a heartbeat (plugin.go:304-320),
    // so a heartbeat reuses the list of the last INITIAL call.
    std::vector<Device> devs;
    int rc = B2DP_OK;
    {
        std::lock_guard<std::mutex> g(c->mu);
        if (heartbeat && c->have_stream_devs) devs = c->stream_devs;
    }
    if (devs.empty()) {
        rc = enumerate_ctx(c, devs);
        if (rc != B2DP_OK) return rc;
        std::lock_guard<std::mutex> g(c->mu);
        c->stream_devs = devs;
        c->have_stream_devs = true;
    }
    const bool homogeneous = partition_histogram(devs).size() <= 1;
    st.homogeneous = homogeneous;
    const double t1 = now_ms();
    st.ms_enumerate = (float)(t1 - t0);

    // plugin.go:241-299: which devices this resource's stream carries
    std::vector<const Device*> sel;
    if (homogeneous) for (auto& d : devs) sel.push_back(&d);
    else {
        const std::string want = resource ? resource : "";
        for (auto& d : devs) if (d.compute + "_" + d.memory == want) sel.push_back(&d);
        if (sel.empty()) { st.ms_total = (float)(now_ms() - t0); if (stats) *stats = st; return B2DP_OK; }
    }

    std::vector<int> healthy(sel.size(), 1);
    st.node_healthy = 1;
    if (heartbeat) {
        const bool def = node_health(c);  // plugin.go:305-309
        st.node_healthy = def;
        std::map<std::string, int> hmap;
        bool have_source = false;
        if (flags & B2DP_LW_EXTERNAL_SOURCE) {
            have_source = true;
            if (opts && opts->src_n > 0 && (!opts->src_ids || !opts->src_health)) return B2DP_E_INVAL;
            for (int j = 0; opts && j < opts->src_n; ++j) hmap[opts->src_ids[j]] = opts->src_health[j] ? 1 : 0;
        } else if (!(flags & B2DP_LW_NO_PROBE) && c->kind == b2dp_ctx::CUDA) {
            std::vector<b2dp_probe_result> res;
            std::string err;
            const double p0 = now_ms();
            rc = cuda_probe(c->cuda, opts ? &opts->probe : nullptr, res, err);
            st.ms_probe = (float)(now_ms() - p0);
            if (rc != B2DP_OK) return fail(rc, err);
            // the probe answers per enumerated device (same order as devs)
            have_source = true;
            st.probe_gbs_min = 1e30f;
            st.probe_frac_min = 1e30f;
            for (auto& r : res) {
                if (r.device >= 0 && r.device < (int)devs.size()) hmap[devs[r.device].id] = r.healthy;
                if (!r.healthy && log_enabled() && r.device >= 0 && r.device < (int)devs.size())  // why the bit flipped
                    logf(1, "%s Unhealthy: err=%d (%s) mismatches=%llu first_bad_word=%llu checksum_%s rate=%.0f GB/s floor=%.0f (%.3f of ceiling %.0f) flags=0x%x",
                         devs[r.device].id.c_str(), r.err, b2dp_strerror(r.err), (unsigned long long)r.mismatches,
                         (unsigned long long)r.first_bad_word, r.checksum == r.expected_checksum ? "ok" : "BAD", r.gbs, r.min_gbs_applied, r.frac,
                         r.gbs_ref, r.flags);
                st.probe_bytes += r.bytes;
                st.probe_gbs_sum += r.gbs;
                if (r.gbs < st.probe_gbs_min) st.probe_gbs_min = r.gbs;
                if (r.ms_device > st.probe_ms_device_max) st.probe_ms_device_max = r.ms_device;
                if (r.gbs_ref > 0 && r.frac < st.probe_frac_min) st.probe_frac_min = r.frac;
            }
            if (res.empty()) st.probe_gbs_min = 0;
            if (st.probe_frac_min > 1e29f) st.probe_frac_min = 0;
            if ((flags & B2DP_LW_LINK_CHECK) && devs.size() > 1) {
                // optional: re-measure the NVLink matrix (both directions at once, one timed pass per
                // pair) and fail a device whose link to any peer delivers corrupt data or has dropped
                // out of the class it had when the topology was first measured
                const int n = (int)devs.size();
                std::vector<float> gbs((size_t)n * n);
                std::vector<int32_t> lt((size_t)n * n);
                std::vector<uint64_t> mm((size_t)n * n);
                b2dp_p2p_opts po{};
                po.bytes = 64ull << 20; po.iters = 1; po.flags = B2DP_P2P_BIDIR;
                const double l0 = now_ms();
                rc = cuda_p2p_matrix(c->cuda, &po, gbs.data(), lt.data(), mm.data(), n, err);
                st.ms_link_check = (float)(now_ms() - l0);
                if (rc != B2DP_OK) return fail(rc, err);
                std::lock_guard<std::mutex> g(c->mu);
                for (int i = 0; i < n; ++i)
                    for (int j = 0; j < n; ++j) {
                        if (i == j) continue;
                        bool bad = mm[(size_t)i * n + j] != 0;
                        if (c->have_links)
                            for (const auto& l : c->links)
                                if (l.from == devs[i].node_id && l.to == devs[j].node_id && l.type == 11 && lt[(size_t)i * n + j] != 11)
                                    bad = true;
                        if (bad) { hmap[devs[i].id] = 0; st.n_link_faults++; }
                    }
            }
        }
        for (size_t i = 0; i < sel.size(); ++i) {  // health.go:93-105
            if (!have_source) { healthy[i] = def; continue; }
            auto it = hmap.find(sel[i]->id);
            healthy[i] = it != hmap.end() ? it->second : (int)def;
        }
    }

    const double e0 = now_ms();
    std::string wire;
    wire.reserve(sel.size() * 48);
    for (size_t i = 0; i < sel.size(); ++i) {
        pb::encode_device(wire, sel[i]->id, healthy[i] ? kHealthy : kUnhealthy, sel[i]->numa);
        if (!healthy[i]) st.n_unhealthy++;
    }
    st.n_devices = (int)sel.size();
    st.ms_encode = (float)(now_ms() - e0);
    *len = wire.size();
    st.ms_total = (float)(now_ms() - t0);
    if (stats) *stats = st;
    if (wire.size() > cap) return B2DP_E_NOSPC;
    if (!wire.empty() && !buf) return B2DP_E_INVAL;
    memcpy(buf, wire.data(), wire.size());
    return B2DP_OK;
}

// ---- native ListAndWatch loop ------------------------------------------------------------
// plugin.go:229-330 as a library-owned thread: the initial list at stream start, then one
// heartbeat cycle per tick -- from the built-in ticker (cmd/k8s-device-plugin/main.go:129-137,
// `-pulse`) or from b2dp_watch_beat() (the reference's `l.Heartbeat <- true`) -- until
// b2dp_watch_stop() (the reference's p.signal, plugin.go:322-329).
struct b2dp_watch {
    b2dp_ctx* ctx = nullptr;
    std::string resource;
    b2dp_cycle_opts opts{};
    uint32_t pulse_ms = 0;
    b2dp_watch_cb cb = nullptr;
    void* user = nullptr;
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    int pending_beats = 0;
    bool stop = false;
    bool self_delete = false;  // stop() was called from the callback: the loop frees the handle on its way out
};

static void watch_send(b2dp_watch* w, uint32_t flags) {
    std::vector<uint8_t> buf(1 << 14);
    b2dp_cycle_opts o = w->opts;
    o.flags = (o.flags & ~(B2DP_LW_INITIAL | B2DP_LW_HEARTBEAT)) | flags;
    size_t len = 0;
    b2dp_cycle_stats st{};
    int rc = b2dp_list_and_watch(w->ctx, w->resource.c_str(), &o, buf.data(), buf.size(), &len, &st);
    if (rc == B2DP_E_NOSPC) {
        buf.resize(len);
        rc = b2dp_list_and_watch(w->ctx, w->resource.c_str(), &o, buf.data(), buf.size(), &len, &st);
    }
    // plugin.go:296-298: a heterogeneous node with no devices of this resource sends nothing
    if (rc == B2DP_OK && (st.n_devices || st.homogeneous)) w->cb(w->user, rc, buf.data(), len, &st);
    else if (rc != B2DP_OK) w->cb(w->user, rc, nullptr, 0, &st);
}

static void watch_loop(b2dp_watch* w) {
    watch_send(w, B2DP_LW_INITIAL);
    auto next = std::chrono::steady_clock::now() + std::chrono::milliseconds(w->pulse_ms);
    for (;;) {
        {
            std::unique_lock<std::mutex> l(w->mu);
            auto pred = [&] { return w->stop || w->pending_beats > 0; };
            if (w->pulse_ms) {
                // launchers=2: wake the helper launcher a moment before the tick so the fan-out finds it spinning
                if (w->ctx->kind == b2dp_ctx::CUDA && w->pulse_ms >= 2 &&
                    !w->cv.wait_until(l, next - std::chrono::microseconds(300), pred))
                    cuda_prearm(w->ctx->cuda);
                if (!w->cv.wait_until(l, next, pred)) {  // ticker fired
                    next += std::chrono::milliseconds(w->pulse_ms);
                    w->pending_beats++;
                }
            } else w->cv.wait(l, pred);
            if (w->stop) {
                const bool del = w->self_delete;
                l.unlock();
                if (del) delete w;
                return;
            }
            w->pending_beats--;
        }
        watch_send(w, B2DP_LW_HEARTBEAT);
    }
}

extern "C" int b2dp_watch_start(b2dp_ctx* c, const char* resource, uint32_t pulse_ms, const b2dp_cycle_opts* opts,
                                b2dp_watch_cb cb, void* user, b2dp_watch** out) {
    if (!c || !cb || !out) return B2DP_E_INVAL;
    auto* w = new b2dp_watch();
    w->ctx = c;
    w->resource = resource ? resource : "gpu";
    if (opts) w->opts = *opts;
    w->pulse_ms = pulse_ms;
    w->cb = cb;
    w->user = user;
    { std::lock_guard<std::mutex> g(c->mu); c->watches.push_back(w); }
    w->th = std::thread(watch_loop, w);
    *out = w;
    return B2DP_OK;
}

extern "C" int b2dp_watch_beat(b2dp_watch* w) {
    if (!w) return B2DP_E_INVAL;
    { std::lock_guard<std::mutex> l(w->mu); w->pending_beats++; }
    w->cv.notify_one();
    return B2DP_OK;
}

extern "C" void b2dp_watch_stop(b2dp_watch* w) {
    if (!w) return;
    {
        std::lock_guard<std::mutex> g(w->ctx->mu);
        auto& ws = w->ctx->watches;
        ws.erase(std::remove(ws.begin(), ws.end(), w), ws.end());
    }
    if (std::this_thread::get_id() == w->th.get_id()) {  // called from the callback: cannot join ourselves
        { std::lock_guard<std::mutex> l(w->mu); w->stop = true; w->self_delete = true; }
        w->th.detach();
        return;
    }
    { std::lock_guard<std::mutex> l(w->mu); w->stop = true; }
    w->cv.notify_all();
    if (w->th.joinable()) w->th.join();
    delete w;
}

// ---- Allocate ----------------------------------------------------------------------------
static int device_specs(b2dp_ctx* c, const char* const* ids, int n_ids, std::vector<b2dp_devspec>& specs) {
    // plugin.go:375 reads p.AMDGPUs, the table built when the ListAndWatch stream started (plugin.go:231):
    // use that snapshot; only a context that never streamed enumerates here
    std::vector<Device> devs;
    bool have = false;
    {
        std::lock_guard<std::mutex> g(c->mu);
        if (c->have_stream_devs) { devs = c->stream_devs; have = true; }
    }
    if (!have) {
        int rc = enumerate_ctx(c, devs);
        if (rc != B2DP_OK) return rc;
    }
    auto push = [&](const std::string& p) {
        b2dp_devspec s{};
        copy_str(s.host_path, sizeof s.host_path, p);
        copy_str(s.container_path, sizeof s.container_path, p);
        copy_str(s.permissions, sizeof s.permissions, "rw");
        specs.push_back(s);
    };
    if (c->kind == b2dp_ctx::KFD) push("/dev/kfd");  // plugin.go:364-370
    else { push("/dev/nvidiactl"); push("/dev/nvidia-uvm"); push("/dev/nvidia-uvm-tools"); }
    for (int i = 0; i < n_ids; ++i) {
        const std::string id = ids[i] ? ids[i] : "";
        for (const auto& d : devs) {
            if (d.id != id) continue;
            if (c->kind == b2dp_ctx::KFD) {  // plugin.go:375-386 (canonical order: card, renderD)
                push("/dev/dri/card" + std::to_string(d.card));
                push("/dev/dri/renderD" + std::to_string(d.render_d));
            } else {  // whole GPU: /dev/nvidia<minor>; MIG instance: the parent's node + its two capability nodes
                std::vector<std::string> paths;
                if (!cuda_device_paths(c->cuda, d.id, paths)) paths.push_back("/dev/nvidia" + std::to_string(d.card));
                for (auto& pth : paths) {
                    bool dup = false;  // instances of one GPU share the parent's node
                    for (auto& spec : specs) dup = dup || pth == spec.host_path;
                    if (!dup) push(pth);
                }
            }
            break;
        }
    }
    return B2DP_OK;
}

extern "C" int b2dp_device_specs(b2dp_ctx* c, const char* const* ids, int n_ids, b2dp_devspec* out, int cap, int* n) {
    if (!c || !n || n_ids < 0 || (n_ids && !ids) || cap < 0) return B2DP_E_INVAL;
    std::vector<b2dp_devspec> specs;
    int rc = device_specs(c, ids, n_ids, specs);
    if (rc != B2DP_OK) return rc;
    *n = (int)specs.size();
    if (*n > cap) return B2DP_E_NOSPC;
    if (*n && !out) return B2DP_E_INVAL;
    memcpy(out, specs.data(), specs.size() * sizeof(b2dp_devspec));
    return B2DP_OK;
}

extern "C" int b2dp_allocate_response(b2dp_ctx* c, const char* const* ids, int n_ids, uint8_t* buf, size_t cap,
                                      size_t* len) {
    if (!c || !len || n_ids < 0 || (n_ids && !ids)) return B2DP_E_INVAL;
    std::vector<b2dp_devspec> specs;
    int rc = device_specs(c, ids, n_ids, specs);
    if (rc != B2DP_OK) return rc;
    std::string wire;
    // The reference's Allocate sets no envs (plugin.go:356-393).  On NVIDIA nodes the container runtime hook selects
    // GPUs from NVIDIA_VISIBLE_DEVICES, so the cuda backend also names the allocated devices there (envs = field 1,
    // map<string,string>) -- by UUID (or NVML index with id_strategy=index), never by /dev/nvidia minor: the runtime
    // reads a bare integer as an NVML index, and minors differ from indices on HGX boards.
    std::vector<std::string> rt_ids;
    if (c->kind == b2dp_ctx::CUDA) {
        for (int i = 0; i < n_ids; ++i) {
            if (!ids[i]) continue;
            const std::string rid = cuda_runtime_id(c->cuda, ids[i], c->ids_by_index);
            if (!rid.empty()) rt_ids.push_back(rid);
        }
        std::string list;
        for (auto& r : rt_ids) list += (list.empty() ? "" : ",") + r;
        std::string entry;
        pb::string_field(entry, 1, "NVIDIA_VISIBLE_DEVICES");
        pb::string_field(entry, 2, list.empty() ? "void" : list);
        pb::bytes_field(wire, 1, entry);
    }
    for (auto& s : specs) pb::encode_devspec(wire, 3, s.container_path, s.host_path, s.permissions);
    if (c->kind == b2dp_ctx::CUDA && !c->cdi_kind.empty()) {
        // cdi=<kind>: ContainerAllocateResponse.cdi_devices (field 5, CDIDevice{name=1}) = "<kind>=<uuid|index>", the
        // fully qualified names of an nvidia-ctk generated CDI spec; a CDI-enabled runtime injects from those
        for (auto& r : rt_ids) {
            std::string cdi;
            pb::string_field(cdi, 1, c->cdi_kind + "=" + r);
            pb::bytes_field(wire, 5, cdi);
        }
    }
    *len = wire.size();
    if (wire.size() > cap) return B2DP_E_NOSPC;
    if (!wire.empty() && !buf) return B2DP_E_INVAL;
    memcpy(buf, wire.data(), wire.size());
    return B2DP_OK;
}

// ---- Start / GetPreferredAllocation ------------------------------------------------------
static int ensure_links(b2dp_ctx* c, const std::vector<Device>& devs) {
    if (c->have_links) return B2DP_OK;
    const int n = (int)devs.size();
    std::vector<float> gbs((size_t)n * n);
    std::vector<int32_t> type((size_t)n * n);
    std::vector<uint64_t> mism((size_t)n * n);
    std::string err;
    int rc = cuda_p2p_matrix(c->cuda, nullptr, gbs.data(), type.data(), mism.data(), n, err);
    if (rc != B2DP_OK) return fail(rc, err);
    c->links.clear();
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j)
            if (i != j) c->links.push_back({devs[i].node_id, devs[j].node_id, type[(size_t)i * n + j]});
    c->p2p_gbs = gbs;
    c->have_links = true;
    return B2DP_OK;
}

extern "C" int b2dp_start(b2dp_ctx* c) {
    if (!c) return B2DP_E_INVAL;
    std::vector<Device> devs;
    int rc = enumerate_ctx(c, devs);  // plugin.go:85 getDevices()
    if (rc != B2DP_OK) return rc;
    std::lock_guard<std::mutex> g(c->mu);
    c->policy = std::shared_ptr<BestEffortPolicy>(policy_new(), policy_free);
    if (c->kind == b2dp_ctx::KFD) rc = policy_init_dir(c->policy.get(), devs, go::join(c->sysroot, "sys/class/kfd/kfd/topology/nodes"));
    else {
        rc = ensure_links(c, devs);
        if (rc == B2DP_OK) rc = policy_init_links(c->policy.get(), devs, c->links);
    }
    c->started = true;
    c->allocator_init_error = rc != B2DP_OK;  // plugin.go:86-90
    if (rc != B2DP_OK && t_last_error.empty()) t_last_error = b2dp_strerror(rc);
    return rc;
}

extern "C" int b2dp_pair_weights(b2dp_ctx* c, b2dp_pair_weight* out, int cap, int* n, int* n_rows) {
    if (!c || !n || cap < 0) return B2DP_E_INVAL;
    std::shared_ptr<BestEffortPolicy> p;
    {
        std::lock_guard<std::mutex> g(c->mu);
        p = c->policy;
    }
    if (!p) return fail(B2DP_E_ALLOC_INIT, b2dp_strerror(B2DP_E_ALLOC_INIT));
    std::vector<b2dp_pair_weight> w;
    int rows = 0;
    policy_pair_weights(p.get(), w, &rows);
    *n = (int)w.size();
    if (n_rows) *n_rows = rows;
    if (*n > cap) return B2DP_E_NOSPC;
    if (*n && !out) return B2DP_E_INVAL;
    memcpy(out, w.data(), w.size() * sizeof(b2dp_pair_weight));
    return B2DP_OK;
}

extern "C" int b2dp_preferred_allocation_available(b2dp_ctx* c, int32_t* available) {
    if (!c || !available) return B2DP_E_INVAL;
    std::lock_guard<std::mutex> g(c->mu);
    *available = c->allocator_init_error ? 0 : 1;  // plugin.go:210-217
    return B2DP_OK;
}

extern "C" int b2dp_preferred_allocation(b2dp_ctx* c, const char* const* available, int na,
                                         const char* const* must_include, int nm, int size, char (*out)[64], int cap,
                                         int* n) {
    if (!c || !n || na < 0 || nm < 0 || (na && !available) || (nm && !must_include) || cap < 0) return B2DP_E_INVAL;
    std::shared_ptr<BestEffortPolicy> p;
    {
        std::lock_guard<std::mutex> g(c->mu);
        if (!c->policy) c->policy = std::shared_ptr<BestEffortPolicy>(policy_new(), policy_free);  // Allocate before Start => "Init method must be called"
        p = c->policy;
    }
    std::vector<std::string> a, r, ids;
    for (int i = 0; i < na; ++i) a.emplace_back(available[i] ? available[i] : "");
    for (int i = 0; i < nm; ++i) r.emplace_back(must_include[i] ? must_include[i] : "");
    *n = 0;
    int rc = policy_allocate(p.get(), a, r, size, ids, nullptr, nullptr, false);
    if (rc != B2DP_OK) return fail(rc, std::string("unable to get preferred allocation list. Error:") + b2dp_strerror(rc));
    *n = (int)ids.size();
    if (*n > cap) return B2DP_E_NOSPC;
    if (*n && !out) return B2DP_E_INVAL;
    for (int i = 0; i < *n; ++i) copy_str(out[i], 64, ids[i]);
    return B2DP_OK;
}

// ---- p2p ---------------------------------------------------------------------------------
extern "C" int b2dp_p2p_matrix(b2dp_ctx* c, const b2dp_p2p_opts* opts, float* gbs, int32_t* link_type,
                               uint64_t* mismatches, int n) {
    if (!c || !gbs || !link_type || n <= 0) return B2DP_E_INVAL;
    if (c->kind != b2dp_ctx::CUDA) return fail(B2DP_E_UNSUPPORTED, "the P2P matrix needs the cuda: backend");
    std::vector<Device> devs;
    int rc = enumerate_ctx(c, devs);
    if (rc != B2DP_OK) return rc;
    if ((int)devs.size() != n) return fail(B2DP_E_INVAL, "n must equal the device count");
    std::vector<uint64_t> mism((size_t)n * n);
    std::string err;
    rc = cuda_p2p_matrix(c->cuda, opts, gbs, link_type, mism.data(), n, err);
    if (rc != B2DP_OK) return fail(rc, err);
    if (mismatches) memcpy(mismatches, mism.data(), mism.size() * sizeof(uint64_t));
    std::lock_guard<std::mutex> g(c->mu);
    c->links.clear();
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j)
            if (i != j) c->links.push_back({devs[i].node_id, devs[j].node_id, link_type[(size_t)i * n + j]});
    c->p2p_gbs.assign(gbs, gbs + (size_t)n * n);
    c->have_links = true;
    return B2DP_OK;
}

// ---- labels ------------------------------------------------------------------------------
int b2dp_emit_labels_internal(const std::map<std::string, std::string>& m, b2dp_label* out, int cap, int* n);

extern "C" int b2dp_generate_labels(b2dp_ctx* c, const char* enabled, b2dp_label* out, int cap, int* n) {
    if (!c || !enabled || !n || cap < 0) return B2DP_E_INVAL;
    std::vector<Device> devs;
    int rc = enumerate_ctx(c, devs);  // main.go:385
    if (rc != B2DP_OK) return rc;
    LabelSource src;
    label_source(c, src);
    if (c->kind == b2dp_ctx::CUDA && strstr(enabled, "p2p-link")) {
        // extension label: interconnect class per GPU = the weakest link class to any peer
        std::lock_guard<std::mutex> g(c->mu);
        rc = ensure_links(c, devs);
        if (rc != B2DP_OK) return rc;
        for (const auto& d : devs) {
            int worst = 11, peers = 0;
            for (const auto& l : c->links)
                if (l.from == d.node_id) { ++peers; if (l.type != 11) worst = l.type == 2 && worst != 0 ? 2 : 0; }
            src.p2p_class.push_back(!peers || worst == 0 ? "none" : worst == 2 ? "pcie" : "nvlink");
        }
    }
    std::map<std::string, std::string> m;
    rc = generate_labels(devs, src, enabled, m);
    if (rc != B2DP_OK) return rc;
    return b2dp_emit_labels_internal(m, out, cap, n);
}

// ---- kfd-tree export ---------------------------------------------------------------------
static bool mkdirs(const std::string& p) {
    std::string cur;
    size_t pos = 0;
    while (pos <= p.size()) {
        size_t e = p.find('/', pos);
        if (e == std::string::npos) e = p.size();
        cur = p.substr(0, e);
        pos = e + 1;
        if (cur.empty()) continue;
        if (::mkdir(cur.c_str(), 0755) != 0 && errno != EEXIST) return false;
    }
    return true;
}
static bool write_file(const std::string& path, const std::string& data) {
    if (!mkdirs(go::dir(path))) return false;
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    bool ok = fwrite(data.data(), 1, data.size(), f) == data.size();
    fclose(f);
    return ok;
}

static std::string link_props(int type, int from, int to, int weight) {
    char lp[512];
    snprintf(lp, sizeof lp,
             "type %d\nversion_major 0\nversion_minor 0\nnode_from %d\nnode_to %d\nweight %d\nmin_latency 0\n"
             "max_latency 0\nmin_bandwidth 0\nmax_bandwidth 0\nrecommended_transfer_size 0\nflags 1\n",
             type, from, to, weight);
    return lp;
}

// The node shape of k8s-device-plugin_b200/synth.py:write_b200_tree, file for file (tests compare the two).
static bool write_synthetic_tree(const std::string& root, int n_gpus, int partitions, int n_cpu_nodes,
                                 const std::string& compute, const std::string& memory) {
    const long long vram_bytes = 192265846784LL;
    const int sm_count = 148;
    auto upper = [](std::string v) { for (auto& ch : v) ch = (char)toupper((unsigned char)ch); return v; };
    const std::string nodes = root + "/sys/class/kfd/kfd/topology/nodes";
    bool ok = mkdirs(root + "/sys/devices/platform");
    for (int k = 0; k < n_cpu_nodes; ++k) {
        char props[512];
        snprintf(props, sizeof props,
                 "cpu_cores_count 64\nsimd_count 0\nmem_banks_count 1\ncaches_count 0\nio_links_count 0\n"
                 "cpu_core_id_base %d\nsimd_id_base 0\nvendor_id 0\ndevice_id 0\nlocation_id 0\ndomain 0\n"
                 "drm_render_minor 0\n", k * 64);
        ok &= write_file(nodes + "/" + std::to_string(k) + "/properties", props);
    }
    std::vector<std::pair<int, int>> gpu_nodes;  // (node id, gpu index)
    int node_id = n_cpu_nodes, minor = 128, card = 0;
    for (int g = 0; g < n_gpus; ++g) {
        const int bus = 0x19 + 0x10 * g;
        char bdf[32];
        snprintf(bdf, sizeof bdf, "0000:%02x:00.0", bus);
        const int numa = g < (n_gpus + 1) / 2 ? 0 : 1;
        const std::string pci = root + "/sys/module/amdgpu/drivers/pci:amdgpu/" + bdf;
        ok &= write_file(pci + "/numa_node", std::to_string(numa) + "\n");
        if (!compute.empty()) {
            ok &= write_file(pci + "/current_compute_partition", upper(compute) + "\n");
            ok &= write_file(pci + "/available_compute_partition", "SPX, " + upper(compute) + "\n");
        }
        if (!memory.empty()) {
            ok &= write_file(pci + "/current_memory_partition", upper(memory) + "\n");
            ok &= write_file(pci + "/available_memory_partition", upper(memory) + "\n");
        }
        for (int p = 0; p < partitions; ++p) {
            const std::string base = p == 0 ? pci : root + "/sys/devices/platform/amdgpu_xcp_" + std::to_string(g * 8 + p);
            ok &= mkdirs(base + "/drm/card" + std::to_string(card));
            ok &= mkdirs(base + "/drm/renderD" + std::to_string(minor));
            const std::string drm = root + "/sys/class/drm/card" + std::to_string(card) + "/device";
            ok &= write_file(drm + "/device", "0x2901\n");
            ok &= write_file(drm + "/product_name", "NVIDIA B200\n");
            ok &= write_file(drm + "/driver/module/version", "580.159.03\n");
            ok &= write_file(drm + "/driver/module/srcversion", "SYNTHETIC0000000000000000\n");
            char props[1024];
            snprintf(props, sizeof props,
                     "cpu_cores_count 0\nsimd_count %d\nmem_banks_count 1\ncaches_count 0\nio_links_count %d\n"
                     "cpu_core_id_base 0\nsimd_id_base 0\nmax_waves_per_simd 16\nwave_front_size 32\nsimd_per_cu 4\n"
                     "gfx_target_version 100000\nvendor_id 4318\ndevice_id 10497\nlocation_id %d\ndomain 0\n"
                     "drm_render_minor %d\nlocal_mem_size %lld\n",
                     sm_count * 4 / partitions, n_gpus * partitions - 1, bus << 8, minor, vram_bytes / partitions);
            const std::string nd = nodes + "/" + std::to_string(node_id);
            ok &= write_file(nd + "/properties", props);
            char mb[256];
            snprintf(mb, sizeof mb, "heap_type 1\nsize_in_bytes %lld\nflags 0\nwidth 8192\nmem_clk_max 3996\n", vram_bytes / partitions);
            ok &= write_file(nd + "/mem_banks/0/properties", mb);
            gpu_nodes.push_back({node_id, g});
            ++node_id; ++minor; ++card;
        }
    }
    for (auto& a : gpu_nodes) {
        int li = 0;
        for (auto& b : gpu_nodes) {
            if (b.first == a.first) continue;
            ok &= write_file(nodes + "/" + std::to_string(a.first) + "/io_links/" + std::to_string(li++) + "/properties",
                             link_props(11, a.first, b.first, b.second == a.second ? 13 : 15));
        }
    }
    return ok;
}

static void remove_tree(const std::string& root) {
    std::vector<std::string> names;
    if (go::list_dir_sorted(root, names))
        for (auto& n : names) {
            const std::string p = root + "/" + n;
            struct stat st;
            if (::lstat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode)) remove_tree(p);
            else ::unlink(p.c_str());
        }
    ::rmdir(root.c_str());
}

extern "C" int b2dp_export_kfd_tree(b2dp_ctx* c, const char* dir_c) {
    if (!c || !dir_c || !*dir_c) return B2DP_E_INVAL;
    if (c->kind != b2dp_ctx::CUDA) return fail(B2DP_E_UNSUPPORTED, "export is for the cuda: backend (kfd trees already are one)");
    std::vector<Device> devs;
    int rc = enumerate_ctx(c, devs);
    if (rc != B2DP_OK) return rc;
    {
        std::lock_guard<std::mutex> g(c->mu);
        rc = ensure_links(c, devs);
        if (rc != B2DP_OK) return rc;
    }
    LabelSource src;
    label_source(c, src);
    const std::string dir = dir_c;
    const std::string nodes = dir + "/sys/class/kfd/kfd/topology/nodes";
    int min_node = INT32_MAX;
    for (auto& d : devs) min_node = std::min(min_node, d.node_id);
    if (devs.empty()) min_node = 1;
    bool ok = true;
    // CPU nodes 0 .. min_node-1
    for (int k = 0; k < min_node; ++k)
        ok &= write_file(nodes + "/" + std::to_string(k) + "/properties",
                         "cpu_cores_count 64\nsimd_count 0\nmem_banks_count 1\ncaches_count 0\nio_links_count 0\n"
                         "cpu_core_id_base 0\nsimd_id_base 0\nvendor_id 0\ndevice_id 0\nlocation_id 0\ndomain 0\n"
                         "drm_render_minor 0\n");
    for (size_t i = 0; i < devs.size(); ++i) {
        const Device& d = devs[i];
        unsigned dom = 0, bus = 0, dv = 0;
        sscanf(d.dev_id.c_str(), "%x:%x:%x", &dom, &bus, &dv);
        const long long loc = ((long long)bus << 8) | ((long long)dv << 3);
        const long long sms = i < src.sm_count.size() ? src.sm_count[i] : 0;
        const long long vram = i < src.vram_bytes.size() ? src.vram_bytes[i] : 0;
        std::string devid_hex = i < src.device_id.size() ? src.device_id[i] : "0x0";
        char props[1024];
        snprintf(props, sizeof props,
                 "cpu_cores_count 0\nsimd_count %lld\nmem_banks_count 1\ncaches_count 0\nio_links_count %zu\n"
                 "cpu_core_id_base 0\nsimd_id_base 0\nmax_waves_per_simd 16\nwave_front_size 32\nsimd_per_cu 4\n"
                 "gfx_target_version 100000\nvendor_id 4318\ndevice_id %ld\nlocation_id %lld\ndomain %u\n"
                 "drm_render_minor %d\nlocal_mem_size %lld\n",
                 sms * 4, devs.size() - 1, strtol(devid_hex.c_str(), nullptr, 16), loc, dom, d.render_d, vram);
        const std::string nd = nodes + "/" + std::to_string(d.node_id);
        ok &= write_file(nd + "/properties", props);
        char mb[256];
        snprintf(mb, sizeof mb, "heap_type 1\nsize_in_bytes %lld\nflags 0\nwidth 8192\nmem_clk_max 3996\n", vram);
        ok &= write_file(nd + "/mem_banks/0/properties", mb);
        int li = 0;
        for (const auto& l : c->links) {
            if (l.from != d.node_id) continue;
            char lp[512];
            snprintf(lp, sizeof lp,
                     "type %d\nversion_major 0\nversion_minor 0\nnode_from %d\nnode_to %d\nweight %d\nmin_latency 0\n"
                     "max_latency 0\nmin_bandwidth 0\nmax_bandwidth 0\nrecommended_transfer_size 0\nflags 1\n",
                     l.type, l.from, l.to, l.type == 11 ? 15 : 20);
            ok &= write_file(nd + "/io_links/" + std::to_string(li++) + "/properties", lp);
        }
        // driver dir (amdgpu.go:155-217) + drm class files the label generators read.  A partition other than the
        // first of its GPU is a platform device (amdgpu.go:221-265): no numa_node / partition files of its own, it
        // inherits them from the PCI function with the same devID.
        auto upper = [](std::string v) { for (auto& ch : v) ch = (char)toupper((unsigned char)ch); return v; };
        if (d.id.compare(0, 11, "amdgpu_xcp_") == 0) {
            const std::string plat = dir + "/sys/devices/platform/" + d.id;
            ok &= mkdirs(plat + "/drm/card" + std::to_string(d.card));
            ok &= mkdirs(plat + "/drm/renderD" + std::to_string(d.render_d));
        } else {
            const std::string pci = dir + "/sys/module/amdgpu/drivers/pci:amdgpu/" + d.id;
            ok &= write_file(pci + "/numa_node", std::to_string(d.numa) + "\n");
            ok &= mkdirs(pci + "/drm/card" + std::to_string(d.card));
            ok &= mkdirs(pci + "/drm/renderD" + std::to_string(d.render_d));
            if (!d.compute.empty()) ok &= write_file(pci + "/current_compute_partition", upper(d.compute) + "\n");
            if (!d.memory.empty()) ok &= write_file(pci + "/current_memory_partition", upper(d.memory) + "\n");
            if (src.part_supported[0]) ok &= write_file(pci + "/available_compute_partition", d.compute.empty() ? "SPX\n" : "SPX, " + upper(d.compute) + "\n");
            if (src.part_supported[1]) ok &= write_file(pci + "/available_memory_partition", d.memory.empty() ? "NPS1\n" : upper(d.memory) + "\n");
        }
        const std::string drm = dir + "/sys/class/drm/card" + std::to_string(d.card) + "/device";
        ok &= write_file(drm + "/device", devid_hex + "\n");
        ok &= write_file(drm + "/product_name", (i < src.product_name.size() ? src.product_name[i] : "") + "\n");
        ok &= write_file(drm + "/driver/module/version", src.driver_version + "\n");
        ok &= write_file(drm + "/driver/module/srcversion", src.driver_src_version + "\n");
        // what the reference reads through libdrm ioctls (family, per-block firmware versions) has no sysfs file; the
        // export carries it as two side files the kfd: backend and the oracle's drm provider read back
        if (i < src.family.size() && !src.family[i].empty()) ok &= write_file(drm + "/b2dp_family", src.family[i] + "\n");
        if (i < src.firmware.size() && !src.firmware[i].empty()) {
            std::string fw;
            for (const auto& bv : src.firmware[i]) fw += bv.first + " " + bv.second + "\n";
            ok &= write_file(drm + "/b2dp_firmware", fw);
        }
    }
    ok &= mkdirs(dir + "/sys/devices/platform");
    return ok ? B2DP_OK : fail(B2DP_E_IO, "failed writing the kfd tree under " + dir);
}
