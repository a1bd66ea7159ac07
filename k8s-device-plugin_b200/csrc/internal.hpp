// internal.hpp -- shared internal declarations of libb200dp (not part of the ABI).
#pragma once
#include <cstdint>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200dp.h"

namespace b2dp {

// ---- diagnostics (ctx.cpp): routed to the host's b2dp_set_log_callback, dropped if there is none ----------------
void logf(int level, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
bool log_enabled();

struct Device {
    std::string id, dev_id, compute, memory;
    int card = 0, render_d = 128, node_id = 0, numa = -1;
};

inline void copy_str(char* dst, size_t cap, const std::string& s) {
    size_t n = s.size() < cap - 1 ? s.size() : cap - 1;
    memcpy(dst, s.data(), n);
    dst[n] = 0;
}
inline void to_abi(const Device& d, b2dp_device* o) {
    memset(o, 0, sizeof *o);
    copy_str(o->id, sizeof o->id, d.id);
    copy_str(o->dev_id, sizeof o->dev_id, d.dev_id);
    copy_str(o->compute_partition, sizeof o->compute_partition, d.compute);
    copy_str(o->memory_partition, sizeof o->memory_partition, d.memory);
    o->card = d.card; o->render_d = d.render_d; o->node_id = d.node_id; o->numa_node = d.numa;
}
inline Device from_abi(const b2dp_device& a) {
    Device d;
    d.id = a.id; d.dev_id = a.dev_id; d.compute = a.compute_partition; d.memory = a.memory_partition;
    d.card = a.card; d.render_d = a.render_d; d.node_id = a.node_id; d.numa = a.numa_node;
    return d;
}

// ---- kfd.cpp: sysfs/kfd readers -------------------------------------------------------
struct TopoMaps {
    std::map<int, std::string> dev_ids;  // render minor -> devID   (amdgpu.go:101-146)
    std::map<int, int> node_ids;         // render minor -> node id (amdgpu.go:496-538)
};
void kfd_topology_maps(const std::string& topo_root, TopoMaps& out);
// GetAMDGPUs on <sysroot>; returns B2DP_OK / B2DP_E_NODRIVER / B2DP_E_PANIC. Sorted by id.
int kfd_enumerate(const std::string& sysroot, std::vector<Device>& out, std::string& err);
int kfd_parse_property(const std::string& path, const char* key, int64_t* value);
bool kfd_simple_health_check(const std::string& topo_root);
int kfd_count_gpu_dev(const std::string& topo_root);
bool kfd_partition_supported(const std::string& sysroot, int which);
std::map<std::string, int> partition_histogram(const std::vector<Device>& devs);
// main.go:53-91; returns B2DP_OK or B2DP_E_HETEROGENEOUS / B2DP_E_INVAL.
int resource_list(const std::vector<Device>& devs, const char* strategy, std::vector<std::string>& out);

// ---- allocator.cpp --------------------------------------------------------------------
struct Link { int from, to, type; };
class BestEffortPolicy;
BestEffortPolicy* policy_new();
void policy_free(BestEffortPolicy*);
int policy_init_dir(BestEffortPolicy*, const std::vector<Device>&, const std::string& topo_nodes_dir);
int policy_init_links(BestEffortPolicy*, const std::vector<Device>&, const std::vector<Link>&);
int policy_allocate(BestEffortPolicy*, const std::vector<std::string>& avail, const std::vector<std::string>& req,
                    int size, std::vector<std::string>& out, int* n_candidates, int* best_weight,
                    bool candidates_only);
void policy_pair_weights(BestEffortPolicy*, std::vector<b2dp_pair_weight>& out, int* n_rows);
int policy_group_count(BestEffortPolicy*);
// Pair weights as kfd link files would give them, for the kfd-tree export.
int calculate_pair_weight(const Device& a, const Device& b, int link_type);

// ---- labels.cpp -----------------------------------------------------------------------
struct LabelSource {  // what the generators read; filled by the backend
    std::string sysroot;  // for kfd-style reads
    // cuda backend answers (one entry per enumerated device, same order)
    bool native = false;
    std::vector<std::string> family, product_name, device_id, vbios;
    std::vector<std::vector<std::pair<std::string, std::string>>> firmware;  // per device: (block, version) -- NVML
    std::vector<int64_t> vram_bytes, sm_count;
    std::string driver_version, driver_src_version;
    bool part_supported[2] = {false, false};
    std::vector<std::string> p2p_class;  // per device: "nvlink" | "pcie" | "none" (extension label p2p-link)
};
void create_labels(const std::string& kind, const std::map<std::string, int>& entries,
                   std::map<std::string, std::string>& out);
extern const char* const kGeneratorNames[12];
int generate_labels(const std::vector<Device>& devs, const LabelSource& src, const std::string& enabled_csv,
                    std::map<std::string, std::string>& out);
void remove_old_node_labels(std::map<std::string, std::string>& labels);

// ---- cuda_backend.cu -------------------------------------------------------------------
class CudaBackend;
struct CudaConfig {
    std::vector<int> devices;  // empty = all
    uint64_t bytes = 1ull << 30;
    int slots = 2;                       // ring of probe buffers per GPU (2 = ping-pong; more = scrub window)
    uint64_t p2p_bytes = 256ull << 20;
    float min_gbs = 0.f;                 // absolute GB/s floor (override); 0 = use min_frac of the calibrated ceiling
    float min_frac = 0.8f;               // Healthy needs >= min_frac x gbs_ref (BASELINE.json: ">= 80 % of HBM peak")
    float ref_gbs = 0.f;                 // the ceiling, if the operator pins it; 0 = calibrate at open
    int calib = 3;                       // calibration passes per GPU at open (best kept)
    bool prearm = false;                 // enqueue the next pass behind a doorbell while the current one runs (see cuda_backend.cu)
    int slow_passes = 1;                 // consecutive below-floor passes that make a device Unhealthy (1 = the first one)
    int launchers = 1;                   // 2: a helper thread enqueues the other NUMA node's GPUs in parallel with the caller
    int spin_us = 500;                   // how long the helper keeps spinning after a fan-out / a pre-arm before it sleeps
    bool pin_caller = false;             // pin=1: the fan-out's calling thread is bound to the CPUs local to its GPUs
    int probe_mode = 0;                  // 0 in-process (default), 1 helpers (one child process per unit), 2 off (NVML only)
    bool mig_auto = true;                // mig=auto: a MIG-enabled GPU is listed as its MIG devices (forces helpers for the node)
    uint64_t mig_bytes = 256ull << 20;   // ring slot size on a MIG instance
    int seed_index = -1;                 // helpers: the enumeration index this one-device context stands for (seed schedule)
    std::string passthrough;             // helpers: the probe-related URI options handed on to every child
    std::string sysroot = "/";
    int busy_policy = 0;                 // 0 probe always, 1 skip busy GPUs, 2 shrink on busy GPUs
    uint64_t shrink_bytes = 64ull << 20;
    bool check_ecc = false;
    bool check_xid = false;
    bool compute = false;                // compute=1: every probe pass is followed by the tensor-core check (tc_check.cuh)
    std::vector<int> break_devices;      // test hook: indices (enumeration order) whose per-GPU setup is treated as failed
};
int cuda_backend_open(const CudaConfig& cfg, CudaBackend** out, std::string& err);
void cuda_backend_close(CudaBackend*);
int cuda_enumerate(CudaBackend*, std::vector<Device>& out, std::string& err);
int cuda_node_health(CudaBackend*);
int cuda_probe(CudaBackend*, const b2dp_probe_opts* opts, std::vector<b2dp_probe_result>& out, std::string& err);
int cuda_inject_fault(CudaBackend*, int device, uint64_t word, uint32_t mask, std::string& err);
int cuda_probe_reset(CudaBackend*, int device, std::string& err);
int cuda_probe_peek(CudaBackend*, int device, uint64_t word, uint32_t* out, uint64_t n, std::string& err);
int cuda_p2p_matrix(CudaBackend*, const b2dp_p2p_opts* opts, float* gbs, int32_t* link_type, uint64_t* mism, int n,
                    std::string& err);
int cuda_device_count(CudaBackend*);
void cuda_label_source(CudaBackend*, LabelSource& src);
float cuda_min_gbs(CudaBackend*);
std::string cuda_runtime_id(CudaBackend*, const std::string& id, bool by_index);
int cuda_set_ref(CudaBackend*, int device, float gbs_ref, std::string& err);
void cuda_prearm(CudaBackend*);
int cuda_describe(CudaBackend*, int device, b2dp_probe_info* out, std::string& err);
// device nodes Allocate mounts for `id` beyond the three global ones (whole GPU: /dev/nvidia<minor>; MIG instance:
// the parent's node plus its two /dev/nvidia-caps nodes); false if the id is unknown
bool cuda_device_paths(CudaBackend*, const std::string& id, std::vector<std::string>& out);
// ---- ctx.cpp: what the entry points kept with the CUDA half (compute.cpp) need of a context --------------------------
CudaBackend* ctx_cuda_backend(b2dp_ctx* c);      // nullptr unless c is a cuda: context
int ctx_fail(int code, const std::string& msg);  // record the calling thread's last error text; returns code

// tensor-core check (tc_check.cuh): B2DP_E_UNSUPPORTED in helper / probe=off mode
int cuda_compute_check(CudaBackend*, const b2dp_compute_opts* opts, std::vector<b2dp_compute_result>& out, std::string& err);
int cuda_compute_tile(CudaBackend*, int device, int kind, int a_set, int b_set, float* c, std::string& err);
int cuda_compute_inject_fault(CudaBackend*, int device, int sm, uint32_t mask, std::string& err);
// xid=1: called (from a backend thread, or from b2dp_probe_inject_fault) when a device-level Xid has been latched
void cuda_set_health_event_callback(CudaBackend*, std::function<void()> fn);

}  // namespace b2dp
