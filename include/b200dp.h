/* b200dp.h -- C ABI of libb200dp.so, the B200-native core of the device plugin + node labeller.
 *
 * This is the drop-in boundary for the hot path named in BASELINE.json (enumerate ->
 * health-probe -> property-read, and the topology / pair-weight path behind
 * GetPreferredAllocation).  Each entry point replaces one piece of the reference's
 * in-process Go API (ROCm/k8s-device-plugin @ dea1db13); the reference file:line it
 * replaces is cited above every declaration.  INTEGRATION.md shows the cgo stub a
 * reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 (B2DP_OK) or a negative B2DP_E_* code; nothing aborts,
 *     exits, prints, or installs signal handlers (the reference glog.Fatalf's at
 *     amdgpu.go:150-152; here that is B2DP_E_NODRIVER).
 *   - no callee-owned memory crosses the boundary: the caller passes arrays + capacity,
 *     the callee writes the element count to *n.  If cap is too small the call returns
 *     B2DP_E_NOSPC and *n holds the needed count.
 *   - strings are NUL-terminated, fixed-size char arrays; inputs are plain `const char*`.
 *   - where the reference's result order is Go-map-random, the ABI order is canonical
 *     (sorted by id / key, bytewise) and says so.
 *   - thread safety: every entry point may be called concurrently from arbitrary OS
 *     threads (cgo).  A context owns one worker thread + CUDA stream + pinned result
 *     block + probe buffers per GPU; callers never need a current CUDA device.
 */
#ifndef B200DP_H
#define B200DP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2DP_ABI_VERSION 3
#if defined(__GNUC__)
#define B2DP_API __attribute__((visibility("default")))
#else
#define B2DP_API
#endif

/* ---- error codes ------------------------------------------------------------------ */
enum {
    B2DP_OK = 0,
    B2DP_E_INVAL = -1,        /* bad argument */
    B2DP_E_NOSPC = -2,        /* output capacity too small; *n = needed */
    B2DP_E_IO = -3,           /* open/read failed (Go: os.Open error) */
    B2DP_E_NOTFOUND = -4,     /* "Topology property not found" (amdgpu.go:448) / unknown id */
    B2DP_E_SYNTAX = -5,       /* strconv.ErrSyntax; *value = what Go returns (0) */
    B2DP_E_RANGE = -6,        /* strconv.ErrRange;  *value = clamped value, as Go returns */
    B2DP_E_NODRIVER = -7,     /* driver dir absent: reference glog.Fatalf (amdgpu.go:150-152) */
    B2DP_E_NOGPU = -8,        /* no usable CUDA device / CUDA runtime failed to initialise */
    B2DP_E_CUDA = -9,         /* a CUDA call failed; see b2dp_last_error() */
    B2DP_E_TIMEOUT = -10,     /* probe deadline expired (device reported Unhealthy) */
    B2DP_E_UNSUPPORTED = -11, /* operation not available on this backend */
    B2DP_E_PANIC = -12,       /* the reference would panic here (nil deref / slice bounds) */
    B2DP_E_NOMEM = -13,
    B2DP_E_HETEROGENEOUS = -14, /* main.go:79: heterogeneous node with `single` strategy */
    /* allocator errors; b2dp_strerror() returns the reference's exact strings
       (besteffort_policy.go:36-43, device.go:222,355,359, besteffort_policy.go:73) */
    B2DP_E_ALLOC_SIZE = -20,          /* "allocation size can not be negative" */
    B2DP_E_ALLOC_AVAILABLE = -21,     /* "available devices count less than allocation size" */
    B2DP_E_ALLOC_REQUIRED = -22,      /* "must_include devices size is more than allocation size" */
    B2DP_E_ALLOC_REQ_AVAILABLE = -23, /* "must_include length should be less than or equal to avilable device size" */
    B2DP_E_ALLOC_INIT = -24,          /* "Init method must be called before Allocate" */
    B2DP_E_ALLOC_NOCANDIDATE = -25,   /* "No candidate subset found with matching criteria" */
    B2DP_E_ALLOC_EMPTY_DEVICES = -26, /* "Devices list is empty. Unable to calculate pair wise weights" */
    B2DP_E_ALLOC_NO_WEIGHTS = -27,    /* "Besteffort Policy init failed to initialize p2pWeights" */
    B2DP_E_ALLOC_SUBSET_SIZE = -28,   /* "subset size should be positive integer" */
    B2DP_E_ALLOC_SUBSET_AVAIL = -29   /* "subset size is more than available devices" */
};

/* Diagnostics.  The library never prints (the reference logs through glog, e.g. the warnings of amdgpu.go:171-195 and
 * the health transitions around plugin.go:304-320); a host that wants those lines installs ONE process-wide callback
 * and routes them to its logger.  level: 0 info, 1 warning, 2 error.  `msg` is valid during the call; the callback may
 * run on any library thread and must not call back into the library.  NULL removes it. */
typedef void (*b2dp_log_cb)(void *user, int level, const char *msg);
B2DP_API void b2dp_set_log_callback(b2dp_log_cb cb, void *user);

/* Static message for a code; allocator codes return the reference's error strings. */
B2DP_API const char *b2dp_strerror(int code);
B2DP_API int b2dp_abi_version(void);

/* ---- records ---------------------------------------------------------------------- */
/* One schedulable device.  Replaces the per-device map built at amdgpu.go:216/264
 * {card, renderD, devID, computePartitionType, memoryPartitionType, numaNode, nodeId}
 * and allocator.Device (allocator/device.go:56-65). */
typedef struct b2dp_device {
    char id[64];                /* kubelet Device.ID: PCI BDF dir name or "amdgpu_xcp_N" */
    char dev_id[24];            /* physical-GPU key "%04x:%02x:%02x:0" (amdgpu.go:141) */
    int32_t card;               /* /dev/dri/card<N>     (cuda backend: /dev/nvidia<N>) */
    int32_t render_d;           /* /dev/dri/renderD<N>  (cuda backend: 128 + index)    */
    int32_t node_id;            /* kfd topology node index (amdgpu.go:525-534) */
    int32_t numa_node;
    char compute_partition[16]; /* lower-cased current_compute_partition, "" if absent */
    char memory_partition[16];
} b2dp_device;

typedef struct b2dp_kv_count { char key[64]; int32_t count; } b2dp_kv_count;
typedef struct b2dp_label { char key[160]; char value[96]; } b2dp_label;
typedef struct b2dp_devspec { char host_path[64]; char container_path[64]; char permissions[8]; } b2dp_devspec;
typedef struct b2dp_pair_weight { int32_t node_from, node_to, weight; } b2dp_pair_weight;
typedef struct b2dp_link { int32_t node_from, node_to, type; } b2dp_link; /* type: 11 XGMI/NVLink, 2 PCIe, else other */
typedef struct b2dp_fw_entry { char name[16]; uint32_t feature; uint32_t firmware; } b2dp_fw_entry;

/* ---- stateless kfd/sysfs readers (package internal/pkg/amdgpu + plugin helpers) --- */

/* amdgpu.go:442-463 ParseTopologyProperties(path, regexp `<key>\s(\d+)`): first matching
 * line wins, unanchored match, value = strconv.ParseInt(m[1], 0, 64).
 * B2DP_OK | B2DP_E_IO | B2DP_E_NOTFOUND | B2DP_E_SYNTAX | B2DP_E_RANGE (*value as Go returns). */
B2DP_API int b2dp_parse_topology_property(const char *path, const char *key, int64_t *value);

/* amdgpu.go:101-146 GetDevIdsFromTopology(topoRoot).  topo_root is the directory that holds
 * `topology/nodes` ("/sys/class/kfd/kfd" live).  Output sorted by render minor. */
B2DP_API int b2dp_dev_ids_from_topology(const char *topo_root, int32_t *render_minor, char (*dev_id)[24], int cap, int *n);

/* amdgpu.go:496-538 GetNodeIdsFromTopology(topoRoot).  Output sorted by render minor. */
B2DP_API int b2dp_node_ids_from_topology(const char *topo_root, int32_t *render_minor, int32_t *node_id, int cap, int *n);

/* plugin.go:123-159 countGPUDevFromTopology(topoRoot). */
B2DP_API int b2dp_count_gpu_dev_from_topology(const char *topo_root, int32_t *count);

/* plugin.go:161-206 simpleHealthCheck() with the kfd root injectable. */
B2DP_API int b2dp_simple_health_check(const char *topo_root, int32_t *healthy);

/* amdgpu.go:467-490 parseDebugFSFirmwareInfo(path).  Output sorted by name; a missing file
 * yields n = 0 (the reference logs and returns empty maps). */
B2DP_API int b2dp_parse_debugfs_firmware_info(const char *path, b2dp_fw_entry *out, int cap, int *n);

/* ---- context (one per process / per backend) ------------------------------------- */
typedef struct b2dp_ctx b2dp_ctx;

/* backend_uri:
 *   "kfd:<sysroot>"   parity mode: <sysroot> plays "/" and holds sys/module/amdgpu/drivers,
 *                     sys/class/kfd/kfd/topology, sys/devices/platform/amdgpu_xcp_*; no GPU work.
 *   "synthetic:<N>[,mig=<k>][,compute=<name>][,memory=<name>][,cpus=<c>]"
 *                     a generated kfd-shaped tree of an N x B200 NVSwitch node (k partitions per GPU for the
 *                     MIG/CPX-style layout), opened through the kfd: reader and removed at close; CPU only.
 *   "cuda:[k=v,...]"  real B200s.  keys: devices=0+1+2 (default all), bytes=<S per buffer,
 *                     default 1073741824>, slots=<buffers in the probe ring, default 2 = ping-pong; with M
 *                     slots pass k verifies slot k mod M (written by pass k-1) and re-keys it into slot
 *                     k+1 mod M, so M heartbeats scrub M*S bytes of HBM>,
 *                     min_frac=<Healthy needs achieved GB/s >= min_frac x the device's ceiling, default 0.8 (BASELINE.json:
 *                     "each per-GPU probe >= 80 % of HBM peak"); the ceiling (gbs_ref) is calibrated when the context
 *                     opens: calib=<K, default 3> warm non-advancing passes per GPU, best kept, then the maximum over the
 *                     GPUs of the same product and ring size, so a part that is already slow at start-up is judged
 *                     against its siblings>, ref_gbs=<pin the ceiling instead of calibrating, e.g. the site's measured
 *                     peak>, min_gbs=<absolute GB/s floor, overrides min_frac; default none>, slow_passes=<K consecutive
 *                     below-floor passes make the device Unhealthy, default 1: the first; earlier ones only carry
 *                     B2DP_RES_SLOW -- pass to pass the rate moves by about 1.5 %; integrity faults are never debounced>.  The fractional floor
 *                     applies to rings that stream from HBM (slot >= 128 MiB, above the 126 MB L2); a pass below the floor
 *                     on a GPU that another process is using at that moment (NVML) is flagged B2DP_RES_CONTENDED and judged
 *                     on integrity alone,
 *                     sysroot=<dir for numa_node lookups, default "/">, p2p_bytes=<default 268435456>,
 *                     busy=probe|skip|shrink (what to do on a GPU another process is using; default probe),
 *                     shrink_bytes=<prefix verified by busy=shrink, default 67108864>, ecc=1 (also fail on new
 *                     uncorrected ECC errors or a failed HBM row remapping, two NVML queries per device per pass), xid=1 (also fail a device
 *                     for good once NVML delivers a critical Xid event for it -- application-level Xids 13, 31,
 *                     43, 45, 68, 109 are ignored; a listener thread waits on the NVML event set and, when a
 *                     device-level Xid arrives, every running b2dp_watch loop of the context sends a heartbeat
 *                     cycle at once instead of at its next pulse).
 *                     cdi=<kind> (e.g. cdi=nvidia.com/gpu): Allocate also returns cdi_devices "<kind>=<GPU UUID>";
 *                     id_strategy=uuid|index (default uuid): what NVIDIA_VISIBLE_DEVICES and the CDI names carry -- the
 *                     GPU/MIG UUID or the NVML index (never the /dev/nvidia minor, which the runtime would misread).
 *                     mig=auto|off (default auto): with MIG mode enabled on a GPU (NVML), its MIG devices are enumerated
 *                     instead of the GPU (ids "nvidia_mig_<gpu>_<gi>_<ci>", dev_id of the parent, partition strings
 *                     "<N>g"/"<M>gb") and probed by one helper process per instance.
 *                     probe=inproc|helpers|off (default inproc): helpers = this process never creates a CUDA context; one
 *                     b200dp_probe_helper child per listed unit (found next to libb200dp.so, or B2DP_PROBE_HELPER), started
 *                     with CUDA_VISIBLE_DEVICES=<unit UUID>, runs the same probe and answers over a socketpair; a child that
 *                     dies is reported Unhealthy (B2DP_E_CUDA) and restarted by the next pass; link classes are declared
 *                     from NVML (no cross-process P2P measurement).  off = enumeration / allocation / labels only (NVML,
 *                     no CUDA, no HBM ring: what a labeller needs); the probe entry points return B2DP_E_UNSUPPORTED.
 *                     mig_bytes=<ring slot on a MIG instance, default 268435456>.
 *                     launchers=1|2 (default 1): 2 = a helper thread enqueues the passes of the GPUs on the other NUMA
 *                     node while the caller enqueues its own (spin_us=<how long it keeps spinning after a fan-out or a
 *                     pre-arm, default 500>); measured neutral at 8 GPUs (the driver serialises launches), so off by
 *                     default.  pin=1: bind the calling thread of the fan-out to the CPUs local to its GPUs.
 *                     prearm=0|1 (default 0; B2DP_PREARM in the environment sets the default): while a pass runs the next one
 *                     is enqueued behind cuStreamWaitValue32 on a host-mapped doorbell (a stream wait occupies no SM), and
 *                     the next heartbeat starts it with one host store per GPU instead of a launch: start-of-work latency
 *                     13 us instead of 34 us after seconds of idle (profiles/r02_doorbell_vs_launch.csv).  Passes with
 *                     non-default options, fault repairs, peek/poke/reset, the P2P matrix and close discard ("flush") an
 *                     armed pass: it is rung, waited for and ignored, the ring state does not advance.  CONSTRAINT: while a
 *                     pass is armed, its stream wait stalls all other GPU work THIS PROCESS submits to that GPU (other streams,
 *                     a second context of this library; measured) -- other processes are not affected (a tenant's kernels
 *                     keep their latency).  Use it only where the library is the process's sole user of the GPU (the daemon).
 *                     compute=0|1 (default 0): after every probe pass, each GPU whose HBM pass ran also runs the tensor-core
 *                     check (b2dp_compute_check with default options: tcgen05 bf16 and e4m3 GEMM tiles on every SM, verified
 *                     bit for bit against host hashes); wrong data, a launch failure or a missed deadline makes that pass
 *                     Unhealthy with B2DP_RES_COMPUTE, reported once (the next pass runs fresh).  busy=skip skips it with the
 *                     pass; it travels through probe=helpers.  compute=1 turns prearm=1 off: a check queued behind an armed
 *                     stream wait would stall until the next heartbeat.
 *                     seed_index=<i>: (helpers) the enumeration index this one-device context stands for.
 *                     A GPU whose own setup fails (or that break=<i>+<j>, a test hook, names by enumeration index)
 *                     stays in the device list and is reported Unhealthy with B2DP_E_CUDA on every pass; the open
 *                     only fails when no GPU could be set up.
 *   "nvml:[k=v,...]"  shorthand for "cuda:probe=off,..." (NVML enumeration only).
 * B2DP_E_NODRIVER (kfd: driver dir absent) | B2DP_E_NOGPU | B2DP_E_CUDA | B2DP_E_INVAL. */
B2DP_API int b2dp_open(const char *backend_uri, b2dp_ctx **out);
B2DP_API void b2dp_close(b2dp_ctx *ctx);
/* Last error text recorded on this context by the calling thread's most recent failing call. */
B2DP_API const char *b2dp_last_error(b2dp_ctx *ctx);

/* amdgpu.go:149-268 GetAMDGPUs().  Re-enumerates on every call (like the reference).
 * Canonical order: sorted by id. */
B2DP_API int b2dp_enumerate(b2dp_ctx *ctx, b2dp_device *out, int cap, int *n);

/* amdgpu.go:270-285 UniquePartitionConfigCount(GetAMDGPUs()); sorted by key. */
B2DP_API int b2dp_partition_histogram(b2dp_ctx *ctx, b2dp_kv_count *out, int cap, int *n);
/* amdgpu.go:287-293 IsHomogeneous(). */
B2DP_API int b2dp_is_homogeneous(b2dp_ctx *ctx, int32_t *homogeneous);
/* amdgpu.go:295-328 Is{Compute,Memory}PartitionSupported(): which = 0 compute, 1 memory. */
B2DP_API int b2dp_partition_supported(b2dp_ctx *ctx, int which, int32_t *supported);
/* cmd/k8s-device-plugin/main.go:53-91 getResourceList(strategy): strategy "single"|"mixed"
 * (main.go:42-51 ParseStrategy => B2DP_E_INVAL otherwise).  Sorted.  B2DP_E_HETEROGENEOUS
 * for a heterogeneous node under "single". */
B2DP_API int b2dp_resource_list(b2dp_ctx *ctx, const char *strategy, char (*names)[64], int cap, int *n);

/* plugin.go:161-206 simpleHealthCheck() for this backend: kfd = the text check on
 * <sysroot>/sys/class/kfd/kfd; cuda = driver answers and >= 1 device enumerates. */
B2DP_API int b2dp_node_health(b2dp_ctx *ctx, int32_t *healthy);

/* ---- GPU health probe (replaces the exporter's per-GPU verdict, health.go:42-82) -- */
typedef struct b2dp_probe_opts {
    uint32_t timeout_ms;   /* per-call deadline; 0 = 5000 (the exporter RPC timeout, health.go:37) */
    uint32_t flags;        /* B2DP_PROBE_* */
    float min_gbs;         /* absolute floor: Healthy needs achieved GB/s >= this; 0 = context default (min_frac x gbs_ref) */
    uint32_t grid_ctas;    /* diagnostic hook: launch the pass on this many CTAs instead of the tuned 2 x SMs (emulates a
                              part that lost bandwidth: the data is verified all the same, only slower); 0 = default */
} b2dp_probe_opts;
#define B2DP_PROBE_VARIANT_TMA 0u        /* smem-staged bulk-copy kernel (default) */
#define B2DP_PROBE_VARIANT_R128 1u       /* register-path kernel (for A/B measurement) */
#define B2DP_PROBE_VARIANT_MASK 0xfu
#define B2DP_PROBE_VIA_WORKERS 0x10u     /* launch + wait on each GPU's own worker thread (full isolation from a
                                            wedged driver call) instead of the default low-latency path where the
                                            calling thread enqueues on every stream and polls the pinned result
                                            blocks */
#define B2DP_PROBE_EVENT_TIMING 0x20u    /* also bracket each kernel with CUDA events and report ms_event (what the
                                            roofline is measured with; ~1.5 us more enqueue work per GPU).  Without
                                            it ms_event = 0 and gbs comes from the in-kernel %globaltimer span */

typedef struct b2dp_probe_result {
    int32_t device;             /* index into b2dp_enumerate() order */
    int32_t healthy;            /* 1 Healthy, 0 Unhealthy */
    int32_t err;                /* B2DP_OK | B2DP_E_CUDA | B2DP_E_TIMEOUT */
    uint32_t seed;              /* pattern seed the pass verified */
    uint64_t checksum;          /* sum of all 32-bit words read, mod 2^64 */
    uint64_t expected_checksum; /* closed form for a clean buffer */
    uint64_t mismatches;        /* words != pattern */
    uint64_t first_bad_word;    /* min bad word index, UINT64_MAX if none */
    uint64_t bytes;             /* algorithmic bytes moved: 2 * S */
    float ms_event;             /* CUDA-event time of the probe kernel (B2DP_PROBE_EVENT_TIMING), else 0 */
    float ms_device;            /* %globaltimer span inside the kernel: first CTA start .. result published */
    float gbs;                  /* bytes / ms_event when event-timed, else bytes / ms_device */
    uint32_t flags;             /* B2DP_RES_* */
    float gbs_ref;              /* this device's ceiling: calibrated at open / ref_gbs= / b2dp_probe_set_ref */
    float frac;                 /* (bytes / ms_device) / gbs_ref: the verdict's rate over the ceiling, both on the in-kernel
                                   clock (0 if there is no ceiling) */
    float min_gbs_applied;      /* the floor the verdict used: min_gbs, else min_frac x gbs_ref, else 0 (none) */
    uint32_t reserved;
} b2dp_probe_result;
#define B2DP_RES_SKIPPED_BUSY 0x1u /* busy=skip: another process owns the GPU, no pass ran, the last verdict stands */
#define B2DP_RES_SHRUNK 0x2u       /* busy=shrink: a prefix (shrink_bytes) was verified without re-keying; no GB/s floor */
#define B2DP_RES_ECC 0x4u          /* ecc=1: NVML reports new uncorrected ECC errors since open, or a failed HBM row
                                      remapping (nvmlDeviceGetRemappedRows) => Unhealthy */
#define B2DP_RES_SMALL_RING 0x10u  /* HBM was short when the context opened (e.g. a restart under running pods): the ring
                                      slots on this GPU are smaller than bytes=; `bytes` reports what a pass moved; no GB/s floor */
#define B2DP_RES_CONTENDED 0x20u   /* the pass ran below its GB/s floor while another process was using the GPU (NVML): not a
                                      verdict on the part -- integrity decides alone */
#define B2DP_RES_NO_FLOOR 0x40u    /* no GB/s floor applied: the ring slot is below 128 MiB (a pass out of the L2 says nothing
                                      about HBM) and no absolute min_gbs was given */
#define B2DP_RES_SLOW 0x80u        /* achieved GB/s was below min_gbs_applied */
#define B2DP_RES_PREARMED 0x100u   /* prearm=1: this pass had been enqueued behind its doorbell while the previous one ran; the
                                      heartbeat only rang the doorbell (no launch on its critical path) */
#define B2DP_RES_COMPUTE 0x200u   /* compute=1: the tensor-core check after the pass failed (wrong product, launch failure or missed
                                      deadline) => Unhealthy; not debounced, not sticky */
#define B2DP_RES_XID 0x8u          /* xid=1: a critical Xid event was delivered for this device since open (or the
                                      last b2dp_probe_reset) => Unhealthy, sticky */

/* Replaces the exporter round trip getGPUHealth (exporter/health.go:42-82) and the evidence behind simpleHealthCheck
 * (plugin.go:161-206): launch the probe on every GPU of the context concurrently (one worker thread + stream per
 * GPU; all launched before any is waited on) and collect one result per device. */
B2DP_API int b2dp_probe_health(b2dp_ctx *ctx, const b2dp_probe_opts *opts, b2dp_probe_result *out, int cap, int *n);

/* Test hook (fault injection): XOR `mask` into 32-bit word `word_index` of the buffer the
 * NEXT probe of `device` will read.  word_index == UINT64_MAX instead queues a synthetic critical-Xid
 * event numbered `mask` for `device` (seen by contexts opened with xid=1).  The reference has no equivalent. */
B2DP_API int b2dp_probe_inject_fault(b2dp_ctx *ctx, int device, uint64_t word_index, uint32_t mask);
/* Re-fill the probe buffers of `device` (-1 = all) with a clean pattern; also clears a latched Xid. */
B2DP_API int b2dp_probe_reset(b2dp_ctx *ctx, int device);
/* Set the bandwidth ceiling (gbs_ref) of `device` (-1 = all) the fractional floor refers to, e.g. to the site's measured
 * HBM peak; gbs_ref <= 0 restores the device's own calibration.  Also how tests move a device across the 0.8 line. */
B2DP_API int b2dp_probe_set_ref(b2dp_ctx *ctx, int device, float gbs_ref);
/* What the probe holds on `device` (enumeration index): ring geometry, the calibrated ceiling, and the identity the
 * container runtime knows the device by.  No pass runs. */
typedef struct b2dp_probe_info {
    uint64_t slot_bytes;     /* bytes per ring slot on this device (bytes= unless HBM was short at open) */
    uint64_t total_memory;   /* device (or MIG instance) memory in bytes */
    int32_t sm_count;
    int32_t slots;
    float gbs_cal;           /* best calibration pass of this device */
    float gbs_ref;           /* the ceiling in force (sibling maximum / ref_gbs= / b2dp_probe_set_ref) */
    int32_t usable;          /* 0: the device could not be set up (listed, always Unhealthy) */
    int32_t via_helper;      /* 1: probed by a b200dp_probe_helper child (probe=helpers, MIG) */
    char uuid[48];           /* "GPU-..." / "MIG-..." */
    char name[64];           /* product name */
} b2dp_probe_info;
B2DP_API int b2dp_probe_describe(b2dp_ctx *ctx, int device, b2dp_probe_info *out);
/* Closed-form checksum of a clean probe buffer of n_words 32-bit words keyed with `seed`, computed on the host
 * (the value b2dp_probe_result.expected_checksum carries).  No context, no GPU. */
B2DP_API int b2dp_expected_checksum(uint64_t n_words, uint32_t seed, uint64_t *checksum);
/* Copy `n_words` words starting at `word_index` of the buffer the next probe will read
 * (parity tests compare it with the oracle's pattern). */
B2DP_API int b2dp_probe_peek(b2dp_ctx *ctx, int device, uint64_t word_index, uint32_t *out, uint64_t n_words);

/* ---- tensor-core check (extends the per-GPU verdict of exporter/health.go:42-82) ----------------------------------
 * One CTA per SM runs T tiles of M=128 N=128 K=128 on the tensor cores (tcgen05.mma, fp32 accumulators in tensor
 * memory) for each of two kinds, back to back: kind::f16 with bf16 operands (kind 0) and kind::f8f6f4 with e4m3
 * operands (kind 1).  Operands are integers in [-7, 7] from a per-device seed, so every product is exact; each
 * accumulator row is hashed on the device and compared with the hash the host computed at open. */
typedef struct b2dp_compute_opts {
    uint32_t timeout_ms;   /* 0 = 5000 */
    uint32_t tiles;        /* tiles per CTA per kind; 0 = the default (B2DP_COMPUTE_DEFAULT_TILES) */
    uint32_t flags;        /* B2DP_COMPUTE_EVENT_TIMING */
    uint32_t reserved;
} b2dp_compute_opts;
#define B2DP_COMPUTE_EVENT_TIMING 0x20u   /* also bracket the two launches with CUDA events and report ms_event */
#define B2DP_COMPUTE_DEFAULT_TILES 8u
#define B2DP_COMPUTE_MAX_TILES 65536u

typedef struct b2dp_compute_result {
    int32_t device;             /* index into b2dp_enumerate() order */
    int32_t healthy;            /* 1: every row of every tile matched */
    int32_t err;                /* B2DP_OK | B2DP_E_CUDA (launch failed / no sequence echo) | B2DP_E_TIMEOUT */
    uint32_t seed;              /* operand pool seed of this device */
    int32_t sms;                /* SMs of the device */
    int32_t sms_covered;        /* SMs that ran a CTA of both kinds (a tenant may hold some: reported, not a verdict) */
    int32_t sms_failed;         /* SMs with at least one bad row */
    int32_t first_bad_sm;       /* lowest %smid with a bad row, -1 if none */
    int32_t first_bad_kind;     /* on first_bad_sm: 0 bf16, 1 e4m3; -1 if none */
    int32_t first_bad_tile;     /* on first_bad_sm, in that kind: the first tile with a bad row; -1 if none */
    int32_t first_bad_row;      /* its first bad row; -1 if none */
    uint32_t reserved0;
    uint64_t tiles;             /* tiles verified over both kinds and all SMs */
    uint64_t bad_rows;          /* accumulator rows whose hash did not match */
    uint32_t bad_sm_mask[8];    /* bit s (word s / 32) = %smid s had a bad row */
    uint32_t covered_mask[8];   /* bit s = %smid s ran a CTA of both kinds */
    float ms_device;            /* %globaltimer span: first CTA start .. result published */
    float ms_event;             /* CUDA-event time of both launches (B2DP_COMPUTE_EVENT_TIMING), else 0 */
    float tflops;               /* 2*128*128*128 * tiles over ms_event if timed, else over ms_device (reported, not judged) */
    uint32_t reserved1;
} b2dp_compute_result;

/* exporter/health.go:42-82 (the per-GPU verdict) and the heartbeat that carries it, plugin.go:304-320: run the
 * tensor-core check on every GPU of the context concurrently and return per-SM detail.  Works whether or not the
 * context was opened with compute=1.  A device that could not be set up gets err = B2DP_E_CUDA and is not launched on.
 * B2DP_E_UNSUPPORTED on kfd:, synthetic:, probe=off and probe=helpers (MIG) contexts. */
B2DP_API int b2dp_compute_check(b2dp_ctx *ctx, const b2dp_compute_opts *opts, b2dp_compute_result *out, int cap, int *n);
/* Bit-exact parity hook for the verdict of exporter/health.go:42-82: one CTA computes one tile C = A[a_set] . B[b_set]^T
 * of `kind` (0 bf16, 1 e4m3) from the device's pool and returns the raw fp32 accumulator, row-major [128][128]. */
B2DP_API int b2dp_compute_tile(b2dp_ctx *ctx, int device, int kind, int a_set, int b_set, float *c);
/* Test hook for the verdict of exporter/health.go:42-82, as b2dp_probe_inject_fault: in the next check on `device`
 * (b2dp_compute_check or a compute=1 pass) the CTA on %smid `sm` XORs `mask` into row 0, column 0 of its first bf16
 * tile after reading it from tensor memory -- a simulated wrong product, no GPU fault.  One-shot. */
B2DP_API int b2dp_compute_inject_fault(b2dp_ctx *ctx, int device, int sm, uint32_t mask);
/* The host reference behind the verdict of exporter/health.go:42-82: the 128 row hashes of tile (a_set, b_set) of
 * `kind` for pool `seed` (oracle/tc_check.py).  No context, no GPU.  cap >= 128. */
B2DP_API int b2dp_compute_expected(uint32_t seed, int kind, int a_set, int b_set, uint64_t *row_hash, int cap, int *n);

/* exporter/health.go:86-106 PopulatePerGPUDHealth(devs, defaultHealth) merge rule.
 * have_source = 0 reproduces "exporter socket absent / RPC failed" (every device gets the
 * default).  src_health[j] follows health.go:74-80: 1 iff the exporter said exactly "healthy". */
B2DP_API int b2dp_merge_health(const char (*ids)[64], int n, int32_t default_healthy, int have_source,
                      const char (*src_ids)[64], const int32_t *src_health, int m, int32_t *out_healthy);

/* ---- ListAndWatch (plugin.go:229-330) --------------------------------------------- */
typedef struct b2dp_cycle_opts {
    uint32_t flags;                /* B2DP_LW_* */
    b2dp_probe_opts probe;
    /* optional external per-device health source merged like health.go:86-106
       (ignored unless B2DP_LW_EXTERNAL_SOURCE) */
    const char (*src_ids)[64];
    const int32_t *src_health;
    int32_t src_n;
    int32_t reserved;
} b2dp_cycle_opts;
#define B2DP_LW_INITIAL 0x1u         /* stream start: enumerate, every device "Healthy" (plugin.go:231-299) */
#define B2DP_LW_HEARTBEAT 0x2u       /* heartbeat tick: node health + per-device health + re-send (plugin.go:304-320);
                                        reuses the device list of the last INITIAL call (the reference builds the
                                        list once per stream), enumerating only if there has been none */
#define B2DP_LW_EXTERNAL_SOURCE 0x4u /* merge src_* instead of running the GPU probe */
#define B2DP_LW_NO_PROBE 0x8u        /* heartbeat without a per-device source: default health only */
#define B2DP_LW_LINK_CHECK 0x10u     /* heartbeat also re-measures the NVLink P2P matrix (64 MiB per directed pair,
                                        both directions at once, ~10 ms on 8 GPUs): a device with a corrupting link or a
                                        link that fell out of its measured class is reported Unhealthy */

typedef struct b2dp_cycle_stats {
    int32_t n_devices;        /* devices in the response */
    int32_t n_unhealthy;
    int32_t homogeneous;
    int32_t node_healthy;     /* simpleHealthCheck result (heartbeat) */
    float ms_total;           /* wall clock of the call */
    float ms_enumerate;
    float ms_probe;           /* launch-all .. last result */
    float ms_encode;
    float probe_gbs_min;      /* over devices, 0 if no probe ran */
    float probe_gbs_sum;
    uint64_t probe_bytes;     /* algorithmic bytes over all devices */
    float ms_link_check;      /* B2DP_LW_LINK_CHECK: time of the P2P matrix */
    int32_t n_link_faults;    /* directed pairs that failed the link check */
    float probe_ms_device_max; /* slowest device's in-kernel span (first CTA start .. result published) this cycle */
    float probe_frac_min;     /* min over devices of gbs / gbs_ref, 0 if no probe ran or no ceiling */
} b2dp_cycle_stats;

/* One ListAndWatch send.  Writes the serialized v1beta1.ListAndWatchResponse protobuf
 * (api.proto: devices[]{ID=1, health=2, topology=3{nodes=1[]{ID=1}}}) for `resource`
 * ("gpu" or a "<compute>_<memory>" partition name, plugin.go:296) into buf.  Devices are in
 * canonical order (sorted by ID).  On a heterogeneous node with no devices of `resource`
 * nothing is sent by the reference (plugin.go:296-298): *len = 0 and n_devices = 0. */
B2DP_API int b2dp_list_and_watch(b2dp_ctx *ctx, const char *resource, const b2dp_cycle_opts *opts, uint8_t *buf, size_t cap,
                        size_t *len, b2dp_cycle_stats *stats);

/* The ListAndWatch loop itself, owned by the library (plugin.go:229-330 + the `-pulse` ticker of
 * cmd/k8s-device-plugin/main.go:129-137): a thread sends the initial list, then one heartbeat cycle per
 * tick -- every pulse_ms (0 = no ticker) and on every b2dp_watch_beat() (the reference's
 * `l.Heartbeat <- true`) -- until b2dp_watch_stop() (the reference's p.signal).  Each send invokes
 * `cb(user, rc, buf, len, stats)` on that thread with the serialized ListAndWatchResponse (valid
 * during the call); rc != 0 reports a failed cycle.  `opts` as for b2dp_list_and_watch (the
 * INITIAL/HEARTBEAT bits are set by the loop).  b2dp_watch_stop() joins that thread (called from the callback
 * itself it only marks the loop to end, and the loop frees the handle on its way out); b2dp_watch_beat() may be
 * called from anywhere, the callback included.  Stop every
 * watch of a context before b2dp_close(). */
typedef void (*b2dp_watch_cb)(void *user, int rc, const uint8_t *buf, size_t len, const b2dp_cycle_stats *stats);
typedef struct b2dp_watch b2dp_watch;
B2DP_API int b2dp_watch_start(b2dp_ctx *ctx, const char *resource, uint32_t pulse_ms, const b2dp_cycle_opts *opts,
                     b2dp_watch_cb cb, void *user, b2dp_watch **out);
B2DP_API int b2dp_watch_beat(b2dp_watch *w);
B2DP_API void b2dp_watch_stop(b2dp_watch *w);

/* plugin.go:356-393 Allocate for one container request: "/dev/kfd" first, then the two
 * /dev/dri paths of every known id (card, then renderD); unknown ids add nothing.  "Known" = the device
 * table of this context's last INITIAL ListAndWatch (the reference reads p.AMDGPUs, plugin.go:231,375);
 * a context that has not streamed yet enumerates instead (the reference would know no id at all).
 * cuda backend: /dev/nvidiactl, /dev/nvidia-uvm, /dev/nvidia-uvm-tools, then /dev/nvidia<minor>. */
B2DP_API int b2dp_device_specs(b2dp_ctx *ctx, const char *const *ids, int n_ids, b2dp_devspec *out, int cap, int *n);
/* Same, serialized as v1beta1.ContainerAllocateResponse (api.proto: devices=3).  The cuda backend also sets
 * envs["NVIDIA_VISIBLE_DEVICES"] = the allocated GPU (or MIG) UUIDs -- NVML indices with id_strategy=index; "void" if
 * none -- and, with the cdi=<kind> URI option, cdi_devices (field 5) "<kind>=<same identifier>"; the kfd backend sets
 * neither, like the reference. */
B2DP_API int b2dp_allocate_response(b2dp_ctx *ctx, const char *const *ids, int n_ids, uint8_t *buf, size_t cap, size_t *len);

/* ---- allocator (internal/pkg/allocator) ------------------------------------------ */
typedef struct b2dp_allocator b2dp_allocator;

/* besteffort_policy.go:52-59 NewBestEffortPolicy(). */
B2DP_API int b2dp_allocator_new(b2dp_allocator **out);
B2DP_API void b2dp_allocator_free(b2dp_allocator *a);
/* besteffort_policy.go:70-86 Init(devs, topoDir): pair weights from the kfd io_links/p2p_links
 * files under topo_nodes_dir ("" = /sys/class/kfd/kfd/topology/nodes, device.go:34).
 * B2DP_E_ALLOC_EMPTY_DEVICES | B2DP_E_ALLOC_NO_WEIGHTS. */
B2DP_API int b2dp_allocator_init(b2dp_allocator *a, const b2dp_device *devs, int n, const char *topo_nodes_dir);
/* Same Init, with the link list measured by b2dp_p2p_matrix() instead of sysfs files
 * (links are applied in order; later entries overwrite earlier ones like device.go:214). */
B2DP_API int b2dp_allocator_init_links(b2dp_allocator *a, const b2dp_device *devs, int n, const b2dp_link *links, int n_links);
/* device.go:220-252 result: p2pWeights as (from < to, weight) rows sorted by (from, to);
 * *n_rows = number of distinct `from` keys (len(p2pWeights), device_test.go:105). */
B2DP_API int b2dp_allocator_pair_weights(b2dp_allocator *a, b2dp_pair_weight *out, int cap, int *n, int *n_rows);
/* device.go:287-304: number of physical-GPU groups. */
B2DP_API int b2dp_allocator_group_count(b2dp_allocator *a, int32_t *groups);
/* device.go:353-442 getCandidateDeviceSubsets(available, required, size): candidate count and
 * the winning (strictly smallest, first wins) total weight. */
B2DP_API int b2dp_allocator_candidates(b2dp_allocator *a, const char *const *available, int na, const char *const *required,
                              int nr, int size, int32_t *n_candidates, int32_t *best_weight);
/* besteffort_policy.go:88-151 Allocate(availableIds, requiredIds, size).  Output ids in the
 * reference's order (subset insertion order; the caller's own order on the two shortcuts). */
B2DP_API int b2dp_allocator_allocate(b2dp_allocator *a, const char *const *available, int na, const char *const *required,
                            int nr, int size, char (*out)[64], int cap, int *n);

/* plugin.go:82-91 Start(): build the context's own allocator from b2dp_enumerate() and the
 * backend's topology (kfd: sysfs link files; cuda: the measured P2P matrix, running it if
 * it has not run yet).  A failure is remembered like allocatorInitError (plugin.go:86-90). */
B2DP_API int b2dp_start(b2dp_ctx *ctx);
/* device.go:220-252 p2pWeights of the context's own allocator (the one b2dp_start() built; cuda: from the measured
 * P2P matrix), same row format as b2dp_allocator_pair_weights.  B2DP_E_ALLOC_INIT before b2dp_start(). */
B2DP_API int b2dp_pair_weights(b2dp_ctx *ctx, b2dp_pair_weight *out, int cap, int *n, int *n_rows);
/* plugin.go:210-217 GetDevicePluginOptions: 1 unless Start() failed. */
B2DP_API int b2dp_preferred_allocation_available(b2dp_ctx *ctx, int32_t *available);
/* plugin.go:337-351 GetPreferredAllocation for one container request. */
B2DP_API int b2dp_preferred_allocation(b2dp_ctx *ctx, const char *const *available, int na, const char *const *must_include,
                              int nm, int size, char (*out)[64], int cap, int *n);

/* ---- NVLink / P2P topology (replaces the kfd link `type` read, device.go:143-149) -- */
typedef struct b2dp_p2p_opts {
    uint64_t bytes;      /* per directed pair; 0 = context default (256 MiB) */
    uint32_t iters;      /* timed repetitions per pair, best kept; 0 = 2 */
    uint32_t flags;      /* B2DP_P2P_* */
} b2dp_p2p_opts;
#define B2DP_P2P_BIDIR 0x1u /* run both directions of a pair concurrently (default: one direction at a time) */
/* For every ordered pair (i != j) a kernel on GPU i pulls a peer-mapped buffer on GPU j over
 * NVLink (bulk copies into shared memory) into local HBM, verifying the pattern on receipt;
 * pairs run in N-1 rounds of disjoint matchings, one direction per half-round.  gbs and link_type are N x N row-major ([i*N + j]: i reads from j);
 * diagonal = local HBM copy GB/s and type 0.  link_type: 11 NVLink-class, 2 PCIe-class,
 * 0 no peer access (oracle/probe.py classify_link).  `n` must equal the device count. */
B2DP_API int b2dp_p2p_matrix(b2dp_ctx *ctx, const b2dp_p2p_opts *opts, float *gbs, int32_t *link_type, uint64_t *mismatches, int n);

/* Write the context's view of the node as a kfd-shaped sysfs tree under `dir` (topology
 * nodes with properties + io_links, pci:amdgpu driver dirs with numa_node and drm/).  The
 * reference algorithm (the oracle) pointed at that tree must reproduce b2dp_enumerate(),
 * b2dp_allocator_pair_weights() and the label set of this context: the "equivalent
 * fixture" of BASELINE.json. */
B2DP_API int b2dp_export_kfd_tree(b2dp_ctx *ctx, const char *dir);

/* ---- node labeller (cmd/k8s-node-labeller/main.go) -------------------------------- */
/* main.go:37-40: the label/resource domain, "amd.com" (and "beta.amd.com") in the reference and by
 * default here.  Process-wide; set once at start-up to publish under another vendor domain. */
B2DP_API int b2dp_set_vendor_domain(const char *domain);
/* main.go:87-108 createLabels(kind, entries).  Output sorted by key. */
B2DP_API int b2dp_create_labels(const char *kind, const b2dp_kv_count *entries, int n_entries, b2dp_label *out, int cap, int *n);
/* main.go:46-53 initLabelLists: the 12 generator names, sorted ("compute-memory-partition", ...). */
B2DP_API int b2dp_label_generator_names(char (*names)[64], int cap, int *n);
/* main.go:383-397 generateLabels(): `enabled` = comma-separated generator names
 * (the labeller's bool flags, main.go:407-409).  Output sorted by key. */
B2DP_API int b2dp_generate_labels(b2dp_ctx *ctx, const char *enabled, b2dp_label *out, int cap, int *n);
/* main.go:55-74 removeOldNodeLabels on a label array: compacts `labels` in place, *n = kept. */
B2DP_API int b2dp_remove_old_node_labels(b2dp_label *labels, int n_in, int *n);

#ifdef __cplusplus
}
#endif
#endif /* B200DP_H */
