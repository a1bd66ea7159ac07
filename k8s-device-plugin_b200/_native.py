"""ctypes binding of libb200dp.so (include/b200dp.h).

The library is built in-tree by `build()` (nvcc, sm_100a) and loaded from the package
directory.  There is no Python/CPU fallback: if the shared object is missing or fails to
load, importing this module raises.
"""
import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libb200dp.so")
CSRC = os.path.join(_PKG, "csrc")


def build(verbose: bool = False) -> str:
    """Compile libb200dp.so for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j", str(min(8, os.cpu_count() or 1))]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("building libb200dp.so failed (see output above)")
    return LIB_PATH


# ---- error codes (b200dp.h) ---------------------------------------------------------------
OK = 0
E_INVAL, E_NOSPC, E_IO, E_NOTFOUND, E_SYNTAX, E_RANGE, E_NODRIVER = -1, -2, -3, -4, -5, -6, -7
E_NOGPU, E_CUDA, E_TIMEOUT, E_UNSUPPORTED, E_PANIC, E_NOMEM, E_HETEROGENEOUS = -8, -9, -10, -11, -12, -13, -14
E_ALLOC_SIZE, E_ALLOC_AVAILABLE, E_ALLOC_REQUIRED, E_ALLOC_REQ_AVAILABLE = -20, -21, -22, -23
E_ALLOC_INIT, E_ALLOC_NOCANDIDATE, E_ALLOC_EMPTY_DEVICES, E_ALLOC_NO_WEIGHTS = -24, -25, -26, -27
E_ALLOC_SUBSET_SIZE, E_ALLOC_SUBSET_AVAIL = -28, -29

PROBE_VARIANT_TMA, PROBE_VARIANT_R128 = 0, 1
PROBE_VIA_WORKERS = 0x10
PROBE_EVENT_TIMING = 0x20
RES_SKIPPED_BUSY, RES_SHRUNK, RES_ECC, RES_XID, RES_SMALL_RING = 1, 2, 4, 8, 16
RES_CONTENDED, RES_NO_FLOOR, RES_SLOW, RES_PREARMED = 0x20, 0x40, 0x80, 0x100
RES_COMPUTE = 0x200
COMPUTE_EVENT_TIMING = 0x20
COMPUTE_DEFAULT_TILES, COMPUTE_MAX_TILES = 8, 65536
COMPUTE_KIND_BF16, COMPUTE_KIND_E4M3 = 0, 1
LW_INITIAL, LW_HEARTBEAT, LW_EXTERNAL_SOURCE, LW_NO_PROBE, LW_LINK_CHECK = 1, 2, 4, 8, 16

Id64 = C.c_char * 64


class Device(C.Structure):
    _fields_ = [("id", C.c_char * 64), ("dev_id", C.c_char * 24), ("card", C.c_int32), ("render_d", C.c_int32),
                ("node_id", C.c_int32), ("numa_node", C.c_int32), ("compute_partition", C.c_char * 16),
                ("memory_partition", C.c_char * 16)]


class KvCount(C.Structure):
    _fields_ = [("key", C.c_char * 64), ("count", C.c_int32)]


class Label(C.Structure):
    _fields_ = [("key", C.c_char * 160), ("value", C.c_char * 96)]


class DevSpec(C.Structure):
    _fields_ = [("host_path", C.c_char * 64), ("container_path", C.c_char * 64), ("permissions", C.c_char * 8)]


class PairWeight(C.Structure):
    _fields_ = [("node_from", C.c_int32), ("node_to", C.c_int32), ("weight", C.c_int32)]


class Link(C.Structure):
    _fields_ = [("node_from", C.c_int32), ("node_to", C.c_int32), ("type", C.c_int32)]


class FwEntry(C.Structure):
    _fields_ = [("name", C.c_char * 16), ("feature", C.c_uint32), ("firmware", C.c_uint32)]


class ProbeOpts(C.Structure):
    _fields_ = [("timeout_ms", C.c_uint32), ("flags", C.c_uint32), ("min_gbs", C.c_float), ("grid_ctas", C.c_uint32)]


class ProbeResult(C.Structure):
    _fields_ = [("device", C.c_int32), ("healthy", C.c_int32), ("err", C.c_int32), ("seed", C.c_uint32),
                ("checksum", C.c_uint64), ("expected_checksum", C.c_uint64), ("mismatches", C.c_uint64),
                ("first_bad_word", C.c_uint64), ("bytes", C.c_uint64), ("ms_event", C.c_float),
                ("ms_device", C.c_float), ("gbs", C.c_float), ("flags", C.c_uint32), ("gbs_ref", C.c_float),
                ("frac", C.c_float), ("min_gbs_applied", C.c_float), ("reserved", C.c_uint32)]


class CycleOpts(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("probe", ProbeOpts), ("src_ids", C.POINTER(Id64)),
                ("src_health", C.POINTER(C.c_int32)), ("src_n", C.c_int32), ("reserved", C.c_int32)]


class CycleStats(C.Structure):
    _fields_ = [("n_devices", C.c_int32), ("n_unhealthy", C.c_int32), ("homogeneous", C.c_int32),
                ("node_healthy", C.c_int32), ("ms_total", C.c_float), ("ms_enumerate", C.c_float),
                ("ms_probe", C.c_float), ("ms_encode", C.c_float), ("probe_gbs_min", C.c_float),
                ("probe_gbs_sum", C.c_float), ("probe_bytes", C.c_uint64), ("ms_link_check", C.c_float),
                ("n_link_faults", C.c_int32), ("probe_ms_device_max", C.c_float), ("probe_frac_min", C.c_float)]


class ProbeInfo(C.Structure):
    _fields_ = [("slot_bytes", C.c_uint64), ("total_memory", C.c_uint64), ("sm_count", C.c_int32), ("slots", C.c_int32),
                ("gbs_cal", C.c_float), ("gbs_ref", C.c_float), ("usable", C.c_int32), ("via_helper", C.c_int32),
                ("uuid", C.c_char * 48), ("name", C.c_char * 64)]


class ComputeOpts(C.Structure):
    _fields_ = [("timeout_ms", C.c_uint32), ("tiles", C.c_uint32), ("flags", C.c_uint32), ("reserved", C.c_uint32)]


class ComputeResult(C.Structure):
    _fields_ = [("device", C.c_int32), ("healthy", C.c_int32), ("err", C.c_int32), ("seed", C.c_uint32),
                ("sms", C.c_int32), ("sms_covered", C.c_int32), ("sms_failed", C.c_int32), ("first_bad_sm", C.c_int32),
                ("first_bad_kind", C.c_int32), ("first_bad_tile", C.c_int32), ("first_bad_row", C.c_int32),
                ("reserved0", C.c_uint32), ("tiles", C.c_uint64), ("bad_rows", C.c_uint64),
                ("bad_sm_mask", C.c_uint32 * 8), ("covered_mask", C.c_uint32 * 8), ("ms_device", C.c_float),
                ("ms_event", C.c_float), ("tflops", C.c_float), ("reserved1", C.c_uint32)]


class P2pOpts(C.Structure):
    _fields_ = [("bytes", C.c_uint64), ("iters", C.c_uint32), ("flags", C.c_uint32)]


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "libb200dp.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
        "(or `make -C k8s-device-plugin_b200/csrc`). There is no CPU fallback.")
lib = C.CDLL(LIB_PATH)

WatchCb = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.c_size_t, C.POINTER(CycleStats))
LogCb = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_char_p)

_P = C.POINTER
_vp, _cp, _i, _ip = C.c_void_p, C.c_char_p, C.c_int, _P(C.c_int)
_i32p, _u8p, _szp = _P(C.c_int32), _P(C.c_uint8), _P(C.c_size_t)
_strs = _P(C.c_char_p)

# name -> (restype, argtypes); every function b200dp.h declares
SIGNATURES = {
    "b2dp_set_log_callback": (None, [LogCb, _vp]),
    "b2dp_strerror": (C.c_char_p, [_i]),
    "b2dp_abi_version": (_i, []),
    "b2dp_parse_topology_property": (_i, [_cp, _cp, _P(C.c_int64)]),
    "b2dp_dev_ids_from_topology": (_i, [_cp, _i32p, _P(C.c_char * 24), _i, _ip]),
    "b2dp_node_ids_from_topology": (_i, [_cp, _i32p, _i32p, _i, _ip]),
    "b2dp_count_gpu_dev_from_topology": (_i, [_cp, _i32p]),
    "b2dp_simple_health_check": (_i, [_cp, _i32p]),
    "b2dp_parse_debugfs_firmware_info": (_i, [_cp, _P(FwEntry), _i, _ip]),
    "b2dp_open": (_i, [_cp, _P(_vp)]),
    "b2dp_close": (None, [_vp]),
    "b2dp_last_error": (C.c_char_p, [_vp]),
    "b2dp_enumerate": (_i, [_vp, _P(Device), _i, _ip]),
    "b2dp_partition_histogram": (_i, [_vp, _P(KvCount), _i, _ip]),
    "b2dp_is_homogeneous": (_i, [_vp, _i32p]),
    "b2dp_partition_supported": (_i, [_vp, _i, _i32p]),
    "b2dp_resource_list": (_i, [_vp, _cp, _P(Id64), _i, _ip]),
    "b2dp_node_health": (_i, [_vp, _i32p]),
    "b2dp_probe_health": (_i, [_vp, _P(ProbeOpts), _P(ProbeResult), _i, _ip]),
    "b2dp_probe_inject_fault": (_i, [_vp, _i, C.c_uint64, C.c_uint32]),
    "b2dp_probe_reset": (_i, [_vp, _i]),
    "b2dp_probe_peek": (_i, [_vp, _i, C.c_uint64, _P(C.c_uint32), C.c_uint64]),
    "b2dp_probe_set_ref": (_i, [_vp, _i, C.c_float]),
    "b2dp_probe_describe": (_i, [_vp, _i, _P(ProbeInfo)]),
    "b2dp_expected_checksum": (_i, [C.c_uint64, C.c_uint32, _P(C.c_uint64)]),
    "b2dp_compute_check": (_i, [_vp, _P(ComputeOpts), _P(ComputeResult), _i, _ip]),
    "b2dp_compute_tile": (_i, [_vp, _i, _i, _i, _i, _P(C.c_float)]),
    "b2dp_compute_inject_fault": (_i, [_vp, _i, _i, C.c_uint32]),
    "b2dp_compute_expected": (_i, [C.c_uint32, _i, _i, _i, _P(C.c_uint64), _i, _ip]),
    "b2dp_merge_health": (_i, [_P(Id64), _i, C.c_int32, _i, _P(Id64), _i32p, _i, _i32p]),
    "b2dp_list_and_watch": (_i, [_vp, _cp, _P(CycleOpts), _u8p, C.c_size_t, _szp, _P(CycleStats)]),
    "b2dp_watch_start": (_i, [_vp, _cp, C.c_uint32, _P(CycleOpts), WatchCb, _vp, _P(_vp)]),
    "b2dp_watch_beat": (_i, [_vp]),
    "b2dp_watch_stop": (None, [_vp]),
    "b2dp_device_specs": (_i, [_vp, _strs, _i, _P(DevSpec), _i, _ip]),
    "b2dp_allocate_response": (_i, [_vp, _strs, _i, _u8p, C.c_size_t, _szp]),
    "b2dp_allocator_new": (_i, [_P(_vp)]),
    "b2dp_allocator_free": (None, [_vp]),
    "b2dp_allocator_init": (_i, [_vp, _P(Device), _i, _cp]),
    "b2dp_allocator_init_links": (_i, [_vp, _P(Device), _i, _P(Link), _i]),
    "b2dp_allocator_pair_weights": (_i, [_vp, _P(PairWeight), _i, _ip, _ip]),
    "b2dp_allocator_group_count": (_i, [_vp, _i32p]),
    "b2dp_allocator_candidates": (_i, [_vp, _strs, _i, _strs, _i, _i, _i32p, _i32p]),
    "b2dp_allocator_allocate": (_i, [_vp, _strs, _i, _strs, _i, _i, _P(Id64), _i, _ip]),
    "b2dp_start": (_i, [_vp]),
    "b2dp_pair_weights": (_i, [_vp, _P(PairWeight), _i, _ip, _ip]),
    "b2dp_preferred_allocation_available": (_i, [_vp, _i32p]),
    "b2dp_preferred_allocation": (_i, [_vp, _strs, _i, _strs, _i, _i, _P(Id64), _i, _ip]),
    "b2dp_p2p_matrix": (_i, [_vp, _P(P2pOpts), _P(C.c_float), _i32p, _P(C.c_uint64), _i]),
    "b2dp_export_kfd_tree": (_i, [_vp, _cp]),
    "b2dp_set_vendor_domain": (_i, [_cp]),
    "b2dp_create_labels": (_i, [_cp, _P(KvCount), _i, _P(Label), _i, _ip]),
    "b2dp_label_generator_names": (_i, [_P(Id64), _i, _ip]),
    "b2dp_generate_labels": (_i, [_vp, _cp, _P(Label), _i, _ip]),
    "b2dp_remove_old_node_labels": (_i, [_P(Label), _i, _ip]),
}
ABI_VERSION = 3          # must equal B2DP_ABI_VERSION in include/b200dp.h (struct layouts above)
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)   # AttributeError here = the .so does not export what the header declares
    _fn.restype = _res
    _fn.argtypes = _args


if lib.b2dp_abi_version() != ABI_VERSION:
    raise ImportError("libb200dp.so has ABI %d, this binding expects %d: rebuild (make -C k8s-device-plugin_b200/csrc)"
                      % (lib.b2dp_abi_version(), ABI_VERSION))


class B2dpError(Exception):
    """A negative return code from the C ABI."""

    def __init__(self, code, detail=""):
        msg = lib.b2dp_strerror(code).decode()
        super().__init__(f"{msg} [{code}]" + (f": {detail}" if detail else ""))
        self.code = code
        self.message = msg
        self.detail = detail


def check(rc, ctx=None):
    if rc != OK:
        detail = lib.b2dp_last_error(ctx).decode() if ctx else ""
        raise B2dpError(rc, detail)
    return rc


def s(b: bytes) -> str:
    return b.decode("utf-8", "replace")


def str_array(items):
    arr = (C.c_char_p * max(1, len(items)))()
    for i, it in enumerate(items):
        arr[i] = it.encode() if isinstance(it, str) else it
    return arr


def grow_call(make_array, call):
    """Call an (out, cap, *n) style function, growing the array on B2DP_E_NOSPC."""
    cap = 64
    while True:
        arr = make_array(cap)
        n = C.c_int(0)
        rc = call(arr, cap, C.byref(n))
        if rc == E_NOSPC:
            cap = max(n.value, cap * 2)
            continue
        return rc, arr, n.value


_log_keepalive = None


def set_log_callback(fn):
    """Route the library's diagnostics to `fn(level, message)` (level 0 info / 1 warning / 2 error); None removes it."""
    global _log_keepalive
    if fn is None:
        lib.b2dp_set_log_callback(C.cast(None, LogCb), None)
        _log_keepalive = None
        return
    cb = LogCb(lambda _user, level, msg: fn(level, msg.decode("utf-8", "replace")))
    lib.b2dp_set_log_callback(cb, None)
    _log_keepalive = cb
