"""Context: one opened backend of libb200dp (`kfd:<sysroot>` parity mode or `cuda:` real B200s)."""
import ctypes as C
import threading
from dataclasses import dataclass
from typing import Dict, List, Optional

from . import _native as N


@dataclass
class ProbeResult:
    device: int
    healthy: bool
    err: int
    seed: int
    checksum: int
    expected_checksum: int
    mismatches: int
    first_bad_word: int
    bytes: int
    ms_event: float
    ms_device: float
    gbs: float
    flags: int = 0
    gbs_ref: float = 0.0           # the device's calibrated ceiling
    frac: float = 0.0              # gbs / gbs_ref
    min_gbs_applied: float = 0.0   # the floor the verdict used


@dataclass
class CycleStats:
    n_devices: int
    n_unhealthy: int
    homogeneous: bool
    node_healthy: bool
    ms_total: float
    ms_enumerate: float
    ms_probe: float
    ms_encode: float
    probe_gbs_min: float
    probe_gbs_sum: float
    probe_bytes: int
    ms_link_check: float = 0.0
    n_link_faults: int = 0
    probe_ms_device_max: float = 0.0
    probe_frac_min: float = 0.0


@dataclass
class ComputeResult:
    """One device's tensor-core check (b2dp_compute_result); masks are ints with bit s = %smid s."""
    device: int
    healthy: bool
    err: int
    seed: int
    sms: int
    sms_covered: int
    sms_failed: int
    first_bad_sm: int
    first_bad_kind: int
    first_bad_tile: int
    first_bad_row: int
    tiles: int
    bad_rows: int
    bad_sm_mask: int
    covered_mask: int
    ms_device: float
    ms_event: float
    tflops: float


def _mask(words) -> int:
    return sum(int(w) << (32 * i) for i, w in enumerate(words))


def compute_expected(seed: int, kind: int, a_set: int, b_set: int):
    """The host's 128 row hashes of tile (a_set, b_set) (b2dp_compute_expected; no context, no GPU)."""
    import numpy as np
    out = np.zeros(128, dtype=np.uint64)
    n = C.c_int()
    N.check(N.lib.b2dp_compute_expected(seed, kind, a_set, b_set, out.ctypes.data_as(C.POINTER(C.c_uint64)), 128,
                                        C.byref(n)))
    return out[:n.value]


class Context:
    def __init__(self, uri: str):
        self.uri = uri
        self._h = C.c_void_p()
        rc = N.lib.b2dp_open(uri.encode(), C.byref(self._h))
        if rc != N.OK:
            raise N.B2dpError(rc, N.lib.b2dp_last_error(None).decode())
        self._buf = (C.c_uint8 * (1 << 16))()
        self._buf_lock = threading.Lock()      # one response buffer, several gRPC handler threads
        self._opts_cache = {}

    def close(self):
        if self._h:
            N.lib.b2dp_close(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- enumerate -----------------------------------------------------------------------
    def enumerate_raw(self):
        rc, arr, n = N.grow_call(lambda cap: (N.Device * cap)(),
                                 lambda a, cap, pn: N.lib.b2dp_enumerate(self._h, a, cap, pn))
        N.check(rc, self._h)
        return arr, n

    def enumerate(self) -> Dict[str, dict]:
        """GetAMDGPUs()-shaped map (amdgpu.go:216), canonical order (sorted by id)."""
        arr, n = self.enumerate_raw()
        return {N.s(d.id): {"card": d.card, "renderD": d.render_d, "devID": N.s(d.dev_id),
                            "computePartitionType": N.s(d.compute_partition),
                            "memoryPartitionType": N.s(d.memory_partition), "numaNode": d.numa_node,
                            "nodeId": d.node_id} for d in arr[:n]}

    def partition_histogram(self) -> Dict[str, int]:
        rc, arr, n = N.grow_call(lambda cap: (N.KvCount * cap)(),
                                 lambda a, cap, pn: N.lib.b2dp_partition_histogram(self._h, a, cap, pn))
        N.check(rc, self._h)
        return {N.s(e.key): e.count for e in arr[:n]}

    def is_homogeneous(self) -> bool:
        v = C.c_int32()
        N.check(N.lib.b2dp_is_homogeneous(self._h, C.byref(v)), self._h)
        return bool(v.value)

    def partition_supported(self, which: int) -> bool:
        v = C.c_int32()
        N.check(N.lib.b2dp_partition_supported(self._h, which, C.byref(v)), self._h)
        return bool(v.value)

    def resource_list(self, strategy: str) -> List[str]:
        rc, arr, n = N.grow_call(lambda cap: (N.Id64 * cap)(),
                                 lambda a, cap, pn: N.lib.b2dp_resource_list(self._h, strategy.encode(), a, cap, pn))
        N.check(rc, self._h)
        return [N.s(arr[i].value) for i in range(n)]

    # ---- health --------------------------------------------------------------------------
    def node_health(self) -> bool:
        v = C.c_int32()
        N.check(N.lib.b2dp_node_health(self._h, C.byref(v)), self._h)
        return bool(v.value)

    def probe_health(self, timeout_ms=0, variant=N.PROBE_VARIANT_TMA, min_gbs=0.0, via_workers=False,
                     timed=True, grid_ctas=0) -> List[ProbeResult]:
        """One fan-out pass.  timed=True brackets each kernel with CUDA events (ms_event, what the roofline
        is measured with); timed=False is the kubelet-facing configuration (completion by the published
        result block alone, GB/s from the in-kernel timer)."""
        opts = N.ProbeOpts(timeout_ms, variant | (N.PROBE_VIA_WORKERS if via_workers else 0)
                           | (N.PROBE_EVENT_TIMING if timed else 0), min_gbs, grid_ctas)
        rc, arr, n = N.grow_call(lambda cap: (N.ProbeResult * cap)(),
                                 lambda a, cap, pn: N.lib.b2dp_probe_health(self._h, C.byref(opts), a, cap, pn))
        N.check(rc, self._h)
        return [ProbeResult(r.device, bool(r.healthy), r.err, r.seed, r.checksum, r.expected_checksum, r.mismatches,
                            r.first_bad_word, r.bytes, r.ms_event, r.ms_device, r.gbs, r.flags, r.gbs_ref, r.frac,
                            r.min_gbs_applied) for r in arr[:n]]

    def probe_inject_fault(self, device: int, word_index: int, mask: int):
        N.check(N.lib.b2dp_probe_inject_fault(self._h, device, word_index, mask), self._h)

    def probe_reset(self, device: int = -1):
        N.check(N.lib.b2dp_probe_reset(self._h, device), self._h)

    def probe_set_ref(self, device: int = -1, gbs_ref: float = 0.0):
        """Pin the bandwidth ceiling the fractional floor refers to (<= 0: back to the device's own calibration)."""
        N.check(N.lib.b2dp_probe_set_ref(self._h, device, gbs_ref), self._h)

    def probe_describe(self, device: int) -> dict:
        """Ring geometry, calibrated ceiling and runtime identity of `device` (b2dp_probe_describe); no pass runs."""
        info = N.ProbeInfo()
        N.check(N.lib.b2dp_probe_describe(self._h, device, C.byref(info)), self._h)
        return {"slot_bytes": info.slot_bytes, "total_memory": info.total_memory, "sm_count": info.sm_count,
                "slots": info.slots, "gbs_cal": info.gbs_cal, "gbs_ref": info.gbs_ref, "usable": bool(info.usable),
                "via_helper": bool(info.via_helper), "uuid": N.s(info.uuid), "name": N.s(info.name)}

    def probe_peek(self, device: int, word_index: int, n_words: int):
        import numpy as np
        out = np.empty(n_words, dtype=np.uint32)
        N.check(N.lib.b2dp_probe_peek(self._h, device, word_index, out.ctypes.data_as(C.POINTER(C.c_uint32)), n_words),
                self._h)
        return out

    # ---- tensor-core check ---------------------------------------------------------------
    def compute_check(self, tiles: int = 0, timeout_ms: int = 0, timed: bool = False) -> List[ComputeResult]:
        """The tensor-core check on every GPU at once (b2dp_compute_check), with per-SM detail."""
        opts = N.ComputeOpts(timeout_ms, tiles, N.COMPUTE_EVENT_TIMING if timed else 0, 0)
        rc, arr, n = N.grow_call(lambda cap: (N.ComputeResult * cap)(),
                                 lambda a, cap, pn: N.lib.b2dp_compute_check(self._h, C.byref(opts), a, cap, pn))
        N.check(rc, self._h)
        return [ComputeResult(r.device, bool(r.healthy), r.err, r.seed, r.sms, r.sms_covered, r.sms_failed,
                              r.first_bad_sm, r.first_bad_kind, r.first_bad_tile, r.first_bad_row, r.tiles, r.bad_rows,
                              _mask(r.bad_sm_mask), _mask(r.covered_mask), r.ms_device, r.ms_event, r.tflops)
                for r in arr[:n]]

    def compute_tile(self, device: int, kind: int, a_set: int, b_set: int):
        """One tile C = A[a_set] . B[b_set]^T of `kind` on one CTA: the raw fp32 accumulator, [128, 128]."""
        import numpy as np
        c = np.zeros((128, 128), dtype=np.float32)
        N.check(N.lib.b2dp_compute_tile(self._h, device, kind, a_set, b_set, c.ctypes.data_as(C.POINTER(C.c_float))),
                self._h)
        return c

    def compute_inject_fault(self, device: int, sm: int, mask: int):
        """One-shot: the next check on `device` flips `mask` into one accumulator word on %smid `sm`."""
        N.check(N.lib.b2dp_compute_inject_fault(self._h, device, sm, mask), self._h)

    # ---- ListAndWatch --------------------------------------------------------------------
    def list_and_watch(self, resource: str = "gpu", flags: int = N.LW_INITIAL, external: Optional[Dict[str, bool]] = None,
                       timeout_ms=0, variant=N.PROBE_VARIANT_TMA, min_gbs=0.0, timed=False):
        """One ListAndWatch send: (serialized ListAndWatchResponse bytes, CycleStats)."""
        key = (flags, timeout_ms, variant, min_gbs, timed)
        opts = self._opts_cache.get(key) if external is None else None      # the heartbeat path re-uses its options block
        if opts is None:
            opts = N.CycleOpts()
            opts.flags = flags
            opts.probe = N.ProbeOpts(timeout_ms, variant | (N.PROBE_EVENT_TIMING if timed else 0), min_gbs, 0)
            if external is None:
                self._opts_cache[key] = opts
        keep = None
        if external is not None:
            opts.flags |= N.LW_EXTERNAL_SOURCE
            ids = (N.Id64 * max(1, len(external)))()
            hl = (C.c_int32 * max(1, len(external)))()
            for i, (k, v) in enumerate(external.items()):
                ids[i].value = k.encode()
                hl[i] = 1 if v else 0
            opts.src_ids, opts.src_health, opts.src_n = ids, hl, len(external)
            keep = (ids, hl)
        ln = C.c_size_t(0)
        st = N.CycleStats()
        with self._buf_lock:
            rc = N.lib.b2dp_list_and_watch(self._h, resource.encode(), C.byref(opts), self._buf, len(self._buf),
                                           C.byref(ln), C.byref(st))
            if rc == N.E_NOSPC:
                self._buf = (C.c_uint8 * (ln.value * 2))()
                rc = N.lib.b2dp_list_and_watch(self._h, resource.encode(), C.byref(opts), self._buf, len(self._buf),
                                               C.byref(ln), C.byref(st))
            N.check(rc, self._h)
            wire = C.string_at(self._buf, ln.value)
        del keep
        stats = CycleStats(st.n_devices, st.n_unhealthy, bool(st.homogeneous), bool(st.node_healthy), st.ms_total,
                           st.ms_enumerate, st.ms_probe, st.ms_encode, st.probe_gbs_min, st.probe_gbs_sum,
                           st.probe_bytes, st.ms_link_check, st.n_link_faults, st.probe_ms_device_max, st.probe_frac_min)
        return wire, stats

    def watch(self, callback, resource: str = "gpu", pulse_ms: int = 0, flags: int = 0, timeout_ms=0, min_gbs=0.0):
        """Start the library-owned ListAndWatch loop (b2dp_watch_start).  `callback(rc, wire, stats)`
        runs on the library's thread for the initial list and every heartbeat.  Returns a Watch."""
        return Watch(self, callback, resource, pulse_ms, flags, timeout_ms, min_gbs)

    # ---- Allocate ------------------------------------------------------------------------
    def device_specs(self, ids: List[str]):
        arr_in = N.str_array(ids)
        rc, arr, n = N.grow_call(lambda cap: (N.DevSpec * cap)(),
                                 lambda a, cap, pn: N.lib.b2dp_device_specs(self._h, arr_in, len(ids), a, cap, pn))
        N.check(rc, self._h)
        return [(N.s(x.host_path), N.s(x.container_path), N.s(x.permissions)) for x in arr[:n]]

    def allocate_response(self, ids: List[str]) -> bytes:
        arr_in = N.str_array(ids)
        buf = (C.c_uint8 * (256 + 256 * max(1, len(ids))))()
        ln = C.c_size_t(0)
        N.check(N.lib.b2dp_allocate_response(self._h, arr_in, len(ids), buf, len(buf), C.byref(ln)), self._h)
        return bytes(buf[:ln.value])

    # ---- Start / GetPreferredAllocation -----------------------------------------------------
    def start(self) -> int:
        """plugin.go:82-91 Start(); returns the allocator-init rc (0 ok) without raising."""
        return N.lib.b2dp_start(self._h)

    def pair_weights(self):
        """p2pWeights of the context's own allocator as {from: {to: weight}} (device.go:220-252); needs start()."""
        cap = 4096
        while True:
            arr = (N.PairWeight * cap)()
            n, rows = C.c_int(0), C.c_int(0)
            rc = N.lib.b2dp_pair_weights(self._h, arr, cap, C.byref(n), C.byref(rows))
            if rc == N.E_NOSPC:
                cap = n.value
                continue
            N.check(rc, self._h)
            break
        w = {}
        for e in arr[:n.value]:
            w.setdefault(e.node_from, {})[e.node_to] = e.weight
        return w

    def preferred_allocation_available(self) -> bool:
        v = C.c_int32()
        N.check(N.lib.b2dp_preferred_allocation_available(self._h, C.byref(v)), self._h)
        return bool(v.value)

    def preferred_allocation(self, available: List[str], must_include: List[str], size: int) -> List[str]:
        a, m = N.str_array(available), N.str_array(must_include)
        out = (N.Id64 * max(1, len(available), len(must_include)))()
        n = C.c_int(0)
        rc = N.lib.b2dp_preferred_allocation(self._h, a, len(available), m, len(must_include), size, out, len(out),
                                             C.byref(n))
        N.check(rc, self._h)
        return [N.s(out[i].value) for i in range(n.value)]

    # ---- P2P / export / labels -------------------------------------------------------------
    def p2p_matrix(self, bytes_per_pair: int = 0, iters: int = 0, bidir: bool = False):
        import numpy as np
        arr, n = self.enumerate_raw()
        gbs = np.zeros((n, n), dtype=np.float32)
        lt = np.zeros((n, n), dtype=np.int32)
        mm = np.zeros((n, n), dtype=np.uint64)
        opts = N.P2pOpts(bytes_per_pair, iters, 1 if bidir else 0)
        N.check(N.lib.b2dp_p2p_matrix(self._h, C.byref(opts), gbs.ctypes.data_as(C.POINTER(C.c_float)),
                                      lt.ctypes.data_as(C.POINTER(C.c_int32)),
                                      mm.ctypes.data_as(C.POINTER(C.c_uint64)), n), self._h)
        return gbs, lt, mm

    def export_kfd_tree(self, directory: str):
        N.check(N.lib.b2dp_export_kfd_tree(self._h, directory.encode()), self._h)

    def generate_labels(self, enabled: List[str]) -> Dict[str, str]:
        csv = ",".join(enabled).encode()
        rc, arr, n = N.grow_call(lambda cap: (N.Label * cap)(),
                                 lambda a, cap, pn: N.lib.b2dp_generate_labels(self._h, csv, a, cap, pn))
        N.check(rc, self._h)
        return {N.s(x.key): N.s(x.value) for x in arr[:n]}


class Watch:
    """Handle of a native ListAndWatch loop: beat() = one heartbeat tick, stop() ends the stream."""

    def __init__(self, ctx: Context, callback, resource, pulse_ms, flags, timeout_ms, min_gbs):
        opts = N.CycleOpts()
        opts.flags = flags
        opts.probe = N.ProbeOpts(timeout_ms, 0, min_gbs, 0)

        def tramp(_user, rc, buf, ln, st):
            s = st.contents
            stats = CycleStats(s.n_devices, s.n_unhealthy, bool(s.homogeneous), bool(s.node_healthy), s.ms_total,
                               s.ms_enumerate, s.ms_probe, s.ms_encode, s.probe_gbs_min, s.probe_gbs_sum, s.probe_bytes,
                               s.ms_link_check, s.n_link_faults, s.probe_ms_device_max, s.probe_frac_min)
            callback(rc, bytes(buf[:ln]) if ln else b"", stats)
        self._cb = N.WatchCb(tramp)          # keep the trampoline alive as long as the loop
        self._h = C.c_void_p()
        N.check(N.lib.b2dp_watch_start(ctx._h, resource.encode(), pulse_ms, C.byref(opts), self._cb, None,
                                       C.byref(self._h)), ctx._h)

    def beat(self):
        N.check(N.lib.b2dp_watch_beat(self._h))

    def stop(self):
        if self._h:
            N.lib.b2dp_watch_stop(self._h)
            self._h = C.c_void_p()
