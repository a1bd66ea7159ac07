#!/usr/bin/env python3
"""bench.py -- the hot path of BASELINE.json on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, 1 rank/GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W

metric  : health_probe_hbm_gbs -- bytes of HBM streamed + verified per second by the per-GPU health
          probe (BASELINE.json "per-GPU health-probe HBM GB/s vs peak"), whole job = sum over GPUs;
          `ms_per_step`/`cycle_ms` carry the second half of the metric ("ListAndWatch cycle ms").
step    : one heartbeat's GPU work on every GPU of the job: 1 GiB src -> 1 GiB dst per GPU, verified
          word by word (algorithmic bytes 2*S = 2 GiB per GPU per step).  Inputs (1 GiB) >> 126 MB L2.
value   : K x b2dp_probe_health() (C ABI; buffers resident in HBM), wall clock bracketed by
          barrier + synchronize, max over ranks.
e2e     : K x b2dp_list_and_watch(HEARTBEAT): enumerate -> node health -> probe fan-out -> health
          merge -> serialized v1beta1.ListAndWatchResponse in a host buffer -- the call a kubelet-facing
          host makes.  The path has no bulk host inputs: per step the host sends kernel arguments and
          receives the 48-byte result block per device through pinned mapped memory plus the response.
roofline: achieved = 2*S / mean CUDA-event time of the probe kernel over the timed steps; peak =
          MEASURED_PEAKS.json hbm_gbs (else the 6650 GB/s fallback of B200_PROFILING.md).
single_process / p2p / parity (rank 0, after the per-rank legs, every other rank idle): the DEPLOYMENT shape --
          ONE plugin process driving all N GPUs (BASELINE.json configs[2], "<10 ms over 8 B200s"): ListAndWatch
          heartbeat cycle p50/p99/max with one N-device response; the NVLink P2P matrix (configs[3]); and, untimed,
          the product's answers against the oracle on the tree the product exports (device table, pair weights from
          the MEASURED links, every allocation size, ListAndWatch list, labels).  A false parity entry fails the run.
"""
import argparse
import importlib
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
PKG = "k8s-device-plugin_b200"
S_BYTES = 1 << 30
METRIC, UNIT = "health_probe_hbm_gbs", "GB/s"
WORKLOAD = "1xB200 enumerate + ListAndWatch with sm_100a HBM health-probe kernel (BASELINE.json configs[1]), per GPU"

SAMPLER = r"""
import sys, time
import pynvml as nv
nv.nvmlInit()
h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
bad = {getattr(nv, n): n for n in dir(nv) if n.startswith("nvmlClocksEventReason") or n.startswith("nvmlClocksThrottleReason")}
mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
out = open(sys.argv[2], "w", buffering=1)
out.write("max,%d\n" % mx)
while True:
    try:
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        out.write("%d,%d,%d\n" % (time.monotonic_ns(), sm, r))
    except Exception as e:
        out.write("err,%s\n" % e)
    time.sleep(0.004)
"""

# NVML clocks-event-reason bits (nvml.h)
REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
           0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
           0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}


def bench_config(n):
    """The workload description, IDENTICAL in both arms (the driver compares the two `config` objects)."""
    return {"workload": WORKLOAD, "n_devices": n, "probe_bytes_per_buffer": S_BYTES,
            "algorithmic_bytes_per_gpu_step": 2 * S_BYTES,
            "l2": "inputs (1 GiB per buffer) larger than the 126 MB L2; buffers ping-pong every step",
            "parallelism": "1 unit per GPU, no data-path collective"}


def pctl(v, q):
    v = sorted(v)
    return v[int(q * (len(v) - 1) + 0.5)] if v else None


def dist3(v, nd=4):
    return {"p50": round(pctl(v, 0.5), nd), "p99": round(pctl(v, 0.99), nd), "max": round(max(v), nd), "n": len(v)}


class ClockSampler:
    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(prefix="b2dp_clk_", suffix=".csv")
        try:
            self.p = subprocess.Popen([sys.executable, "-c", SAMPLER, str(gpu_index), self.path],
                                      stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        time.sleep(0.3)

    def stop(self, windows):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        sm, bits = [], 0
        try:
            for line in open(self.path):
                a = line.strip().split(",")
                if a[0] == "max":
                    out["sm_max_mhz"] = int(a[1])
                elif a[0].isdigit():
                    t = int(a[0])
                    if any(lo <= t <= hi for lo, hi in windows):
                        sm.append(int(a[1]))
                        bits |= int(a[2])
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
        out["samples"] = len(sm)
        out["reasons"] = [n for b, n in REASONS.items() if bits & b and n != "gpu_idle"]
        return out


def peak_hbm():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_per_launch():
    """dram__bytes_read.sum + dram__bytes_write.sum of one probe launch, from the committed ncu capture (a constant
    read from profiles/traffic.json -- ncu cannot run inside a timed bench)."""
    try:
        d = json.load(open(os.path.join(REPO, "profiles", "traffic.json")))
        return d["hbm_probe_tma_bytes_per_launch"], d.get("source", "profiles/traffic.json")
    except Exception:
        return None, None


def load_synth():
    """The synthetic kfd-tree writer, loaded by FILE PATH: it is pure Python, and importing the product package
    (which maps libb200dp.so) has no place in the CPU legs."""
    spec = importlib.util.spec_from_file_location("b2dp_synth", os.path.join(REPO, PKG, "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cpu_probe_baseline(threads, budget_s=6.0, sample_bytes=S_BYTES):
    """The oracle's C restatement of the probe pass streamed through host DRAM (bounded sample)."""
    import numpy as np
    from oracle import cbind
    import ctypes as C
    cbind.build()
    lib = cbind.probe_lib()
    n_words = sample_bytes // 4
    src = np.empty(n_words, dtype=np.uint32)
    dst = np.empty(n_words, dtype=np.uint32)
    seed = 0x5EED0000
    lib.oracle_fill(src.ctypes.data, n_words, seed, threads)
    out = (C.c_uint64 * 3)()
    lib.oracle_probe_pass(src.ctypes.data, dst.ctypes.data, n_words, seed, 0, threads, out)   # warm-up / page-in
    passes, t0 = 0, time.perf_counter()
    while True:
        lib.oracle_probe_pass(src.ctypes.data, dst.ctypes.data, n_words, seed, 0, threads, out)
        passes += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or passes >= 400:
            break
    assert out[1] == 0
    return 2.0 * sample_bytes * passes / dt / 1e9, passes, dt


def kfd_walk_baseline(n_devices, reps=200):
    """Reference-shaped CPU cycle (C port of the Go walk) on a synthetic N-device kfd tree in /dev/shm."""
    from oracle import cbind
    cbind.build()
    k = cbind.kfd_lib()
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    root = tempfile.mkdtemp(prefix="b2dp_bench_kfd_", dir=base)
    load_synth().write_b200_tree(root, n_gpus=n_devices)
    r = root.encode()
    for _ in range(3):
        k.kfdwalk_cycle(r, 1)
    t0 = time.perf_counter()
    for _ in range(reps):
        k.kfdwalk_cycle(r, 1)
    start_ms = (time.perf_counter() - t0) / reps * 1e3
    t0 = time.perf_counter()
    for _ in range(reps):
        k.kfdwalk_cycle(r, 0)
    beat_ms = (time.perf_counter() - t0) / reps * 1e3
    import shutil
    shutil.rmtree(root, ignore_errors=True)
    return start_ms, beat_ms


def run_reference(args, rank, world):
    """The reference's CPU path on the box's host cores: per step, the reference-shaped
    ListAndWatch cycle (kfd walk: enumerate x2 + text health check, C port of the Go code) followed
    by the CPU restatement of the probe over the same S = 1 GiB buffer per device.  Touches nothing of the product:
    no package import, no libb200dp.so."""
    if rank != 0:
        return
    import numpy as np
    import ctypes as C
    from oracle import cbind
    cbind.build()
    lib, k = cbind.probe_lib(), cbind.kfd_lib()
    threads = os.cpu_count() or 1
    n = args.gpus
    warmup = max(3, args.warmup)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    root = tempfile.mkdtemp(prefix="b2dp_ref_kfd_", dir=base)
    load_synth().write_b200_tree(root, n_gpus=n)
    r = root.encode()
    sample = S_BYTES                                  # the product arm's S: 1 GiB read + 1 GiB written per device per step
    n_words = sample // 4
    src = np.empty(n_words, dtype=np.uint32)
    dst = np.empty(n_words, dtype=np.uint32)
    seed = 0x5EED0000
    lib.oracle_fill(src.ctypes.data, n_words, seed, threads)
    out = (C.c_uint64 * 3)()
    lib.oracle_probe_pass(src.ctypes.data, dst.ctypes.data, n_words, seed, 0, threads, out)      # page-in
    t0 = time.perf_counter()
    lib.oracle_probe_pass(src.ctypes.data, dst.ctypes.data, n_words, seed, 0, threads, out)
    per_pass = time.perf_counter() - t0
    # bounded: the whole run stays within ~2 minutes; only a slow host ever shrinks the sample, and says so
    while sample > (16 << 20) and per_pass * n * (args.steps + warmup) > 120.0:
        sample //= 2
        per_pass /= 2
    n_words = sample // 4

    for _ in range(warmup):
        k.kfdwalk_cycle(r, 1)
        for _ in range(n):
            lib.oracle_probe_pass(src.ctypes.data, dst.ctypes.data, n_words, seed, 0, threads, out)
    walk, step_ms = 0.0, []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        w0 = time.perf_counter()
        k.kfdwalk_cycle(r, 1)
        walk += time.perf_counter() - w0
        for _ in range(n):
            lib.oracle_probe_pass(src.ctypes.data, dst.ctypes.data, n_words, seed, 0, threads, out)
        step_ms.append((time.perf_counter() - w0) * 1e3)
    dt = time.perf_counter() - t0
    assert out[1] == 0
    import shutil
    shutil.rmtree(root, ignore_errors=True)
    value = n * 2.0 * sample * args.steps / dt / 1e9
    sample_desc = ("%d MiB of the %d MiB per-device probe buffer per device per step (%s), %d device(s), host DRAM, %d threads"
                   % (sample >> 20, S_BYTES >> 20, "the full buffer" if sample == S_BYTES else "shrunk to bound the run", n, threads))
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": n,
        "steps": args.steps, "warmup": warmup, "ms_per_step": round(dt / args.steps * 1e3, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": bench_config(n),
        "arm": "CPU: C port of the reference's kfd walk (no Go toolchain here; the reference has no GPU probe) + CPU "
               "restatement of the probe pass, all host threads",
        "step_ms": dist3(step_ms),
        "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample_desc,
                         "cycle_ms_kfd_walk": round(walk / args.steps * 1e3, 4)},
        "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---- rank-0-only legs of the product arm ---------------------------------------------------------------------------
def single_process_leg(pkg, n, steps, warmup, variant):
    """ONE context over all N GPUs (the daemon's shape): the kubelet-facing heartbeat cycle, per-GPU roofline
    fractions, and the NVLink P2P matrix.  Returns (ctx, single_process dict, p2p dict)."""
    N = pkg._native
    peak, _ = peak_hbm()
    uri = "cuda:bytes=%d,devices=%s" % (S_BYTES, "+".join(str(i) for i in range(n)))
    t0 = time.perf_counter()
    ctx = pkg.Context(uri)
    open_s = time.perf_counter() - t0
    ctx.list_and_watch("gpu", N.LW_INITIAL)
    t_w, i = time.perf_counter(), 0
    while i < warmup or time.perf_counter() - t_w < 0.1:
        ctx.list_and_watch("gpu", N.LW_HEARTBEAT, variant=variant)
        i += 1
    cyc, kmax, host, unhealthy = [], [], [], 0
    for _ in range(steps):
        t0 = time.perf_counter()
        wire, st = ctx.list_and_watch("gpu", N.LW_HEARTBEAT, variant=variant)
        dt = (time.perf_counter() - t0) * 1e3
        cyc.append(dt)
        kmax.append(st.probe_ms_device_max)
        host.append(dt - st.probe_ms_device_max)
        unhealthy += st.n_unhealthy
    msg = pkg.v1beta1.ListAndWatchResponse.FromString(wire)
    assert len(msg.devices) == n and all(d.health == "Healthy" for d in msg.devices), msg
    per_gpu = [[] for _ in range(n)]
    refs = [0.0] * n
    for _ in range(max(20, steps // 10)):
        for r in ctx.probe_health(variant=variant):              # CUDA-event timed, like the roofline leg
            per_gpu[r.device].append(r.gbs)
            refs[r.device] = r.gbs_ref
    p50 = pctl(cyc, 0.5)
    sp = {"n_devices": n, "uri": uri, "open_s": round(open_s, 3), "cycles": steps,
          "cycle_ms_p50": round(p50, 4), "cycle_ms_p99": round(pctl(cyc, 0.99), 4), "cycle_ms_max": round(max(cyc), 4),
          "response_bytes": len(wire), "unhealthy_verdicts": unhealthy,
          "per_gpu_gbs": [round(statistics.median(g), 1) for g in per_gpu],
          "per_gpu_frac": [round(statistics.median(g) / peak, 4) for g in per_gpu],
          "per_gpu_calibrated_ceiling_gbs": [round(x, 1) for x in refs],
          "aggregate_gbs": round(n * 2.0 * S_BYTES / (p50 * 1e-3) / 1e9, 1),
          # tail attribution: the slowest GPU's in-kernel span (first CTA start .. result published) of each cycle vs
          # everything the host adds around it (enqueue on N streams, polling, merge, protobuf, the Python call)
          "slowest_kernel_ms": dist3(kmax), "host_overhead_ms": dist3(host),
          "target_ms": 10.0, "under_target": bool(pctl(cyc, 0.99) < 10.0)}
    p2p = {"pairs": 0}
    if n > 1:
        t0 = time.perf_counter()
        gbs, lt, mm = ctx.p2p_matrix()
        off = sorted(float(gbs[i, j]) for i in range(n) for j in range(n) if i != j)
        classes = {}
        for i in range(n):
            for j in range(n):
                if i != j:
                    classes[str(int(lt[i, j]))] = classes.get(str(int(lt[i, j])), 0) + 1
        p2p = {"pairs": len(off), "bytes_per_pair": 256 << 20, "matrix_s": round(time.perf_counter() - t0, 3),
               "gbs_min": round(off[0], 1), "gbs_median": round(statistics.median(off), 1), "gbs_max": round(off[-1], 1),
               "frac_of_770": round(statistics.median(off) / 770.0, 4), "mismatches": int(mm.sum()),
               "link_classes": classes,
               "note": "one direction of every pair per half-round, N-1 rounds of disjoint matchings; 770 GB/s = measured "
                       "peer-copy reference (B200_PROFILING.md)"}
    return ctx, sp, p2p


def parity_block(pkg, ctx, n):
    """UNTIMED checker leg (after every timed region): the product's answers on the live node against the oracle
    (the CPU restatement of the reference) on the kfd-shaped tree the product exports -- BASELINE.json's
    "bit-exact on integer fields ... when both are pointed at equivalent fixtures"."""
    import shutil
    from oracle import allocator as oalloc
    from oracle import amdgpu as oamd
    from oracle import labeller as olab
    from oracle import plugin as oplug
    from oracle import probe as oprobe
    N = pkg._native
    root = tempfile.mkdtemp(prefix="b2dp_parity_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    out = {}
    try:
        devs = ctx.enumerate()
        ctx.export_kfd_tree(root)                       # measures the P2P links if they have not been yet
        want = oamd.GetAMDGPUs(root)
        out["enumerate"] = devs == want and len(devs) == n
        ids = sorted(devs)
        rc = ctx.start()
        opol = oalloc.BestEffortPolicy()
        oerr = opol.Init(oplug.getDevices(root), root + "/sys/class/kfd/kfd/topology/nodes")
        if n > 1:
            out["pair_weights"] = rc == 0 and oerr is None and ctx.pair_weights() == opol.p2pWeights
            ok = rc == 0 and oerr is None
            for size in range(1, n + 1):
                ok = ok and ctx.preferred_allocation(ids, [], size) == opol.Allocate(list(ids), [], size)[0]
            for must in (ids[-1:], ids[:1] + ids[-1:]):
                for size in range(len(must), n + 1):
                    ok = ok and ctx.preferred_allocation(ids, must, size) == opol.Allocate(list(ids), list(must), size)[0]
            out["allocations_all_sizes"] = ok
        else:                                           # one device: both sides must refuse the same way
            out["pair_weights"] = rc == N.E_ALLOC_NO_WEIGHTS and oerr is not None
            out["allocations_all_sizes"] = not ctx.preferred_allocation_available()
        wire, _ = ctx.list_and_watch("gpu", N.LW_INITIAL)
        homog, lw = oplug.list_and_watch_devices(want, "gpu")
        msg = pkg.v1beta1.ListAndWatchResponse.FromString(wire)
        out["list_and_watch"] = ([(d.ID, d.health, d.topology.nodes[0].ID) for d in msg.devices] == lw
                                 and msg.SerializeToString() == wire
                                 and ctx.resource_list("single") == oplug.getResourceList("single", root)[0])
        out["node_health"] = ctx.node_health() == oplug.simpleHealthCheck(root + "/sys/class/kfd/kfd")
        gens = ["driver-version", "driver-src-version", "device-id", "product-name", "vram", "simd-count", "cu-count",
                "compute-memory-partition", "compute-partitioning-supported", "memory-partitioning-supported",
                "family", "firmware"]
        drm = {}
        for v in want.values():
            b = "%s/sys/class/drm/card%d/device/" % (root, v["card"])
            fw = dict(ln.split(" ", 1) for ln in open(b + "b2dp_firmware").read().splitlines()) if os.path.exists(b + "b2dp_firmware") else {}
            fw = {k: "".join(ch if ch.isalnum() or ch in ".-_" else "_" for ch in ver.strip()) for k, ver in fw.items()}
            fam = open(b + "b2dp_family").read().strip() if os.path.exists(b + "b2dp_family") else ""
            drm["card%d" % v["card"]] = {"family": fam, "feat": {}, "fw": fw}
        got = ctx.generate_labels(gens)
        out["labels"] = got == olab.generateLabels({g: True for g in gens}, root, drm=drm) and len(got) >= 10
        # the probe's integer results against the oracle's closed form, every device, 1 GiB
        ok = True
        for r in ctx.probe_health():
            ok = ok and r.mismatches == 0 and r.checksum == r.expected_checksum == oprobe.expected_checksum(S_BYTES // 4, r.seed)
        out["probe_checksums"] = ok
        out["label_count"] = len(got)
    finally:
        shutil.rmtree(root, ignore_errors=True)
    return out


DUMP_CHUNKS, DUMP_CHUNK_WORDS = 256, 4096          # 1 Mi words of the probe buffer: 8 MiB as float64


def dump_chunks():
    """First word of each chunk of the probe buffer that --dump-outputs samples: fixed, seeded, ascending."""
    import numpy as np
    rng = np.random.default_rng(0)
    return [int(c) * DUMP_CHUNK_WORDS for c in np.sort(rng.choice(S_BYTES // 4 // DUMP_CHUNK_WORDS, DUMP_CHUNKS, replace=False))]


def probe_outputs(ctx, res):
    """What the value leg's last step returned (--dump-outputs), as float64 arrays.  64-bit integers are split into
    [high, low] 32-bit halves so that float64 holds them exactly; timings are left out, they differ from run to run.
    probe_buffer_sample: the dump_chunks() of the 1 GiB buffer the step wrote (what the next pass verifies)."""
    import numpy as np

    def u64(values):
        return [[v >> 32, v & 0xFFFFFFFF] for v in values]
    return {"probe_seed": [r.seed for r in res], "probe_checksum": u64(r.checksum for r in res),
            "probe_expected_checksum": u64(r.expected_checksum for r in res),
            "probe_mismatches": u64(r.mismatches for r in res), "probe_first_bad_word": u64(r.first_bad_word for r in res),
            "probe_bytes": u64(r.bytes for r in res), "probe_healthy": [float(r.healthy) for r in res],
            "probe_err": [r.err for r in res],
            "probe_buffer_sample": np.concatenate([ctx.probe_peek(0, w, DUMP_CHUNK_WORDS) for w in dump_chunks()])}


def write_outputs(directory, outputs):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, dtype=np.float64))


class FileFlag:
    """Rank 0 works alone while the other ranks sleep on a file (an NCCL barrier would park a spinning kernel on
    every GPU that rank 0 is about to measure)."""

    def __init__(self):
        key = "%s_%s_%d" % (os.environ.get("MASTER_PORT", "0"), os.environ.get("TORCHELASTIC_RUN_ID", "none"), os.getppid())
        self.path = os.path.join(tempfile.gettempdir(), "b2dp_bench_flag_" + key)

    def clear(self):
        try:
            os.unlink(self.path)
        except OSError:
            pass

    def set(self):
        open(self.path, "w").close()

    def wait(self, timeout=900.0):
        t0 = time.time()
        while not os.path.exists(self.path):
            if time.time() - t0 > timeout:
                raise SystemExit("rank 0 never finished its single-process leg")
            time.sleep(0.02)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--variant", type=int, default=0, help="0 = TMA-staged kernel (default), 1 = register path")
    ap.add_argument("--single-cycles", type=int, default=0, help="cycles of the single-process leg (default --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    # stdout carries exactly ONE JSON line: libraries (NCCL prints its version banner there) are
    # diverted to stderr for the whole run and the line is written to the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs dumps the B200 arm's outputs; the reference arm has none to compare")
        run_reference(args, rank, world)
        return
    warmup = max(3, args.warmup)

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the probe has no CPU fallback")
    torch.cuda.set_device(local_rank)
    pkg = importlib.import_module(PKG)      # raises if libb200dp.so is missing
    N = pkg._native
    ranks = importlib.import_module(PKG + ".ranks")
    flag = FileFlag()
    if rank == 0:
        flag.clear()
    rg = ranks.RankGroup(backend="nccl")   # barrier + timing reductions only; no data-path collective
    ctx = pkg.Context("cuda:devices=%d,bytes=%d" % (local_rank, S_BYTES))
    barrier, max_over_ranks, sum_over_ranks = rg.barrier, rg.max, rg.sum

    sampler = ClockSampler(local_rank) if rank == 0 else None
    windows = []

    def warm(fn):
        """W untimed warm-up steps, and never less than 100 ms of them: the first NCCL barrier
        (communicator init) idles the GPU for seconds, so clocks and the driver must be warm
        again before a timed region starts."""
        t_w, i = time.perf_counter(), 0
        while i < warmup or time.perf_counter() - t_w < 0.1:
            fn()
            i += 1

    barrier()   # pays the NCCL communicator init before any warm-up
    # ---- value leg: the probe through the C ABI, buffers resident ------------------------------
    # Every pass re-keys the buffer with the next seed, so the timed passes' inputs depend on how many passes came
    # before them.  The time-bounded warm-up therefore runs on a scratch context over the same GPU, and the measured
    # context runs exactly `warmup` passes: its inputs, and so its results, follow from the arguments alone.
    with pkg.Context(ctx.uri) as scratch:
        warm(lambda: scratch.probe_health(variant=args.variant))
    for _ in range(warmup):
        ctx.probe_health(variant=args.variant)
    barrier()
    kernel_ms, unhealthy, value_ms, fracs = [], 0, [], []
    w0 = time.monotonic_ns()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s0 = time.perf_counter()
        res = ctx.probe_health(variant=args.variant)
        value_ms.append((time.perf_counter() - s0) * 1e3)
        kernel_ms.append(res[0].ms_event)
        fracs.append(res[0].frac)
        unhealthy += sum(0 if r.healthy else 1 for r in res)
    torch.cuda.synchronize()
    t_value = time.perf_counter() - t0
    windows.append((w0, time.monotonic_ns()))
    gbs_ref = res[0].gbs_ref
    outputs = probe_outputs(ctx, res) if args.dump_outputs and rank == 0 else None
    barrier()
    t_value = max_over_ranks(t_value)

    # ---- context for the roofline: the driver's own device-to-device copy of the same size, in this run, on this
    # GPU, timed the same way (CUDA events, after warm-up) -- what a plain copy achieves on this part today -------
    drv_copy_gbs = None
    try:
        a_t = torch.empty(S_BYTES, dtype=torch.uint8, device="cuda")
        b_t = torch.empty(S_BYTES, dtype=torch.uint8, device="cuda")
        a_t.zero_()
        for _ in range(5):
            b_t.copy_(a_t)
        torch.cuda.synchronize()
        best = None
        for _ in range(20):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            b_t.copy_(a_t)
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None or ms < best else best
        drv_copy_gbs = 2.0 * S_BYTES / (best * 1e-3) / 1e9
        del a_t, b_t
        torch.cuda.empty_cache()
    except Exception as e:      # noqa: BLE001
        print("driver copy reference skipped: %r" % (e,), file=sys.stderr)
    barrier()

    # ---- e2e leg: the kubelet-facing call ----------------------------------------------------------
    warm(lambda: ctx.list_and_watch("gpu", N.LW_HEARTBEAT, variant=args.variant))
    barrier()
    enum_ms = enc_ms = 0.0
    e2e_ms = []
    w0 = time.monotonic_ns()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s0 = time.perf_counter()
        wire, st = ctx.list_and_watch("gpu", N.LW_HEARTBEAT, variant=args.variant)
        e2e_ms.append((time.perf_counter() - s0) * 1e3)
        unhealthy += st.n_unhealthy
        enum_ms += st.ms_enumerate
        enc_ms += st.ms_encode
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    windows.append((w0, time.monotonic_ns()))
    barrier()
    t_e2e = max_over_ranks(t_e2e)
    unhealthy = sum_over_ranks(float(unhealthy))
    kernel_ms_mean = sum(kernel_ms) / len(kernel_ms)
    kernel_ms_max_rank = max_over_ranks(kernel_ms_mean)
    e2e_p99_max_rank = max_over_ranks(pctl(e2e_ms, 0.99))
    msg = pkg.v1beta1.ListAndWatchResponse.FromString(wire)
    assert len(msg.devices) == 1 and msg.devices[0].health == "Healthy", msg
    if outputs is not None:
        outputs["list_and_watch_healthy"] = [float(d.health == "Healthy") for d in msg.devices]

    # ---- stream start: the initial ListAndWatch list (enumerate + homogeneity + encode; the reference does
    # two GetAMDGPUs() walks here, plugin.go:231,237) -- reported next to reference_cpu_path ------
    starts = []
    for i in range(60):
        t0 = time.perf_counter()
        ctx.list_and_watch("gpu", N.LW_INITIAL)
        if i >= 10:
            starts.append((time.perf_counter() - t0) * 1e3)
    starts.sort()
    stream_start_ms = max_over_ranks(starts[len(starts) // 2])

    # ---- the kubelet's view: heartbeat tick -> ListAndWatchResponse received over the plugin's unix
    # socket (grpcio server + client stream in this process); informative, not the timed `e2e` ------
    grpc_ms = None
    try:
        import grpc
        srv_mod = importlib.import_module(PKG + ".server")
        V = pkg.v1beta1
        d = tempfile.mkdtemp(prefix="b2b_", dir="/tmp")
        plugin = pkg.plugin.AMDGPUPlugin(ctx, "gpu")
        plugin.Start = lambda: None
        server = srv_mod.PluginServer(plugin, plugin_dir=d).start()
        with grpc.insecure_channel("unix://" + server.socket_path) as ch:
            stream = ch.unary_stream(V.LIST_AND_WATCH, request_serializer=lambda m: m.SerializeToString(),
                                     response_deserializer=lambda b: b)(V.Empty())
            next(stream)
            lat = []
            for i in range(105):
                t0 = time.perf_counter()
                plugin.Heartbeat.put(True)
                next(stream)
                if i >= 5:
                    lat.append((time.perf_counter() - t0) * 1e3)
            stream.cancel()
        server.stop()
        grpc_ms = max_over_ranks(statistics.median(lat))
    except Exception as e:      # noqa: BLE001
        print("grpc leg skipped: %r" % (e,), file=sys.stderr)
        grpc_ms = max_over_ranks(-1.0)

    # ---- the per-rank legs are over: every rank gives its GPU back, then rank 0 alone drives all N GPUs from ONE
    # process (the deployment shape) while the others sleep on a file ----------------------------------------------
    ctx.close()
    barrier()
    sp = p2p = parity = native_ms = None
    failed = None
    if rank == 0:
        try:
            w0 = time.monotonic_ns()
            cycles = args.single_cycles or args.steps
            sctx, sp, p2p = single_process_leg(pkg, world, cycles, warmup, args.variant)
            windows.append((w0, time.monotonic_ns()))
            try:
                parity = parity_block(pkg, sctx, world)
            finally:
                sctx.close()
            # the same with the native daemon (b200dp_plugind: C++ gRPC host, own process, its own context over all N
            # GPUs): SIGUSR1 "heartbeat now" -> probe fan-out -> ListAndWatchResponse received by a grpcio client
            try:
                dp = importlib.import_module(PKG + ".daemon_probe")
                native_ms = dp.heartbeat_latency_ms(sp["uri"], iters=100)
            except Exception as e:      # noqa: BLE001
                print("native daemon leg skipped: %r" % (e,), file=sys.stderr)
        except BaseException as e:      # noqa: BLE001  (the other ranks must be released whatever happens here)
            failed = e
        flag.set()
    else:
        flag.wait()
    barrier()
    if rank == 0:
        flag.clear()

    clocks = sampler.stop(windows) if sampler else None
    if rank != 0:
        rg.close()
        return
    if failed is not None:
        rg.close()
        raise failed

    bytes_per_step_per_gpu = 2.0 * S_BYTES
    n = world
    value = n * bytes_per_step_per_gpu * args.steps / t_value / 1e9
    e2e_value = n * bytes_per_step_per_gpu * args.steps / t_e2e / 1e9
    peak, peak_src = peak_hbm()
    achieved = bytes_per_step_per_gpu / (kernel_ms_mean * 1e-3) / 1e9
    traffic, traffic_src = traffic_per_launch()
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": n, "steps": args.steps, "warmup": warmup,
        "ms_per_step": round(t_value / args.steps * 1e3, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": bench_config(n),
        "arm": "B200: " + ("hbm_probe_tma<4,1024,3> grid=2xSMs" if args.variant == 0 else "hbm_probe_r128<512,2> grid=2xSMs")
               + ", 1 process per GPU for value/e2e (the driver's launch shape), ONE process over all GPUs for single_process/p2p",
        "step_ms": dist3(value_ms),
        "cycle_ms": round(t_e2e / args.steps * 1e3, 4),
        "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 48 * 1 + len(wire),
                "cycle_ms": round(t_e2e / args.steps * 1e3, 4), "cycle_ms_dist": dist3(e2e_ms),
                "cycle_ms_p99_slowest_rank": round(e2e_p99_max_rank, 4),
                "ms_enumerate": round(enum_ms / args.steps, 5),
                "ms_encode": round(enc_ms / args.steps, 5), "response_bytes": len(wire),
                "stream_start_ms": round(stream_start_ms, 4),
                "heartbeat_to_kubelet_grpc_ms": None if grpc_ms is None or grpc_ms < 0 else round(grpc_ms, 4),
                "heartbeat_to_kubelet_native_daemon_ms": native_ms,
                "note": "no bulk host buffers exist on this path, so there is nothing to copy host->device: per step the host "
                        "passes kernel arguments and reads back the 48-byte result block the last CTA publishes into pinned "
                        "mapped memory plus the serialized response -- those %d bytes ARE the entire per-step result (the "
                        "device->host 'copy' is the GPU's own store, not a cudaMemcpy). The value leg brackets every kernel "
                        "with CUDA events (the roofline's clock); the kubelet-facing call completes on the published result "
                        "block alone. heartbeat_to_kubelet_native_daemon_ms is one daemon over all %d GPU(s)."
                        % (48 + len(wire), n)},
        "gpu_launches": args.steps * n,
        "unhealthy_verdicts": int(unhealthy),
        "health_floor": {"min_frac": 0.8, "calibrated_ceiling_gbs": round(gbs_ref, 1),
                         "frac_of_ceiling": dist3(fracs), "floor_gbs": round(0.8 * gbs_ref, 1),
                         "note": "Healthy needs >= 0.8 x the ceiling calibrated when the context opened (best warm pass, max over "
                                 "sibling GPUs); expected_checksum is the host's closed form"},
        "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "kernel_ms_mean": round(kernel_ms_mean, 5), "kernel_ms_mean_slowest_rank": round(kernel_ms_max_rank, 5),
                     "kernel_ms_dist": dist3(kernel_ms, 5),
                     "driver_d2d_copy_gbs_same_run": None if drv_copy_gbs is None else round(drv_copy_gbs, 1),
                     "note": "driver_d2d_copy = torch copy_ of the same 1 GiB (best of 20, CUDA events): the mixed read+write ceiling of this part; the probe verifies and re-keys every word at that rate"},
        "single_process": sp, "p2p": p2p, "parity": parity,
        "clocks": clocks,
    }
    # the reference's own sysfs/kfd CPU path on this box's host cores, in the same run, at every N
    # (C port of the Go walk on a synthetic N-device kfd tree in /dev/shm; single thread like the
    # reference's single goroutine): ~0.2 s of CPU work
    start_ms, beat_ms = kfd_walk_baseline(n)
    line["reference_cpu_path"] = {"kfd_walk_stream_start_ms": round(start_ms, 4), "kfd_walk_heartbeat_ms": round(beat_ms, 4),
                                  "n_devices": n, "threads": 1, "host_cores": os.cpu_count(), "kind": "port"}
    threads = os.cpu_count() or 1
    cpu_gbs, passes, dt = cpu_probe_baseline(threads, budget_s=6.0 if n == 1 else 3.0)
    line["cpu_baseline"] = {"value": round(cpu_gbs, 2), "unit": UNIT, "cores": threads, "kind": "port",
                            "sample": "the 1 GiB probe buffer of ONE device, %d passes in %.1f s, host DRAM, %d threads" % (passes, dt, threads),
                            "cycle_ms_kfd_walk": round(start_ms, 4), "kfd_walk_heartbeat_ms": round(beat_ms, 4)}
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    rg.close()
    bad = [k for k, v in (parity or {}).items() if v is False]
    if bad:
        raise SystemExit("parity FAILED against the oracle: %s" % ", ".join(bad))


if __name__ == "__main__":
    main()
