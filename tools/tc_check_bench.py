"""Measures the tensor-core check (b2dp_compute_check) on the GPUs of this node and writes one JSON file:

  - the card's name, power limit and max SM clock (nvidia-smi, query only), read in the same run as the numbers;
  - per tile count: event-timed ms of one check (bf16 + e4m3 launches) over --checks checks after --warmup, per GPU;
  - FLOPs from the shapes, 2*128*128*128 per tile per kind per CTA, and the rate over the event time;
  - the share of the data sheet's dense peak (2,250 TFLOP/s bf16, 4,500 fp8 per GPU): the least time the two launches
    could take at those rates over the measured time -- a share, not a rate reached;
  - the one-process ListAndWatch heartbeat over all GPUs, p50/p99, for a compute=0 and a compute=1 context, the two
    alternating cycle by cycle in one run.

    python tools/tc_check_bench.py --out profiles/r03_tc_check_b200.json
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

PEAK_TFLOPS = {"bf16": 2250.0, "e4m3": 4500.0}   # HGX B200 data sheet, one GPU, dense
FLOP_PER_TILE = 2 * 128 * 128 * 128


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    rows = [[x.strip() for x in line.split(",")] for line in r.stdout.strip().splitlines()]
    return [{"index": int(x[0]), "name": x[1], "power_limit": x[2], "clocks_max_sm": x[3]} for x in rows if len(x) == 4]


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(q * (len(v) - 1) + 0.5))] if v else 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--checks", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--tiles", default="1,2,4,8,16,32,64")
    ap.add_argument("--cycles", type=int, default=300)
    ap.add_argument("--bytes", type=int, default=1 << 30)
    a = ap.parse_args()
    pkg = importlib.import_module("k8s-device-plugin_b200")
    N = pkg._native
    out = {"tool": "tools/tc_check_bench.py", "gpus": card(), "checks": a.checks, "warmup": a.warmup,
           "flop_per_tile_per_kind": FLOP_PER_TILE, "peak_tflops_datasheet": PEAK_TFLOPS, "by_tiles": []}
    with pkg.Context("cuda:bytes=%d,calib=0" % (1 << 20)) as ctx:
        n = len(ctx.enumerate())
        out["n_gpus"] = n
        for tiles in [int(t) for t in a.tiles.split(",")]:
            for _ in range(a.warmup):
                ctx.compute_check(tiles=tiles, timed=True)
            ms = [[] for _ in range(n)]
            ms_dev = [[] for _ in range(n)]
            res = []
            for _ in range(a.checks):
                res = ctx.compute_check(tiles=tiles, timed=True)
                assert all(r.healthy for r in res), res
                for i, r in enumerate(res):
                    ms[i].append(r.ms_event)
                    ms_dev[i].append(r.ms_device)
            per_gpu = []
            for i, r in enumerate(res):
                ctas = r.sms_covered
                flops_kind = FLOP_PER_TILE * tiles * r.sms                  # one kind, every CTA
                t = pct(ms[i], 0.5)
                t_min_s = flops_kind / (PEAK_TFLOPS["bf16"] * 1e12) + flops_kind / (PEAK_TFLOPS["e4m3"] * 1e12)
                per_gpu.append({"device": i, "sms": r.sms, "sms_covered": ctas, "tiles_total": r.tiles,
                                "ms_event_p50": t, "ms_event_p99": pct(ms[i], 0.99), "ms_event_min": min(ms[i]),
                                "ms_device_p50": pct(ms_dev[i], 0.5),
                                "flops": 2 * flops_kind, "tflops": 2 * flops_kind / (t * 1e-3) * 1e-12 if t > 0 else 0.0,
                                "share_of_datasheet_dense_peak": t_min_s / (t * 1e-3) if t > 0 else 0.0})
            out["by_tiles"].append({"tiles": tiles, "per_gpu": per_gpu})
            print("tiles %3d: ms p50 %s" % (tiles, " ".join("%.4f" % g["ms_event_p50"] for g in per_gpu)), flush=True)

    # the heartbeat with and without the check, alternating in one run
    buf = (C.c_uint8 * (1 << 16))()
    ln = C.c_size_t()
    lw = {0: [], 1: []}
    ctxs = {c: pkg.Context("cuda:bytes=%d,compute=%d" % (a.bytes, c)) for c in (0, 1)}
    try:
        for c, ctx in ctxs.items():
            ctx.list_and_watch("gpu", N.LW_INITIAL)
        for k in range(a.cycles + 20):
            for c, ctx in ctxs.items():
                opts = N.CycleOpts()
                opts.flags = N.LW_HEARTBEAT
                st = N.CycleStats()
                t0 = time.perf_counter()
                rc = N.lib.b2dp_list_and_watch(ctx._h, b"gpu", C.byref(opts), buf, len(buf), C.byref(ln), C.byref(st))
                dt = (time.perf_counter() - t0) * 1e3
                assert rc == 0 and st.n_unhealthy == 0, (rc, st.n_unhealthy)
                if k >= 20:
                    lw[c].append(dt)
    finally:
        for ctx in ctxs.values():
            ctx.close()
    out["list_and_watch"] = {"bytes": a.bytes, "cycles": a.cycles,
                             "compute0_ms_p50": pct(lw[0], 0.5), "compute0_ms_p99": pct(lw[0], 0.99),
                             "compute1_ms_p50": pct(lw[1], 0.5), "compute1_ms_p99": pct(lw[1], 0.99)}
    print(json.dumps(out["list_and_watch"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
