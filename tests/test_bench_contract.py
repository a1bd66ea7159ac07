"""bench.py's reference arm runs on CPU, so its JSON contract is checked here on every round: one line on
stdout, the keys the driver reads, and the product arm refusing to run without a GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "health_probe_hbm_gbs" and d["unit"] == "GB/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data"):
        assert k in d, k
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["n_gpus"] == 1
    assert "workload" in d["config"] and "model" not in d["config"]
    # the two arms print the SAME config object (the driver compares them)
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.bench_config(1)
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"] > 0
    assert cb["cycle_ms_kfd_walk"] > 0 and "the full buffer" in cb["sample"]
    e = d["e2e"]
    assert (e["value"], e["unit"], e["h2d_bytes_per_step"], e["d2h_bytes_per_step"]) == (d["value"], d["unit"], 0, 0)


def test_product_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_pass(tmp_path):
    """--dump-outputs writes what the value leg's last timed pass returned.  The measured context runs exactly --warmup
    passes and then --steps timed ones, so that pass verified the seed W+K-1 steps after the initial one whatever the
    warm-up's time floor did, and its results and the buffer it re-keyed equal the oracle's."""
    import numpy as np
    from oracle import probe as oprobe
    sys.path.insert(0, ROOT)
    import bench
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "4", "--warmup", "3",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 4 and d["warmup"] == 3 and d["single_process"]["cycles"] == 4
    assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20

    def load(name):
        a = np.load(out / (name + ".npy"))
        assert a.dtype == np.float64
        return a

    def u64(name):
        return [int(hi) << 32 | int(lo) for hi, lo in load(name)]
    seed = oprobe.initial_seed(0)
    for _ in range(3 + 4 - 1):
        seed = oprobe.next_seed(seed)
    n_words = bench.S_BYTES // 4
    assert load("probe_seed").tolist() == [seed]
    assert u64("probe_checksum") == u64("probe_expected_checksum") == [oprobe.expected_checksum(n_words, seed)]
    assert (u64("probe_mismatches"), u64("probe_first_bad_word"), u64("probe_bytes")) == ([0], [oprobe.NO_BAD], [2 * bench.S_BYTES])
    assert load("probe_healthy").tolist() == [1.0] and load("probe_err").tolist() == [0.0]
    assert load("list_and_watch_healthy").tolist() == [1.0]
    want = np.concatenate([oprobe.pattern(bench.DUMP_CHUNK_WORDS, oprobe.next_seed(seed), w) for w in bench.dump_chunks()])
    assert np.array_equal(load("probe_buffer_sample"), want.astype(np.float64))


def test_product_never_imports_links_or_executes_the_oracle():
    """oracle/ is test infrastructure: only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
    --impl reference legs may touch it.  The package, its native sources, the tools and the headers must not."""
    import re
    pat = re.compile(r"^\s*(from\s+oracle\b|import\s+oracle\b)|#include\s+[\"<][^\">]*oracle/|dlopen\([^)]*oracle|oracle/_build", re.M)
    offenders = []
    for top in ("k8s-device-plugin_b200", "tools", "include"):
        for dirpath, dirnames, files in os.walk(os.path.join(ROOT, top)):
            dirnames[:] = [d for d in dirnames if d not in ("build", "__pycache__")]
            for f in files:
                if not f.endswith((".py", ".cpp", ".cu", ".cuh", ".hpp", ".h", ".inc")):
                    continue
                p = os.path.join(dirpath, f)
                if pat.search(open(p, errors="replace").read()):
                    offenders.append(os.path.relpath(p, ROOT))
    assert offenders == []
    # bench.py: the oracle appears only inside the CPU-baseline / reference-arm functions
    src = open(os.path.join(ROOT, "bench.py")).read()
    for m in re.finditer(r"^\s*from oracle import (\w+)", src, re.M):
        head = src[:m.start()]
        func = re.findall(r"^def (\w+)\(", head, re.M)[-1]
        # parity_block: the untimed product-vs-oracle checker leg that runs after every timed region
        assert func in ("cpu_probe_baseline", "kfd_walk_baseline", "run_reference", "parity_block"), func


def test_reference_arm_does_not_load_the_product():
    """The CPU arm must not import the product package or map libb200dp.so (the driver records the .so files each arm
    loads): run it under a tracer that lists the shared objects mapped at exit."""
    code = ("import sys, runpy\n"
            "sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '1']\n"
            "try:\n    runpy.run_path(%r, run_name='__main__')\nexcept SystemExit:\n    pass\n"
            "maps = open('/proc/self/maps').read()\n"
            "sys.stderr.write('PRODUCT_SO=%%d\\n' %% ('libb200dp' in maps))\n"
            "sys.stderr.write('PRODUCT_PKG=%%d\\n' %% any(m.startswith('k8s-device-plugin_b200') for m in sys.modules))\n"
            % os.path.join(ROOT, "bench.py"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert "PRODUCT_SO=0" in r.stderr and "PRODUCT_PKG=0" in r.stderr, r.stderr[-2000:]


def test_reference_arm_under_torchrun_prints_once():
    """N>1: the driver launches both arms with torchrun; in the CPU arm rank 0 alone works and prints, the other rank
    exits 0 without a line."""
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["config"]["n_devices"] == 2 and d["value"] > 0


def test_file_flag_releases_the_waiting_ranks(tmp_path, monkeypatch):
    """bench.py's rank-0-alone leg: the other ranks sleep on a file, not on an NCCL barrier."""
    import threading
    import time
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setenv("MASTER_PORT", "29534")
    monkeypatch.setenv("TORCHELASTIC_RUN_ID", "t%d" % os.getpid())
    a, b = bench.FileFlag(), bench.FileFlag()
    assert a.path == b.path
    a.clear()
    t0 = time.time()
    th = threading.Thread(target=lambda: (time.sleep(0.2), a.set()))
    th.start()
    b.wait(timeout=10)
    th.join()
    assert 0.15 < time.time() - t0 < 5
    a.clear()
    import pytest
    with pytest.raises(SystemExit):
        b.wait(timeout=0.1)
