"""Tensor-core check, the parts that need no GPU: the host reference (b2dp_compute_expected) equals the specification
(oracle/tc_check.py), which equals the pinned vectors; the new ABI structs have the layout the ctypes mirror assumes;
the option is validated before any GPU is touched; backends without in-process GPUs refuse the check; and the built
library's kernels are tcgen05 code without spills."""
import ctypes
import json
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import tc_check as otc

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
CSRC = os.path.join(REPO, "k8s-device-plugin_b200", "csrc")
SEEDS = (otc.seed_for(0), otc.seed_for(5), 0xDEADBEEF)


@pytest.fixture(scope="module")
def P(pkg):
    return pkg


def test_host_reference_equals_the_oracle(P):
    for seed in SEEDS:
        for kind in otc.KINDS:
            for a_set in range(otc.NSETS):
                for b_set in range(otc.NSETS):
                    got = P.compute_expected(seed, kind, a_set, b_set)
                    assert got.dtype == np.uint64 and got.shape == (otc.M,)
                    assert np.array_equal(got, otc.expected(seed, kind, a_set, b_set)), (hex(seed), kind, a_set, b_set)


def test_oracle_equals_the_golden_vectors():
    g = json.load(open(os.path.join(HERE, "golden", "tc_check_vectors.json")))
    assert (g["M"], g["N"], g["K"], g["nsets"]) == (otc.M, otc.N, otc.K, otc.NSETS)
    assert len(g["seeds"]) == 3
    for e in g["seeds"]:
        seed, rows = e["seed"], e["rows"]
        a = otc.operand(seed, "a", e["a_set"])
        b = otc.operand(seed, "b", e["b_set"])
        c = otc.exact_c(a, b)
        assert np.array_equal(a[rows], np.array(e["a"])) and np.array_equal(b[rows], np.array(e["b"]))
        assert np.array_equal(c[rows], np.array(e["c"]))
        assert [int(x) for x in otc.encode(a[0], otc.KIND_BF16)] == e["a_bf16_row0"]
        assert [int(x) for x in otc.encode(a[0], otc.KIND_E4M3)] == e["a_e4m3_row0"]
        assert otc.expected_table(seed).tolist() == [[int(h) for h in row] for row in e["row_hash"]]


def test_products_stay_exact():
    """|C| < 2^13 for every combination: exact in fp32 in any order and in a narrow accumulator."""
    assert otc.K * otc.VMAX * otc.VMAX < (1 << 13)
    for seed in SEEDS:
        for a_set in range(otc.NSETS):
            for b_set in range(otc.NSETS):
                c = otc.exact_c(otc.operand(seed, "a", a_set), otc.operand(seed, "b", b_set))
                assert np.abs(c).max() < (1 << 13)


def test_encodings_are_exact():
    v = np.arange(-otc.VMAX, otc.VMAX + 1)
    bf = otc.encode(v, otc.KIND_BF16).astype(np.uint32) << 16
    assert np.array_equal(bf.view(np.float32), v.astype(np.float32))
    e4 = otc.encode(v, otc.KIND_E4M3)
    sign = np.where(e4 & 0x80, -1.0, 1.0)
    exp = (e4 >> 3) & 0xF
    man = e4 & 7
    val = np.where(exp == 0, 0.0, sign * (1 + man / 8.0) * 2.0 ** (exp.astype(np.int64) - 7))
    assert np.array_equal(val, v.astype(np.float64))


def test_one_flipped_bit_changes_the_row_hash():
    bits = otc.fp32_bits(otc.exact_c(otc.operand(SEEDS[0], "a", 0), otc.operand(SEEDS[0], "b", 0)))
    h = otc.row_hash(bits)
    rng = np.random.default_rng(1)
    for _ in range(64):
        r, col, bit = rng.integers(otc.M), rng.integers(otc.N), rng.integers(32)
        b2 = bits.copy()
        b2[r, col] ^= np.uint64(1 << int(bit))
        h2 = otc.row_hash(b2)
        assert h2[r] != h[r] and np.array_equal(np.delete(h2, r), np.delete(h, r))
    # order-independent in evaluation, position-dependent in meaning: swapping two different columns changes it
    swapped = bits.copy()
    swapped[:, [0, 1]] = swapped[:, [1, 0]]
    differ = bits[:, 0] != bits[:, 1]
    assert np.all(otc.row_hash(swapped)[differ] != h[differ])


def test_expected_argument_checks(P):
    N = P._native
    out = np.zeros(128, dtype=np.uint64)
    n = ctypes.c_int()
    ptr = out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))
    assert N.lib.b2dp_compute_expected(1, 2, 0, 0, ptr, 128, ctypes.byref(n)) == N.E_INVAL
    assert N.lib.b2dp_compute_expected(1, 0, 3, 0, ptr, 128, ctypes.byref(n)) == N.E_INVAL
    assert N.lib.b2dp_compute_expected(1, 0, 0, -1, ptr, 128, ctypes.byref(n)) == N.E_INVAL
    assert N.lib.b2dp_compute_expected(1, 0, 0, 0, ptr, 127, ctypes.byref(n)) == N.E_NOSPC and n.value == 128


def test_struct_layouts_match_the_c_header(P, tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    N = P._native
    pairs = [("b2dp_compute_opts", N.ComputeOpts), ("b2dp_compute_result", N.ComputeResult)]
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "b200dp.h"', 'int main(void) {']
    for cname, ct in pairs:
        src.append('printf("%s %%zu", sizeof(%s));' % (cname, cname))
        for fname, _ in ct._fields_:
            src.append('printf(" %s=%%zu", offsetof(%s, %s));' % (fname, cname, fname))
        src.append('printf("\\n");')
    src.append('printf("%d %d %d\\n", B2DP_RES_COMPUTE, B2DP_COMPUTE_EVENT_TIMING, B2DP_COMPUTE_DEFAULT_TILES);')
    src += ['return 0; }']
    c = tmp_path / "layout.c"
    c.write_text("\n".join(src))
    exe = str(tmp_path / "layout")
    r = subprocess.run(["gcc", "-std=c11", "-I", os.path.join(REPO, "include"), str(c), "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([exe], capture_output=True, text=True).stdout.splitlines()
    for line, (cname, ct) in zip(out, pairs):
        parts = line.split()
        assert parts[0] == cname and int(parts[1]) == ctypes.sizeof(ct), (cname, parts[1], ctypes.sizeof(ct))
        for tok, (fname, _) in zip(parts[2:], ct._fields_):
            k, v = tok.split("=")
            assert k == fname and int(v) == getattr(ct, fname).offset, (cname, fname, v)
    assert out[2].split() == [str(N.RES_COMPUTE), str(N.COMPUTE_EVENT_TIMING), str(N.COMPUTE_DEFAULT_TILES)]
    assert ctypes.sizeof(N.ProbeResult) == 88 and ctypes.sizeof(N.CycleStats) == 64
    assert N.lib.b2dp_abi_version() == 3


@pytest.mark.parametrize("value", ["2", "x", "", "yes"])
def test_compute_option_is_validated_before_any_gpu(P, value):
    with pytest.raises(P._native.B2dpError) as e:
        P.Context("cuda:devices=0,compute=%s" % value)
    assert e.value.code == P._native.E_INVAL and "compute=" in str(e.value)


def _unsupported(P, ctx):
    with pytest.raises(P._native.B2dpError) as e:
        ctx.compute_check()
    assert e.value.code == P._native.E_UNSUPPORTED
    for call in (lambda: ctx.compute_tile(0, 0, 0, 0), lambda: ctx.compute_inject_fault(0, 0, 1)):
        with pytest.raises(P._native.B2dpError) as e:
            call()
        assert e.value.code == P._native.E_UNSUPPORTED


def test_synthetic_backend_refuses_the_check(P):
    with P.Context("synthetic:2") as ctx:
        _unsupported(P, ctx)


def test_kfd_fixture_refuses_the_check(P, tmp_path):
    for d in ("sys/module/amdgpu/drivers", "sys/class/kfd/kfd/topology/nodes"):
        (tmp_path / d).mkdir(parents=True)
    with P.Context("kfd:%s" % tmp_path) as ctx:
        _unsupported(P, ctx)


@pytest.fixture(scope="module")
def nvml_stub():
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    build = os.path.join(HERE, "native", "_build")
    os.makedirs(build, exist_ok=True)
    out = os.path.join(build, "libnvml_stub_tc%d.so" % os.getpid())
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-shared", "-fPIC", "-fvisibility=hidden",
                        os.path.join(HERE, "native", "nvml_stub.cpp"), "-o", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    yield out
    os.remove(out)


def test_nvml_backend_refuses_the_check(P, monkeypatch, nvml_stub, tmp_path):
    monkeypatch.setenv("B2DP_NVML_LIBRARY", nvml_stub)
    monkeypatch.setenv("B2DP_NVML_STUB", "gpus=2,mig=0")
    (tmp_path / "sys/module/nvidia").mkdir(parents=True)
    with P.Context("nvml:sysroot=%s,compute=1" % tmp_path) as ctx:
        assert len(ctx.enumerate()) == 2
        _unsupported(P, ctx)


def _objects():
    lib = os.path.join(REPO, "k8s-device-plugin_b200", "libb200dp.so")
    log = os.path.join(CSRC, "build", "cuda_backend.ptxas.log")
    if not os.path.exists(lib) or not os.path.exists(log):
        pytest.skip("library not built")
    return lib, log


def test_kernels_are_tcgen05_code():
    lib, _ = _objects()
    if shutil.which("cuobjdump") is None and not os.path.exists("/usr/local/cuda/bin/cuobjdump"):
        pytest.skip("no cuobjdump")
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    sass = subprocess.run([exe, "-sass", lib], capture_output=True, text=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)
    tc = {f.split("\n", 1)[0].strip(): f for f in funcs if "tc_check" in f.split("\n", 1)[0]}
    assert len(tc) == 2, list(tc)
    bf16 = [body for name, body in tc.items() if "ILi0E" in name][0]
    e4m3 = [body for name, body in tc.items() if "ILi1E" in name][0]
    assert "UTCHMMA" in bf16 and "UTCQMMA" in e4m3
    for body in tc.values():
        assert "LDTM" in body and not re.search(r"\bHMMA\b", body)


def test_kernels_do_not_spill():
    _, log = _objects()
    text = open(log).read()
    blocks = re.split(r"ptxas info\s*: Compiling entry function", text)
    tc = [b for b in blocks if "tc_check" in b.split("\n", 1)[0]]
    assert len(tc) == 2
    for b in tc:
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", b)
        assert m and m.groups() == ("0", "0"), b
