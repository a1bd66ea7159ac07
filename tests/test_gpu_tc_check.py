"""Tensor-core check on a B200 (run with -m gpu): the tcgen05 tiles equal the oracle's exact product bit for bit, a full
check covers every SM and verifies, injected wrong products are attributed to the SM that made them, and the verdict
reaches probe_health and ListAndWatch through compute=1.  The oracle is oracle/tc_check.py."""
import numpy as np
import pytest

from oracle import tc_check as otc

pytestmark = pytest.mark.gpu

MiB = 1 << 20


@pytest.fixture(scope="module")
def P(pkg):
    return pkg


def _bits(mask):
    return [s for s in range(256) if (mask >> s) & 1]


def _heartbeat_health(P, ctx):
    wire, _ = ctx.list_and_watch("gpu", P._native.LW_HEARTBEAT)
    return [d.health for d in P.v1beta1.ListAndWatchResponse.FromString(wire).devices]


@pytest.mark.parametrize("kind", [otc.KIND_BF16, otc.KIND_E4M3])
def test_tile_parity_bit_exact(P, kind):
    """compute_tile returns the raw fp32 accumulator: it equals the oracle's exact C for every (A, B) combination."""
    with P.Context("cuda:devices=0,bytes=%d,calib=0" % MiB) as ctx:
        (r,) = ctx.compute_check()
        seed = r.seed
        assert seed == otc.seed_for(0)
        for a_set in range(otc.NSETS):
            for b_set in range(otc.NSETS):
                c = ctx.compute_tile(0, kind, a_set, b_set)
                want = otc.exact_c(otc.operand(seed, "a", a_set), otc.operand(seed, "b", b_set)).astype(np.float32)
                assert np.array_equal(c.view(np.uint32), want.view(np.uint32)), (kind, a_set, b_set)
                assert np.array_equal(otc.row_hash(c.view(np.uint32)), otc.expected(seed, kind, a_set, b_set))


def test_full_check_one_gpu(P):
    with P.Context("cuda:devices=0,bytes=%d,calib=0" % MiB) as ctx:
        sms = ctx.probe_describe(0)["sm_count"]
        for tiles in (0, 1, 37):
            (r,) = ctx.compute_check(tiles=tiles, timed=True)
            t = tiles or P._native.COMPUTE_DEFAULT_TILES
            assert r.err == 0 and r.healthy, r
            assert r.bad_rows == 0 and r.sms_failed == 0 and r.first_bad_sm == -1 and r.bad_sm_mask == 0
            assert r.sms == sms and r.sms_covered == sms and bin(r.covered_mask).count("1") == sms
            assert r.tiles == 2 * t * sms
            assert r.ms_device > 0 and r.ms_event > 0 and r.tflops > 0


def test_attribution_to_the_faulty_sm(P):
    with P.Context("cuda:devices=0,bytes=%d,calib=0" % MiB) as ctx:
        (r,) = ctx.compute_check()
        smids = _bits(r.covered_mask)
        for sm in (smids[0], smids[len(smids) // 2], smids[-1]):
            ctx.compute_inject_fault(0, sm, 0x1)
            (r,) = ctx.compute_check()
            assert r.err == 0 and not r.healthy
            assert r.bad_sm_mask == 1 << sm and r.sms_failed == 1 and r.first_bad_sm == sm
            assert (r.first_bad_kind, r.first_bad_tile, r.first_bad_row, r.bad_rows) == (0, 0, 0, 1)
            (r,) = ctx.compute_check()                  # one-shot: the next check is clean
            assert r.healthy and r.bad_rows == 0


def test_heartbeat_verdict_with_compute(P):
    nbytes = 8 * MiB
    with P.Context("cuda:devices=0,bytes=%d,calib=0,compute=1" % nbytes) as ctx:
        (r,) = ctx.probe_health(min_gbs=1e-3)
        assert r.healthy and not (r.flags & P._native.RES_COMPUTE), r
        ctx.list_and_watch("gpu", P._native.LW_INITIAL)
        assert _heartbeat_health(P, ctx) == ["Healthy"]
        (c,) = ctx.compute_check()
        ctx.compute_inject_fault(0, _bits(c.covered_mask)[0], 0x80000000)
        (r,) = ctx.probe_health(min_gbs=1e-3)
        assert not r.healthy and (r.flags & P._native.RES_COMPUTE) and r.mismatches == 0, r
        assert r.checksum == r.expected_checksum
        (r,) = ctx.probe_health(min_gbs=1e-3)              # reported once: the next pass runs fresh
        assert r.healthy and not (r.flags & P._native.RES_COMPUTE)
        ctx.compute_inject_fault(0, _bits(c.covered_mask)[-1], 0x4)
        assert _heartbeat_health(P, ctx) == ["Unhealthy"]
        assert _heartbeat_health(P, ctx) == ["Healthy"]


def test_multi_gpu_injection_fails_only_that_device(P):
    with P.Context("cuda:bytes=%d,calib=0,compute=1" % (8 * MiB)) as ctx:
        n = len(ctx.enumerate())
        res = ctx.compute_check()
        assert len(res) == n and all(r.healthy and r.sms_covered == r.sms for r in res)
        assert len({r.seed for r in res}) == n
        victim = n - 1
        ctx.compute_inject_fault(victim, _bits(res[victim].covered_mask)[0], 0x10)
        res = ctx.compute_check()
        assert [r.healthy for r in res] == [i != victim for i in range(n)]
        ctx.compute_inject_fault(victim, _bits(res[victim].covered_mask)[0], 0x10)
        pr = ctx.probe_health(min_gbs=1e-3)
        assert [r.healthy for r in pr] == [i != victim for i in range(n)]
        assert [bool(r.flags & P._native.RES_COMPUTE) for r in pr] == [i == victim for i in range(n)]


def test_compute_with_prearm_never_arms(P):
    with P.Context("cuda:devices=0,bytes=%d,calib=0,compute=1,prearm=1" % (8 * MiB)) as ctx:
        for _ in range(4):
            (r,) = ctx.probe_health(min_gbs=1e-3, timed=False)
            assert r.healthy and not (r.flags & (P._native.RES_PREARMED | P._native.RES_COMPUTE)), r


def test_compute_through_helpers_on_whole_gpus(P):
    with P.Context("cuda:probe=helpers,bytes=%d,calib=0,compute=1" % (8 * MiB)) as ctx:
        res = ctx.probe_health(min_gbs=1e-3)
        assert res and all(r.healthy and not (r.flags & P._native.RES_COMPUTE) for r in res), res
        with pytest.raises(P._native.B2dpError) as e:
            ctx.compute_check()
        assert e.value.code == P._native.E_UNSUPPORTED


def test_compute_off_never_sets_the_flag(P):
    with P.Context("cuda:devices=0,bytes=%d,calib=0" % (8 * MiB)) as ctx:
        (c,) = ctx.compute_check()
        ctx.compute_inject_fault(0, _bits(c.covered_mask)[0], 0x1)   # pending, but compute=0 passes never run a check
        for _ in range(2):
            (r,) = ctx.probe_health(min_gbs=1e-3)
            assert r.healthy and not (r.flags & P._native.RES_COMPUTE)
