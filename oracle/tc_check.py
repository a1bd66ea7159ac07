"""Specification of the tensor-core health check (csrc/tc_check.cuh, csrc/tc_math.hpp), in numpy.

Every CTA of the check runs T tiles; a tile is one M=128, N=128, K=128 accumulation chain C = A . B^T on the tensor
cores (tcgen05.mma, fp32 accumulator in tensor memory) over one (A_i, B_j) pair of a small operand pool: NSETS A tiles
and NSETS B tiles, both K-major (row r of A and row n of B each hold K contiguous values).

Operands are integers in [-7, 7]: bf16 and e4m3 both hold them exactly, every partial sum is an integer with
|x| <= K * 49 = 6272 < 2^13, so fp32 holds every partial sum exactly and the result does not depend on the order (or
the internal width) of the accumulation.  A mismatch is a fault, never rounding.  Keep K * 7 * 7 < 2^24 (and the
accumulator-width margin, < 2^13) if K or the range changes.

The device folds each accumulator row into an order-independent 64-bit row hash and compares it with the host's.
"""
import numpy as np

M = N = K = 128
NSETS = 3                     # A tiles and B tiles in the pool
NCOMB = NSETS * NSETS         # (A_i, B_j) combinations
VMAX = 7
KIND_BF16, KIND_E4M3 = 0, 1
KINDS = (KIND_BF16, KIND_E4M3)
GOLD = 0x9E3779B9
SALT2 = 0x7F4A7C15
SALT3 = 0x5BD1E995
M32 = 0xFFFFFFFF


def mix32(x):
    """murmur3 fmix32 on uint32 arrays (a bijection of 32-bit words)."""
    x = np.asarray(x, dtype=np.uint64) & M32
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x85EBCA6B)) & np.uint64(M32)
    x ^= x >> np.uint64(13)
    x = (x * np.uint64(0xC2B2AE35)) & np.uint64(M32)
    x ^= x >> np.uint64(16)
    return x


def seed_for(index: int) -> int:
    """The pool seed of the device at enumeration index `index`."""
    return (0x7C5E0000 | (index & 0xFFFF)) & M32


def operand(seed: int, which: str, s: int) -> np.ndarray:
    """Tile `s` of the A pool (which='a') or B pool (which='b'): int64 [128, 128] in [-7, 7], row-major = K-major.

    value(seed, set_id, r, k) = mix32(((set_id * 128 + r) * 128 + k) * GOLD ^ seed) % 15 - 7, set_id = s (A), 3 + s (B)."""
    set_id = s if which == "a" else NSETS + s
    idx = (np.uint64(set_id * M) + np.arange(M, dtype=np.uint64)[:, None]) * np.uint64(K) + np.arange(K, dtype=np.uint64)[None, :]
    h = mix32(((idx * np.uint64(GOLD)) & np.uint64(M32)) ^ np.uint64(seed))
    return (h % np.uint64(2 * VMAX + 1)).astype(np.int64) - VMAX


def combination(smid: int, check: int, tile: int):
    """The (a_set, b_set) tile `tile` of the CTA on SM `smid` uses in check number `check` (0, 1, ...): every SM meets
    every combination within NCOMB consecutive checks."""
    c = (smid + check + tile) % NCOMB
    return c // NSETS, c % NSETS


def exact_c(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """C = A . B^T in int64 (exact)."""
    return a.astype(np.int64) @ b.astype(np.int64).T


def fp32_bits(c: np.ndarray) -> np.ndarray:
    """The fp32 bit patterns of an integer matrix (exact for |x| < 2^24)."""
    assert np.abs(c).max(initial=0) < (1 << 24)
    return c.astype(np.float32).view(np.uint32).astype(np.uint64)


def row_hash(bits: np.ndarray) -> np.ndarray:
    """Order-independent 64-bit hash of each row of uint32 bit patterns [rows, cols]:
    sum_j ( mix32(b_j ^ j*GOLD) << 32 | mix32(b_j ^ (j*SALT2 ^ SALT3)) )  mod 2^64.
    Each term is a bijection of b_j, so one changed word always changes the hash."""
    bits = np.asarray(bits, dtype=np.uint64) & np.uint64(M32)
    j = np.arange(bits.shape[1], dtype=np.uint64)[None, :]
    hi = mix32(bits ^ ((j * np.uint64(GOLD)) & np.uint64(M32)))
    lo = mix32(bits ^ (((j * np.uint64(SALT2)) & np.uint64(M32)) ^ np.uint64(SALT3)))
    terms = (hi << np.uint64(32)) | lo
    with np.errstate(over="ignore"):
        return terms.sum(axis=1, dtype=np.uint64)


def expected(seed: int, kind: int, a_set: int, b_set: int) -> np.ndarray:
    """The 128 row hashes of tile (a_set, b_set).  Both kinds accumulate the same integers exactly, so `kind` does not
    change the answer; it is an argument so that the specification says so."""
    assert kind in KINDS
    return row_hash(fp32_bits(exact_c(operand(seed, "a", a_set), operand(seed, "b", b_set))))


def expected_table(seed: int) -> np.ndarray:
    """[NCOMB, 128] uint64: the hash table the device compares against, indexed by combination a_set*NSETS + b_set."""
    return np.stack([expected(seed, KIND_BF16, c // NSETS, c % NSETS) for c in range(NCOMB)])


def encode(v: np.ndarray, kind: int) -> np.ndarray:
    """Exact encodings of integers in [-7, 7]: bf16 (uint16) or e4m3 (uint8)."""
    v = np.asarray(v, dtype=np.int64)
    assert np.abs(v).max(initial=0) <= VMAX
    if kind == KIND_BF16:
        return (v.astype(np.float32).view(np.uint32) >> 16).astype(np.uint16)
    out = np.zeros(v.shape, dtype=np.uint8)
    for x in range(1, VMAX + 1):
        e = x.bit_length() - 1
        code = ((e + 7) << 3) | (((x << 3) >> e) & 7)
        out[v == x] = code
        out[v == -x] = code | 0x80
    return out


def flops_per_tile() -> int:
    return 2 * M * N * K
