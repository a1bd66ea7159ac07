"""Writes tc_check_vectors.json: the tensor-core check's specification (oracle/tc_check.py) pinned for a few seeds --
operand and product rows (the first and last 8) of one combination per seed, and the full row-hash table.

    python tests/golden/make_tc_vectors.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import tc_check as tc  # noqa: E402

SEEDS = [tc.seed_for(0), tc.seed_for(7), 0xDEADBEEF]
ROWS = list(range(8)) + list(range(tc.M - 8, tc.M))


def main():
    out = {"M": tc.M, "N": tc.N, "K": tc.K, "nsets": tc.NSETS, "seeds": []}
    for i, seed in enumerate(SEEDS):
        a_set, b_set = i % tc.NSETS, (i + 1) % tc.NSETS
        a = tc.operand(seed, "a", a_set)
        b = tc.operand(seed, "b", b_set)
        c = tc.exact_c(a, b)
        out["seeds"].append({
            "seed": seed,
            "a_set": a_set, "b_set": b_set,
            "rows": ROWS,
            "a": a[ROWS].tolist(), "b": b[ROWS].tolist(), "c": c[ROWS].tolist(),
            "a_bf16_row0": [int(x) for x in tc.encode(a[0], tc.KIND_BF16)],
            "a_e4m3_row0": [int(x) for x in tc.encode(a[0], tc.KIND_E4M3)],
            "row_hash": [[str(int(h)) for h in row] for row in tc.expected_table(seed)],
        })
    with open(os.path.join(HERE, "tc_check_vectors.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")


if __name__ == "__main__":
    main()
