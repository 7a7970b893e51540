"""Generate tests/golden/withdrawal.npz by running the REFERENCE itself (authoring container only).

    PYTHONPATH=oracle/pyshim:/root/reference/src python tests/golden/gen_golden_withdrawal.py

480 verdicts of the reference's withdrawal_circuit.verify_circuit in 12 scenarios (see withdrawal_cases below); the
file layout and the mutations are in tests/withdrawal_cases.py.  The shared helpers (limbs, to_matrix, corrupt_value,
n_of) are the other golden files' (gen_golden.py).  Seeded: an unchanged reference gives a byte-identical file.
/root/reference does not exist on the GPU box, so tests only ever read the .npz file.
"""
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from gen_golden import P, corrupt_value, limbs, n_of, to_matrix  # noqa: E402


def withdrawal_cases():
    """The reference's withdrawal_circuit.verify_circuit (withdrawal_circuit.py:127-201) run UNMODIFIED on witnesses built
    like its tests (tests/test_withdrawal_circuit.py: withdrawals2witness, mock_mpt_update with root = prev + 5, one
    WithdrawalRoot block row) plus hand-built padded witnesses (a Row with amount 0, a continuing id and a
    NonExistingAccountProof MPT row), field-edge values (id = p - 1, fields of 0 / below 128 / 32 bytes, a payload of 56
    bytes and more) and MAX_WITHDRAWALS of 0, 1, below, equal to and above len(rows).  Vectors: single-cell corruptions
    of rows and of every table, dropped table rows, a duplicated block row with another block_number, hash halves of
    2^128 and more.  The failing row is the loop's row_index when the exception left verify_circuit (MAX - 1 for the
    block lookup after the loop; 0 when the loop is empty)."""
    sys.path.insert(0, os.path.dirname(HERE))
    import rlp
    import withdrawal_cases as wc
    from eth_utils import keccak
    from zkevm_specs import withdrawal_circuit as wdc
    from zkevm_specs.evm_circuit.table import BlockContextFieldTag, BlockTableRow, MPTProofType, MPTTableRow
    from zkevm_specs.util import FQ, Word, WordOrValue

    r = FQ(0x2718281828459045235360287471352662497757247093699959574966967627 % P)
    rng = random.Random(31)

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def halves(v):
        return [v & ((1 << 128) - 1), v >> 128]

    def build(wds, n_pad=0, pad_style="continuing"):
        """wds: [(id, validator_id, address, amount)] -> cells of rows / keccak / mpt / block (sorted table rows)"""
        rows, K, M = [], {(0, 0, 0, 0, 0)}, set()
        prev = 0
        for (i, v, a, m) in wds:
            enc = rlp.encode([i, v, a, m])
            h = keccak(enc)
            K.add((1, n_of(wdc.RLC(bytes(reversed(enc)), r, n_bytes=len(enc)).expr()), len(enc),
                   int.from_bytes(h[:16], "little"), int.from_bytes(h[16:], "little")))
            root = prev + 5
            hw = [int.from_bytes(h[:16], "little"), int.from_bytes(h[16:], "little")]
            M.add((a, int(MPTProofType.WithdrawalMod), *halves(i), *halves(root), *halves(prev), *hw, 0, 0))
            rows.append([i, v, a, m, *hw, *halves(root)])
            prev = root
        last_id = wds[-1][0] if wds else 0
        for k in range(n_pad):
            pid = (last_id + 1 + k) % P if pad_style == "continuing" else 0
            rows.append([pid, 0, 0, 0, 0, 0, *halves(prev)])
            M.add((0, int(MPTProofType.NonExistingAccountProof), *halves(pid), *halves(prev), *halves(prev), 0, 0, 0, 0))
        B = [[int(BlockContextFieldTag.WithdrawalRoot), 0, *halves(prev)]]
        return {"rows": to_matrix(rows) if rows else np.zeros((8, 0, 4), dtype=np.uint64),
                "keccak": to_matrix(sorted(K)), "mpt": to_matrix(sorted(M)), "block": to_matrix(B)}

    def cells_of(a):
        return [[sum(int(a[c, i, k]) << (64 * k) for k in range(4)) for c in range(a.shape[0])] for i in range(a.shape[1])]

    def run(w, MAX):
        rows = [wdc.Row(FQ(c[0]), FQ(c[1]), FQ(c[2]), FQ(c[3]), W(c[4], c[5]), W(c[6], c[7])) for c in cells_of(w["rows"])]
        kt = wdc.KeccakTable()
        kt.table = set((FQ(c[0]), FQ(c[1]), FQ(c[2]), W(c[3], c[4])) for c in cells_of(w["keccak"]))
        mt = wdc.MPTTable(set(MPTTableRow(FQ(c[0]), FQ(c[1]), W(c[2], c[3]), W(c[4], c[5]), W(c[6], c[7]), W(c[8], c[9]),
                                          W(c[10], c[11])) for c in cells_of(w["mpt"])))
        bt = wdc.BlockTable(set(BlockTableRow(FQ(c[0]), FQ(c[1]), WordOrValue(W(c[2], c[3]))) for c in cells_of(w["block"])))
        try:
            wdc.verify_circuit(wdc.Witness(rows, mt, kt, bt), MAX, r)
        except Exception as e:  # noqa: BLE001
            tb, row = e.__traceback__, None
            while tb is not None:
                if tb.tb_frame.f_code.co_name == "verify_circuit" and "row_index" in tb.tb_frame.f_locals:
                    row = tb.tb_frame.f_locals["row_index"]
                tb = tb.tb_next
            return (0 if row is None else row), type(e).__name__
        return -1, ""

    def gen_wds(n, id0=None, big=False):
        id0 = rng.randrange(0, 1 << 64) if id0 is None else id0
        out = []
        for k in range(n):
            if big:
                out.append(((id0 + k) % P, rng.randrange(1 << 248, P), rng.randrange(1 << 248, P), rng.randrange(1 << 248, P)))
            else:
                out.append(((id0 + k) % P, rng.randrange(0, 1 << 64), rng.randrange(1, 1 << 160), rng.randrange(1, 1 << 64)))
        return out

    base5 = gen_wds(5)
    edge = [(P - 2, 0, 0, 1), (P - 1, 127, 128, 0x7F), (0, P - 1, (1 << 160) - 1, P - 1), (1, 255, 1, 256)]
    scen = [  # (name, witness, MAX, corruptions)
        ("basic", build(base5), 5, 140),                      # test_withdrawal_basic and its four corruption tests
        ("amount_max2", build(gen_wds(2)), 2, 40),            # test_withdrawal_inconsistent_amount
        ("padded", build(gen_wds(3), n_pad=2), 5, 80),
        ("padded_id0", build(gen_wds(3), n_pad=2, pad_style="zero"), 5, 10),
        ("field_edges", build(edge), 4, 80),
        ("payload56", build(gen_wds(3, big=True)), 3, 50),
        ("max0", build(base5), 0, 15),
        ("max1", build(base5[:1]), 1, 15),
        ("max_below_len", build(base5), 3, 15),
        ("max_above_len", build(base5), 7, 15),
        ("empty_max0", build([]), 0, 0),
        ("empty_max2", build([]), 2, 0),
    ]
    # the reference's four corruption tests on the basic witness: rows[1].id -= 1, rows[0].id = 999,
    # rows[0].validator_id = 999, rows[0].address = 0xDEADBEEF
    b = cells_of(scen[0][1]["rows"])
    fixed = {"basic": [(wc.ROW_CELL, 1, 0, (b[1][0] - 1) % P), (wc.ROW_CELL, 0, 0, 999), (wc.ROW_CELL, 0, 1, 999),
                       (wc.ROW_CELL, 0, 2, 0xDEADBEEF)],
             "amount_max2": [(wc.ROW_CELL, 0, 3, 10)],
             "padded": [(wc.ROW_CELL, 4, 4, 1 << 128), (wc.ROW_CELL, 1, 5, (1 << 128) + 7), (wc.ROW_CELL, 2, 4, P - 1)]}
    out = {"r": np.array(limbs(r.n), dtype=np.uint64), "scenarios": np.array([s[0] for s in scen])}
    tot = nfail = 0
    for name, w, MAX, n_mut in scen:
        muts = []
        exp = run(w, MAX)
        muts.append((-1, 0, 0, 0) + exp)
        cand = list(fixed.get(name, []))
        tries = 0
        while len(cand) < len(fixed.get(name, [])) + n_mut and tries < 10 * n_mut:
            tries += 1
            which = rng.choice([0, 0, 0, 0, 0, 1, 1, 2, 2, 2, 3, 4, 5, 6])
            if which == 0 and w["rows"].shape[1]:
                i, c = rng.randrange(w["rows"].shape[1]), rng.randrange(8)
                old = cells_of(w["rows"][:, i:i + 1])[0][c]
                v = (1 << 128) + rng.randrange(1 << 64) if (c in (4, 5) and rng.random() < 0.3) else corrupt_value(rng, old)
                cand.append((wc.ROW_CELL, i, c, v))
            elif which in (1, 2, 3):
                t = wc.TABLES[which - 1]
                n_cols = w[t].shape[0]
                i, c = rng.randrange(w[t].shape[1]), rng.randrange(n_cols)
                cand.append((which, i, c, corrupt_value(rng, cells_of(w[t][:, i:i + 1])[0][c])))
            elif which == 4:
                t = rng.randrange(1, 4)
                cand.append((wc.DROP_ROW, rng.randrange(w[wc.TABLES[t - 1]].shape[1]), t, 0))
            elif which == 5:
                cand.append((wc.DUP_BLOCK, 0, 0, rng.randrange(1, 1 << 32)))
            elif which == 6 and w["block"].shape[1]:  # a flipped tag: the block row's field tag / the MPT proof type
                if rng.random() < 0.5:
                    cand.append((wc.BLOCK_CELL, 0, 0, rng.choice([1, 2, 8, 10])))
                elif w["mpt"].shape[1]:
                    i = rng.randrange(w["mpt"].shape[1])
                    pt = cells_of(w["mpt"][:, i:i + 1])[0][1]
                    cand.append((wc.MPT_CELL, i, 1, 4 if pt == 8 else 8))
        for kind, i, c, v in cand:
            fr_, ex_ = run(wc.apply_mutation(w, kind, i, c, v), MAX)
            muts.append((kind, i, c, v, fr_, ex_))
        for k in ("rows",) + wc.TABLES:
            out[f"{name}/{k}"] = w[k]
        out[f"{name}/max"] = np.array(MAX, dtype=np.int64)
        out[f"{name}/mut_kind"] = np.array([m[0] for m in muts], dtype=np.int64)
        out[f"{name}/mut_row"] = np.array([m[1] for m in muts], dtype=np.int64)
        out[f"{name}/mut_col"] = np.array([m[2] for m in muts], dtype=np.int64)
        out[f"{name}/mut_val"] = np.array([limbs(m[3]) for m in muts], dtype=np.uint64)
        out[f"{name}/exp_row"] = np.array([m[4] for m in muts], dtype=np.int64)
        out[f"{name}/exp_exc"] = np.array([m[5] for m in muts])
        tot += len(muts)
        nfail += sum(m[4] >= 0 for m in muts)
        print(name, MAX, len(muts), "vectors", sorted(set(m[5] for m in muts)))
    np.savez_compressed(os.path.join(HERE, "withdrawal.npz"), **out)
    print(f"withdrawal: {tot} vectors, {nfail} failing")


if __name__ == "__main__":
    withdrawal_cases()
