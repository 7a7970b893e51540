"""Withdrawal-circuit test helpers: the golden file's layout (tests/golden/withdrawal.npz), the mutations its vectors
apply to a scenario's matrices, and the ctypes binding of the CPU oracle's withdrawal restatement (oracle/withdrawal.c)."""
import ctypes
import os

import numpy as np

import oracle_lib

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "withdrawal.npz")
TABLES = ("keccak", "mpt", "block")

# mutation kinds: 0 = row cell, 1/2/3 = keccak / MPT / block cell, 4 = drop a row of table `col` (1, 2, 3 as above),
# 5 = duplicate block row `row` with block_number `val`
ROW_CELL, KECCAK_CELL, MPT_CELL, BLOCK_CELL, DROP_ROW, DUP_BLOCK = range(6)


def _cell(v: int) -> np.ndarray:
    return np.array([(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(4)], dtype=np.uint64)


def apply_mutation(w: dict, kind: int, row: int, col: int, val: int) -> dict:
    """w: {"rows", "keccak", "mpt", "block"} uint64[n_cols][n][4] -> mutated copies"""
    out = {k: np.array(w[k]) for k in ("rows",) + TABLES}
    if kind < 0:
        return out
    if kind in (ROW_CELL, KECCAK_CELL, MPT_CELL, BLOCK_CELL):
        key = ("rows",) + TABLES
        out[key[kind]][col, row] = _cell(val)
    elif kind == DROP_ROW:
        t = TABLES[col - 1]
        out[t] = np.ascontiguousarray(np.delete(out[t], row, axis=1))
    elif kind == DUP_BLOCK:
        extra = out["block"][:, row:row + 1].copy()
        extra[1, 0] = _cell(val)
        out["block"] = np.ascontiguousarray(np.concatenate([out["block"], extra], axis=1))
    return out


def scenarios():
    """[(name, base matrices, max, r limbs, [(kind, row, col, val, exp_row, exp_exc)])] from the golden file"""
    z = np.load(GOLDEN)
    names = [str(s) for s in z["scenarios"]]
    r = z["r"]
    out = []
    for s in names:
        base = {k: z[f"{s}/{k}"] for k in ("rows",) + TABLES}
        muts = list(zip(z[f"{s}/mut_kind"].tolist(), z[f"{s}/mut_row"].tolist(), z[f"{s}/mut_col"].tolist(),
                        [oracle_lib.from_limbs(v) for v in z[f"{s}/mut_val"]], z[f"{s}/exp_row"].tolist(),
                        [str(e) for e in z[f"{s}/exp_exc"]]))
        out.append((s, base, int(z[f"{s}/max"]), r, muts))
    return out


def vectors():
    """every golden vector: (name, k, mutated matrices, max, r, exp_row, exp_exc)"""
    for name, base, mx, r, muts in scenarios():
        for k, (kind, row, col, val, exp_row, exp_exc) in enumerate(muts):
            yield name, k, apply_mutation(base, kind, row, col, val), mx, r, exp_row, exp_exc


def plan(n_rows: int, max_withdrawals: int):
    """what verify_circuit checks of n_rows rows: (rows used, row_end, index_error_row or None) —
    withdrawal_circuit.verify_circuit's split between the device check and Python's list indexing"""
    if n_rows == 0:
        return 0, 0, 0
    if max_withdrawals == 0:
        return 1, 1, None  # rows[-1], placed at global row 0
    if n_rows < max_withdrawals:
        return n_rows, n_rows - 1, n_rows - 1
    return max_withdrawals, max_withdrawals, None


def used_rows(rows: np.ndarray, max_withdrawals: int) -> np.ndarray:
    n = rows.shape[1]
    used, _, _ = plan(n, max_withdrawals)
    return np.ascontiguousarray(rows[:, n - 1:] if (max_withdrawals == 0 and n) else rows[:, :used])


# ---- the CPU oracle (oracle/withdrawal.c) ----------------------------------------------------------------------
def n_constraints() -> int:
    return oracle_lib.lib().orc_wd_n_constraints()


def classes():
    L = oracle_lib.lib()
    return [L.orc_wd_constraint_class(i) for i in range(L.orc_wd_n_constraints())]


def oracle_check(rows, keccak, mpt, block, r, max_withdrawals, row_begin=0, row_end=None, row_base=0):
    rows, keccak, mpt, block = [np.ascontiguousarray(a, dtype=np.uint64) for a in (rows, keccak, mpt, block)]
    n = n_constraints()
    ff = np.zeros(n, dtype=np.uint32)
    fc = np.zeros(n, dtype=np.uint64)
    c = ctypes.c_uint64
    if row_end is None:
        row_end = rows.shape[1]
    rr = np.ascontiguousarray(r, dtype=np.uint64)
    p = oracle_lib.p64
    rc = oracle_lib.lib().orc_check_withdrawal(
        p(rows), c(rows.shape[1]), p(keccak), c(keccak.shape[1]), p(mpt), c(mpt.shape[1]), p(block), c(block.shape[1]),
        p(rr), c(max_withdrawals), c(row_begin), c(row_end), c(row_base), ff.ctypes.data_as(oracle_lib.U32P), p(fc))
    assert rc == 0
    return ff, fc


def oracle_keccak_rows(rows, r) -> np.ndarray:
    """the keccak table withdrawals2witness builds for `rows` (hash cells as given): [5][n + 1][4]"""
    rows = np.ascontiguousarray(rows, dtype=np.uint64)
    out = np.zeros((5, rows.shape[1] + 1, 4), dtype=np.uint64)
    rr = np.ascontiguousarray(r, dtype=np.uint64)
    oracle_lib.lib().orc_wd_keccak_rows(oracle_lib.p64(rows), ctypes.c_uint64(rows.shape[1]), oracle_lib.p64(rr),
                                        oracle_lib.p64(out))
    return out


def verdict(ff, max_withdrawals, n_rows, cls=None):
    """(row, exception name) of a check of the rows `plan` selects, IndexError included"""
    row, exc = oracle_lib.first_failure(ff, cls or classes())
    if row >= 0:
        return row, exc
    _, _, ie = plan(n_rows, max_withdrawals)
    return (ie, "IndexError") if ie is not None else (-1, "")


def oracle_verdict(w, max_withdrawals, r):
    n = w["rows"].shape[1]
    _, end, _ = plan(n, max_withdrawals)
    if end == 0:
        return verdict(np.full(n_constraints(), 0xFFFFFFFF, dtype=np.uint32), max_withdrawals, n)
    ff, _ = oracle_check(used_rows(w["rows"], max_withdrawals), w["keccak"], w["mpt"], w["block"], r, max_withdrawals, 0, end)
    return verdict(ff, max_withdrawals, n)
