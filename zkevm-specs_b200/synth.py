"""Seeded synthetic witnesses as cell matrices (numpy), for parity tests at scale and bench.py.

They follow the witness rules of the reference's own builders (the small cases are checked
against the reference / oracle in tests) but skip the Python row objects: 2^20 steps would
need tens of millions of FQ objects.

evm_trace: BASELINE cfg2 — straight-line groups `PUSH32 b, PUSH32 a, OP, POP` with OP cycling
ADD, SUB, MUL, DIV, MOD and a final STOP step (recipe validated on the reference at 20 groups,
SURVEY.md §8d).  One contract holds the whole trace; its code_hash is a seeded 256-bit tag,
not a real keccak (the EVM circuit never recomputes the hash, it only matches it against the
bytecode table)."""
from __future__ import annotations

from typing import Dict

import numpy as np

from .evm_circuit.spec import ExecutionState, Target

M256 = (1 << 256) - 1
M64 = (1 << 64) - 1
P = 21888242871839275222246405745257275088548364400416034343698204186575808495617  # BN254 Fr
NASTY_AB_VALUES = (
    (0, 0), (1, 0), (0, 1), (1, 1), (255, 0), (0, 255), (255, 255), (256, 0), (0, 256), (256, 256),
    (260, 513), (65535, 0), (0, 65535), (65535, 65535), (65536, 0), (0, 65536), (65536, 65536),
    (M256, M256 - 1), (M256 - 1, M256), (M256, 0), (0, M256),
)  # the reference's edge operands, tests/common.py:23-45
OPS = ("ADD", "SUB", "MUL", "DIV", "MOD")
OPCODE = {"ADD": 0x01, "SUB": 0x03, "MUL": 0x02, "DIV": 0x04, "MOD": 0x06}
GAS = {"ADD": 3, "SUB": 3, "MUL": 5, "DIV": 5, "MOD": 5}


def ints_to_cells(vals) -> np.ndarray:
    """list of python ints (< 2^256) -> uint64[n][4]"""
    buf = b"".join(int(v).to_bytes(32, "little") for v in vals)
    return np.frombuffer(buf, dtype="<u8").reshape(-1, 4).copy()


def _operands(n: int, rng: np.random.Generator):
    kind = rng.integers(0, 4, n)
    raw = rng.integers(0, 1 << 63, (n, 2, 5), dtype=np.int64).astype(object)
    a, b = [], []
    nasty = rng.integers(0, len(NASTY_AB_VALUES), n)
    for i in range(n):
        k = kind[i]
        if k < 2:  # uniform 256-bit
            x = (raw[i, 0, 0] | raw[i, 0, 1] << 63 | raw[i, 0, 2] << 126 | raw[i, 0, 3] << 189 | raw[i, 0, 4] << 252) & M256
            y = (raw[i, 1, 0] | raw[i, 1, 1] << 63 | raw[i, 1, 2] << 126 | raw[i, 1, 3] << 189 | raw[i, 1, 4] << 252) & M256
        elif k == 2:  # 64-bit
            x, y = int(raw[i, 0, 0]) | (int(raw[i, 0, 1]) & 1) << 63, int(raw[i, 1, 0]) | (int(raw[i, 1, 1]) & 1) << 63
        else:
            x, y = NASTY_AB_VALUES[nasty[i]]
        a.append(int(x))
        b.append(int(y))
    return a, b


def evm_trace(n_groups: int, seed: int = 2, call_id: int = 1) -> Dict[str, np.ndarray]:
    """returns matrices: steps [13][4g+1][4], bytecode [6][68g+2][4], rw [14][6g][4]"""
    rng = np.random.default_rng(seed)
    g = n_groups
    a, b = _operands(g, rng)
    ops = [OPS[i % 5] for i in range(g)]
    c = []
    for op, x, y in zip(ops, a, b):
        if op == "ADD":
            c.append((x + y) & M256)
        elif op == "SUB":
            c.append((x - y) & M256)
        elif op == "MUL":
            c.append((x * y) & M256)
        elif op == "DIV":
            c.append(0 if y == 0 else x // y)
        else:
            c.append(0 if y == 0 else x % y)
    A, B, C = ints_to_cells(a), ints_to_cells(b), ints_to_cells(c)  # [g][4] limbs of the 256-bit values
    code_hash = int.from_bytes(rng.bytes(32), "little")
    h_lo, h_hi = code_hash & ((1 << 128) - 1), code_hash >> 128

    # ---- bytecode table: header + 68 bytes per group + STOP ---------------------------------
    code = np.zeros((g, 68), dtype=np.uint8)
    code[:, 0] = 0x7F
    code[:, 1:33] = np.ascontiguousarray(B).view(np.uint8).reshape(g, 32)[:, ::-1]  # big-endian push data
    code[:, 33] = 0x7F
    code[:, 34:66] = np.ascontiguousarray(A).view(np.uint8).reshape(g, 32)[:, ::-1]
    code[:, 66] = np.array([OPCODE[o] for o in ops], dtype=np.uint8)
    code[:, 67] = 0x50
    is_code = np.zeros((g, 68), dtype=np.uint8)
    is_code[:, [0, 33, 66, 67]] = 1
    code_len = 68 * g + 1
    nb = code_len + 1
    bytecode = np.zeros((6, nb, 4), dtype=np.uint64)
    bytecode[0, :, 0] = h_lo & 0xFFFFFFFFFFFFFFFF
    bytecode[0, :, 1] = h_lo >> 64
    bytecode[1, :, 0] = h_hi & 0xFFFFFFFFFFFFFFFF
    bytecode[1, :, 1] = h_hi >> 64
    bytecode[2, 0, 0] = 1  # Header: index 0, is_code 0, value = length
    bytecode[5, 0, 0] = code_len
    bytecode[2, 1:, 0] = 2
    bytecode[3, 1:, 0] = np.arange(code_len, dtype=np.uint64)
    bytecode[4, 1:-1, 0] = is_code.reshape(-1)
    bytecode[5, 1:-1, 0] = code.reshape(-1)
    bytecode[4, -1, 0] = 1  # STOP
    bytecode[5, -1, 0] = 0x00

    # ---- rw table: 6 stack rows per group ------------------------------------------------
    nr = 6 * g
    rw = np.zeros((14, nr, 4), dtype=np.uint64)
    rw[0, :, 0] = np.arange(1, nr + 1, dtype=np.uint64)
    rw[1, :, 0] = np.tile(np.array([1, 1, 0, 0, 1, 0], dtype=np.uint64), g)
    rw[2, :, 0] = int(Target.Stack)
    rw[3, :, 0] = call_id
    rw[4, :, 0] = np.tile(np.array([1023, 1022, 1022, 1023, 1023, 1023], dtype=np.uint64), g)
    vals = np.stack([B, A, A, B, C, C], axis=1).reshape(nr, 4)  # [nr][4] limbs of each 256-bit value
    rw[8, :, 0], rw[8, :, 1] = vals[:, 0], vals[:, 1]  # value.lo
    rw[9, :, 0], rw[9, :, 1] = vals[:, 2], vals[:, 3]  # value.hi

    # ---- steps: PUSH, PUSH, OP, POP per group + STOP --------------------------------------
    ns = 4 * g + 1
    steps = np.zeros((13, ns, 4), dtype=np.uint64)
    op_state = np.array([int(ExecutionState.ADD) if o in ("ADD", "SUB") else int(ExecutionState.MUL) for o in ops],
                        dtype=np.uint64)
    st = np.empty((g, 4), dtype=np.uint64)
    st[:, 0] = st[:, 1] = int(ExecutionState.PUSH)
    st[:, 2] = op_state
    st[:, 3] = int(ExecutionState.POP)
    steps[0, :-1, 0] = st.reshape(-1)
    steps[0, -1, 0] = int(ExecutionState.STOP)
    grp = np.arange(g, dtype=np.uint64)
    rwc = np.stack([6 * grp + 1, 6 * grp + 2, 6 * grp + 3, 6 * grp + 6], axis=1)
    steps[1, :-1, 0] = rwc.reshape(-1)
    steps[1, -1, 0] = 6 * g + 1
    steps[2, :, 0] = call_id
    steps[3, :, 0] = 1  # is_root
    steps[5, :, 0], steps[5, :, 1] = h_lo & 0xFFFFFFFFFFFFFFFF, h_lo >> 64
    steps[6, :, 0], steps[6, :, 1] = h_hi & 0xFFFFFFFFFFFFFFFF, h_hi >> 64
    pc = np.stack([68 * grp, 68 * grp + 33, 68 * grp + 66, 68 * grp + 67], axis=1)
    steps[7, :-1, 0] = pc.reshape(-1)
    steps[7, -1, 0] = 68 * g
    steps[8, :-1, 0] = np.tile(np.array([1024, 1023, 1022, 1023], dtype=np.uint64), g)
    steps[8, -1, 0] = 1024
    gas_op = np.array([GAS[o] for o in ops], dtype=np.uint64)
    cost = np.stack([np.full(g, 3, np.uint64), np.full(g, 3, np.uint64), gas_op, np.full(g, 2, np.uint64)], axis=1).reshape(-1)
    total = int(cost.sum())
    spent_before = np.concatenate([[0], np.cumsum(cost)]).astype(np.uint64)
    steps[9, :, 0] = np.uint64(total + 7) - spent_before
    # the same bytecode as raw bytes, for zk_upload_bytecode_table_from_code (one contract)
    code_bytes = np.concatenate([code.reshape(-1), np.zeros(1, dtype=np.uint8)])  # ... + STOP
    is_code_all = np.concatenate([is_code.reshape(-1), np.ones(1, dtype=np.uint8)])
    src = {"code": code_bytes, "is_code_bits": np.packbits(is_code_all, bitorder="little"),
           "code_offsets": np.array([0, code_len], dtype=np.uint64),
           "hashes": np.array([[h_lo & 0xFFFFFFFFFFFFFFFF, h_lo >> 64, h_hi & 0xFFFFFFFFFFFFFFFF, h_hi >> 64]],
                              dtype=np.uint64)}
    return {"steps": steps, "bytecode": bytecode, "rw": rw, "n_steps": ns - 1, "bytecode_src": src}


def state_rows(n_rows: int, seed: int = 3, n_start: int = 1024) -> Dict[str, np.ndarray]:
    """BASELINE cfg3 — a sorted RW-table witness for the state circuit as cell matrices:
    `n_start` Start padding rows, then Memory ~40 %, Stack ~40 %, Storage ~5 %, CallContext ~10 %,
    Account ~5 % (tag order of state_circuit.Tag), each key written once then read, with the
    mock MPT table of the reference (`_mock_mpt_updates`, state_circuit.py:903-933: root starts
    at 3, +5 per first touch of a Storage/Account key).  Returns rows [57][n][4], flags [n],
    mpt [12][m][4]."""
    rng = np.random.default_rng(seed)
    n_start = min(n_start, n_rows // 2)
    body = n_rows - n_start
    per = 4  # accesses per key: 1 write + 3 reads
    n_keys = body // per
    counts = {"mem": int(n_keys * 0.40), "stack": int(n_keys * 0.40), "sto": int(n_keys * 0.05),
              "cc": int(n_keys * 0.10)}
    counts["acc"] = n_keys - sum(counts.values())
    extra = body - n_keys * per  # leftover rows become extra Start rows
    n_start += extra
    n = n_rows

    tag = np.zeros(n, np.uint64); idc = np.zeros(n, np.uint64); addr = np.zeros(n, np.uint64)
    ft = np.zeros(n, np.uint64); key = np.zeros((n, 4), np.uint64)
    is_write = np.zeros(n, np.uint64); val = np.zeros((n, 4), np.uint64); init = np.zeros((n, 4), np.uint64)
    flags = np.zeros(n, np.uint8); selector = np.ones(n, np.uint64)
    tag[:n_start] = 1
    selector[0] = 0
    pos = n_start

    def fill(kind, nk):
        nonlocal pos
        if nk == 0:
            return None
        sl = slice(pos, pos + nk * per)
        w = np.tile(np.array([1] + [0] * (per - 1), np.uint64), nk)
        is_write[sl] = w
        pos += nk * per
        return sl

    # Memory (tag 2): call_id 1.., consecutive addresses; value a byte
    nk = counts["mem"]; sl = fill("mem", nk)
    if sl:
        k = np.repeat(np.arange(nk, dtype=np.uint64), per)
        tag[sl] = 2; idc[sl] = 1 + k // np.uint64(1 << 16); addr[sl] = k % np.uint64(1 << 16)
        val[sl, 0] = np.repeat(rng.integers(0, 256, nk, dtype=np.uint64), per)
    # Stack (tag 3): per call 1024 slots, pointer ascending; value a 256-bit word
    nk = counts["stack"]; sl = fill("stack", nk)
    if sl:
        k = np.repeat(np.arange(nk, dtype=np.uint64), per)
        tag[sl] = 3; idc[sl] = 1 + k // np.uint64(1024); addr[sl] = k % np.uint64(1024)
        val[sl] = np.repeat(rng.integers(0, 1 << 63, (nk, 4), dtype=np.uint64) * np.uint64(2) + np.uint64(1), per, axis=0)
        flags[sl] |= 1
    # Storage (tag 4): tx 1, one address, increasing keys; committed value = value
    nk_sto = counts["sto"]; sl_sto = fill("sto", nk_sto)
    if sl_sto:
        k = np.repeat(np.arange(nk_sto, dtype=np.uint64), per)
        tag[sl_sto] = 4; idc[sl_sto] = 1; addr[sl_sto] = 0x12345678
        key[sl_sto, 0] = k + np.uint64(1); key[sl_sto, 2] = k * np.uint64(7)
        v = np.repeat(rng.integers(1, 1 << 62, (nk_sto, 4), dtype=np.uint64), per, axis=0)
        val[sl_sto] = v; init[sl_sto] = v
        is_write[sl_sto] = 0  # reads of the committed value (a write would change value within the group)
        flags[sl_sto] |= 3
    # CallContext (tag 5): field tag 14 (IsStatic)
    nk = counts["cc"]; sl = fill("cc", nk)
    if sl:
        k = np.repeat(np.arange(nk, dtype=np.uint64), per)
        tag[sl] = 5; idc[sl] = 1 + k; ft[sl] = 14
        val[sl, 0] = np.repeat(rng.integers(0, 2, nk, dtype=np.uint64), per)
    # Account (tag 6): increasing addresses, field tag Balance (2); committed value = value
    nk_acc = counts["acc"]; sl_acc = fill("acc", nk_acc)
    if sl_acc:
        k = np.repeat(np.arange(nk_acc, dtype=np.uint64), per)
        tag[sl_acc] = 6; addr[sl_acc] = np.uint64(0x1000) + k; ft[sl_acc] = 2
        v = np.repeat(rng.integers(1, 1 << 62, (nk_acc, 4), dtype=np.uint64), per, axis=0)
        val[sl_acc] = v; init[sl_acc] = v
        is_write[sl_acc] = 0
        flags[sl_acc] |= 3
    assert pos == n

    # rw_counter: Start rows 1..n_start; the others any increasing counter (unique per row)
    rwc = np.arange(1, n + 1, dtype=np.uint64)
    # roots: MPT rows carry the root before their key's update; everything else the next one's
    rp = np.full(n + 1, -1, np.int64)
    groups = []
    if sl_sto:
        g = np.arange(nk_sto, dtype=np.int64)
        rp[sl_sto] = np.repeat(3 + 5 * g, per)
        groups.append((sl_sto, nk_sto, 0, 6))
    if sl_acc:
        g = np.arange(nk_acc, dtype=np.int64) + nk_sto
        rp[sl_acc] = np.repeat(3 + 5 * g, per)
        groups.append((sl_acc, nk_acc, nk_sto, 2))
    n_upd = nk_sto + nk_acc
    rp[n] = 3 + 5 * n_upd
    big = np.where(rp >= 0, rp, np.int64(1) << 62)
    nxt = np.minimum.accumulate(big[::-1])[::-1]  # next non-None root at or after k
    root = nxt[1:].astype(np.uint64)  # row k carries roots[k + 1]

    rows = np.zeros((57, n, 4), dtype=np.uint64)
    rows[0, :, 0] = rwc; rows[1, :, 0] = is_write; rows[2, :, 0] = tag; rows[3, :, 0] = idc
    rows[4, :, 0] = addr; rows[5, :, 0] = ft
    rows[6, :, 0], rows[6, :, 1] = key[:, 0], key[:, 1]
    rows[7, :, 0], rows[7, :, 1] = key[:, 2], key[:, 3]
    for k in range(10):  # 16-bit address limbs (addresses here fit 64 bits)
        rows[8 + k, :, 0] = (addr >> np.uint64(16 * k)) & np.uint64(0xFFFF) if k < 4 else 0
    kb = np.ascontiguousarray(key).view(np.uint8).reshape(n, 32)
    for b in range(32):
        rows[18 + b, :, 0] = kb[:, b]
    rows[50, :, 0], rows[50, :, 1] = val[:, 0], val[:, 1]
    rows[51, :, 0], rows[51, :, 1] = val[:, 2], val[:, 3]
    rows[52, :, 0], rows[52, :, 1] = init[:, 0], init[:, 1]
    rows[53, :, 0], rows[53, :, 1] = init[:, 2], init[:, 3]
    rows[54, :, 0] = root
    rows[56, :, 0] = selector

    mpt = np.zeros((12, n_upd, 4), dtype=np.uint64)
    for sl, nk, g0, proof in groups:
        first = np.arange(sl.start, sl.stop, per)
        d = slice(g0, g0 + nk)
        mpt[0, d, 0] = addr[first]; mpt[1, d, 0] = proof
        mpt[2, d, 0], mpt[2, d, 1] = key[first, 0], key[first, 1]
        mpt[3, d, 0], mpt[3, d, 1] = key[first, 2], key[first, 3]
        mpt[4, d, 0] = 3 + 5 * (np.arange(nk, dtype=np.uint64) + np.uint64(g0)) + np.uint64(5)  # root
        mpt[6, d, 0] = 3 + 5 * (np.arange(nk, dtype=np.uint64) + np.uint64(g0))  # root_prev
        mpt[8, d, 0], mpt[8, d, 1] = val[first, 0], val[first, 1]
        mpt[9, d, 0], mpt[9, d, 1] = val[first, 2], val[first, 3]
        mpt[10, d, 0], mpt[10, d, 1] = init[first, 0], init[first, 1]
        mpt[11, d, 0], mpt[11, d, 1] = init[first, 2], init[first, 3]
    return {"rows": rows, "flags": flags, "mpt": mpt}


FR_P = 21888242871839275222246405745257275088548364400416034343698204186575808495617


def copy_events(n_events: int, length: int, seed: int = 4, r: int = 0x2545F4914F6CDD1D5851F42D4C957F2D14057B7EF767814F) -> Dict[str, np.ndarray]:
    """BASELINE cfg4 — copy-circuit witness as cell matrices: n_events/2 SHA3-style events
    (Memory -> RlcAcc) and n_events/2 root CALLDATACOPY events (TxCalldata -> Memory whose last
    10 % of bytes are out of bounds => padding), `length` bytes each, two rows per byte
    (CopyCircuit.copy, evm_circuit/typing.py:1010-1091), with the rw-table memory rows and tx-table
    calldata rows they look up.  Returns copy [20][2*n_events*length][4] (+copy_flags), rw [14][..]
    (+rw_flags), tx [5][..] (+tx_flags), bytecode [6][0], r."""
    rng = np.random.default_rng(seed)
    L = length
    n_sha = n_events // 2
    n_cdc = n_events - n_sha
    n_rows = 2 * n_events * L
    C = np.zeros((20, n_rows, 4), dtype=np.uint64)
    data = rng.integers(0, 256, (n_events, L), dtype=np.uint64)
    i_idx = np.arange(L, dtype=np.uint64)
    rw_rows = []
    tx_rows = []
    events = []  # rows of zk_assign_copy_circuit's events array (assign.copy_event)
    rwc = 1
    pos = 0

    def put(col, sl, vals):
        C[col, sl, 0] = vals

    for e in range(n_events):
        is_sha = e < n_sha
        rd = slice(pos, pos + 2 * L, 2)
        wr = slice(pos + 1, pos + 2 * L, 2)
        ev = slice(pos, pos + 2 * L)
        b = data[e].copy()
        put(0, rd, 1)  # q_step
        C[1, pos, 0] = 1  # is_first
        C[2, pos + 2 * L - 1, 0] = 1  # is_last
        put(8, rd, np.uint64(L) - i_idx)  # bytes_left
        if is_sha:
            call_id, src = 1 + e, 64 * e
            put(3, ev, call_id)
            put(5, rd, 2); put(5, wr, 5)  # Memory -> RlcAcc
            put(6, rd, np.uint64(src) + i_idx); put(6, wr, i_idx)
            put(7, rd, src + L)
            put(9, rd, b)
            acc, accs = 0, []
            for v in b.tolist():
                acc = (acc * r + int(v)) % FR_P
                accs.append(acc)
            cells = ints_to_cells(accs)
            C[9, wr, :] = cells
            C[10, ev, :] = cells[-1]
            put(13, rd, np.uint64(rwc) + i_idx); put(13, wr, np.uint64(rwc) + i_idx + np.uint64(1))
            put(14, rd, np.uint64(L) - i_idx); put(14, wr, np.uint64(L) - i_idx - np.uint64(1))
            put(15, rd, 1); put(19, wr, 1)
            events.append([2, 5, src, src + L, 0, L, 0, rwc, call_id, 0, 0, 0, call_id, 0, 0, 0])
            rw_rows.append(np.stack([np.uint64(rwc) + i_idx, np.zeros(L, np.uint64), np.full(L, 9, np.uint64),
                                     np.full(L, call_id, np.uint64), np.uint64(src) + i_idx, b]))
            rwc += L
        else:
            tx_id, call_id, dst = 1 + (e - n_sha), 1 + e, 32 * e
            n_real = L - L // 10  # the last 10 % read past the end of calldata
            b[n_real:] = 0
            put(3, rd, tx_id); put(3, wr, call_id)
            put(5, rd, 3); put(5, wr, 2)  # TxCalldata -> Memory
            put(6, rd, i_idx); put(6, wr, np.uint64(dst) + i_idx)
            put(7, rd, n_real)
            put(9, ev, np.repeat(b, 2))
            put(12, rd, (i_idx >= np.uint64(n_real)).astype(np.uint64))  # is_pad
            put(13, ev, np.repeat(np.uint64(rwc) + i_idx, 2))
            put(14, ev, np.repeat(np.uint64(L) - i_idx, 2))
            put(17, rd, 1); put(15, wr, 1)
            events.append([3, 2, 0, n_real, dst, L, 0, rwc, tx_id, 0, 0, 0, call_id, 0, 0, 0])
            data[e] = b
            rw_rows.append(np.stack([np.uint64(rwc) + i_idx, np.ones(L, np.uint64), np.full(L, 9, np.uint64),
                                     np.full(L, call_id, np.uint64), np.uint64(dst) + i_idx, b]))
            tx_rows.append(np.stack([np.full(n_real, tx_id, np.uint64), np.full(n_real, 13, np.uint64),
                                     i_idx[:n_real], b[:n_real]]))
            rwc += L
        pos += 2 * L
    RWs = np.concatenate(rw_rows, axis=1) if rw_rows else np.zeros((6, 0), np.uint64)
    rw = np.zeros((14, RWs.shape[1], 4), dtype=np.uint64)
    rw[0, :, 0], rw[1, :, 0], rw[2, :, 0], rw[3, :, 0], rw[4, :, 0], rw[8, :, 0] = RWs
    TXs = np.concatenate(tx_rows, axis=1) if tx_rows else np.zeros((4, 0), np.uint64)
    tx = np.zeros((5, TXs.shape[1], 4), dtype=np.uint64)
    tx[0, :, 0], tx[1, :, 0], tx[2, :, 0], tx[3, :, 0] = TXs
    return {"copy": C, "copy_flags": np.zeros(n_rows, np.uint8), "rw": rw, "rw_flags": np.zeros(rw.shape[1], np.uint8),
            "tx": tx, "tx_flags": np.zeros(tx.shape[1], np.uint8), "bytecode": np.zeros((6, 0, 4), np.uint64),
            "events": np.array(events, dtype=np.uint64).reshape(-1, 16), "data": data.astype(np.uint8).reshape(-1), "r_int": r,
            "r": np.array([(r >> (64 * k)) & 0xFFFFFFFFFFFFFFFF for k in range(4)], dtype=np.uint64)}


def bytecode_circuit_rows(k: int, n_contracts: int = 4, seed: int = 5,
                          r: int = 0x1D5851F42D4C957F2D14057B7EF767814F2545F4914F6CDD) -> Dict[str, np.ndarray]:
    """BASELINE cfg5's bytecode-circuit share — 2^k rows of assign_bytecode_circuit
    (src/zkevm_specs/bytecode_circuit.py:104-167) for `n_contracts` random contracts that fill the
    circuit, as cell matrices: rows [12][2^k][4], push table [2][256][4], keccak table [5][n][4].
    The value_rlc prefix (one Fr product per byte) is computed with Python ints."""
    from .util.hash import keccak256

    rng = np.random.default_rng(seed)
    size = 1 << k
    per = (size - 1) // n_contracts - 1  # bytes per contract; the rest is Header padding
    rows = np.zeros((12, size, 4), dtype=np.uint64)
    keccak_rows, at, codes = [], 0, []
    push_size = np.zeros(256, dtype=np.int64)
    push_size[0x60:0x80] = np.arange(1, 33)

    def put(col, lo, hi, vals):  # python ints / arrays of small ints
        rows[col, lo:hi, 0] = vals

    for _ in range(n_contracts):
        code = rng.integers(0, 256, per, dtype=np.uint8)
        codes.append(bytes(code))
        h = int.from_bytes(keccak256(bytes(code)), "big")
        # push_data_left / is_code: sequential scan over the code (get_push_size, opcode.py:427-433)
        left = np.zeros(per, dtype=np.int64)
        pending = 0
        sizes = push_size[code]
        for i in range(per):
            left[i] = pending
            pending = int(sizes[i]) if pending == 0 else pending - 1
        is_code = (left == 0).astype(np.uint64)
        acc, rlc = 0, []
        for b in code:
            acc = (acc * r + int(b)) % P
            rlc.append(acc)
        lo, hi = at, at + per + 1
        h_lo, h_hi = h & ((1 << 128) - 1), h >> 128
        rows[2, lo:hi, 0], rows[2, lo:hi, 1] = h_lo & M64, h_lo >> 64
        rows[3, lo:hi, 0], rows[3, lo:hi, 1] = h_hi & M64, h_hi >> 64
        put(4, lo, lo + 1, 1)                      # Header: value = length
        put(6, lo, lo + 1, per)
        put(10, lo, hi, per)
        put(4, lo + 1, hi, 2)                      # Byte rows
        put(5, lo + 1, hi, np.arange(per, dtype=np.uint64))
        put(6, lo + 1, hi, code.astype(np.uint64))
        put(7, lo + 1, hi, is_code)
        put(8, lo + 1, hi, left.astype(np.uint64))
        rows[9, lo + 1:hi, :] = ints_to_cells(rlc)
        put(11, lo + 1, hi, sizes.astype(np.uint64))  # get_push_size(value) on every Byte row (:122)
        keccak_rows.append([2, rlc[-1], per, h & ((1 << 128) - 1), h >> 128])
        at = hi
    # Header padding with the empty hash (bytecode_circuit.py:150-165)
    e = int.from_bytes(keccak256(b""), "big")
    e_lo, e_hi = e & ((1 << 128) - 1), e >> 128
    rows[2, at:, 0], rows[2, at:, 1] = e_lo & M64, e_lo >> 64
    rows[3, at:, 0], rows[3, at:, 1] = e_hi & M64, e_hi >> 64
    rows[4, at:, 0] = 1
    rows[0, 0, 0] = 1
    rows[1, size - 1, 0] = 1
    push = np.zeros((2, 256, 4), dtype=np.uint64)
    push[0, :, 0] = np.arange(256)
    push[1, :, 0] = push_size
    kec = np.zeros((5, len(keccak_rows), 4), dtype=np.uint64)
    for i, row in enumerate(keccak_rows):
        for c, v in enumerate(row):
            kec[c, i, :] = [(v >> (64 * j)) & M64 for j in range(4)]
    return {"rows": rows, "push": push, "keccak": kec, "r": np.array([(r >> (64 * j)) & M64 for j in range(4)], dtype=np.uint64),
            "codes": codes, "r_int": r}


# ------------------------------------------------------------------------------------------------
def block_trace(n_txs: int, groups_per_contract: int, n_contracts: int, seed: int = 6, n_padding: int = 8,
                real_hashes: bool = False) -> Dict[str, np.ndarray]:
    """A whole-block EVM trace, the shape `verify_steps(begin_with_first_step=True, end_with_last_step=True)` checks:

        BeginTx, [PUSH32 b, PUSH32 a, OP, POP] x groups, STOP, EndTx     ... once per transaction
        EndBlock                                                          (the last step; + the dummy step)

    `n_contracts` contracts of `groups_per_contract` groups each (68 bytes per group + STOP); transaction t (id t + 1,
    its own caller account) calls contract t % n_contracts with no value and no call data.  The rw table is laid out
    head + tail: every row of the trace by rw_counter (1 ..), then `n_padding` Start padding rows (rw_counter 1 ..), the
    layout EndBlock's two rw_table_start_lookups count (end_block.py:30-38, 168-171).  Code hashes are seeded tags
    unless `real_hashes` (the EVM circuit only matches them against the bytecode table).
    Returns steps [13][n+1][4] (dummy EndBlock step included), bytecode (table + source form), rw + rw_flags, tx +
    tx_flags, block + block_flags, wd (empty), n_steps, flags = FIRST | LAST.  Validated on the reference at small
    sizes by tests/golden/gen_golden.py synth."""
    from .evm_circuit.spec import AccountFieldTag as AF, CallContextFieldTag as CC, TxContextFieldTag as TXF, TxReceiptFieldTag as RF
    from .util.hash import keccak256

    rng = np.random.default_rng(seed)
    G, C, T = groups_per_contract, n_contracts, n_txs
    code_len = 68 * G + 1
    # ---- contracts: operands, code, hashes
    a, b = _operands(G * C, rng)
    ops_idx = np.arange(G * C) % 5
    ops = [OPS[i] for i in ops_idx]
    c_res = []
    for op, x, y in zip(ops, a, b):
        c_res.append((x + y) & M256 if op == "ADD" else (x - y) & M256 if op == "SUB" else (x * y) & M256 if op == "MUL"
                     else (0 if y == 0 else x // y) if op == "DIV" else (0 if y == 0 else x % y))
    A, B, Cv = ints_to_cells(a), ints_to_cells(b), ints_to_cells(c_res)
    code = np.zeros((C, code_len), dtype=np.uint8)
    grp = code[:, :-1].reshape(C, G, 68)
    grp[:, :, 0] = 0x7F
    grp[:, :, 1:33] = np.ascontiguousarray(B).view(np.uint8).reshape(C, G, 32)[:, :, ::-1]
    grp[:, :, 33] = 0x7F
    grp[:, :, 34:66] = np.ascontiguousarray(A).view(np.uint8).reshape(C, G, 32)[:, :, ::-1]
    grp[:, :, 66] = np.array([OPCODE[o] for o in ops], dtype=np.uint8).reshape(C, G)
    grp[:, :, 67] = 0x50
    is_code = np.zeros((C, code_len), dtype=np.uint8)
    ic = is_code[:, :-1].reshape(C, G, 68)
    ic[:, :, [0, 33, 66, 67]] = 1
    is_code[:, -1] = 1  # STOP
    if real_hashes:
        hashes_int = [int.from_bytes(keccak256(bytes(code[k])), "big") for k in range(C)]
    else:
        hashes_int = [int.from_bytes(rng.bytes(32), "little") | 1 for _ in range(C)]
    H = ints_to_cells(hashes_int)  # [C][4]: lo limbs 0,1; hi limbs 2,3
    # bytecode table (unrolled) and source form
    nb = C * (code_len + 1)
    bytecode = np.zeros((6, nb, 4), dtype=np.uint64)
    rows_per = code_len + 1
    hrep = np.repeat(H, rows_per, axis=0)
    bytecode[0, :, 0], bytecode[0, :, 1] = hrep[:, 0], hrep[:, 1]
    bytecode[1, :, 0], bytecode[1, :, 1] = hrep[:, 2], hrep[:, 3]
    tagcol = np.full((C, rows_per), 2, dtype=np.uint64); tagcol[:, 0] = 1
    idxcol = np.zeros((C, rows_per), dtype=np.uint64); idxcol[:, 1:] = np.arange(code_len, dtype=np.uint64)
    iscol = np.zeros((C, rows_per), dtype=np.uint64); iscol[:, 1:] = is_code
    valcol = np.zeros((C, rows_per), dtype=np.uint64); valcol[:, 0] = code_len; valcol[:, 1:] = code
    bytecode[2, :, 0], bytecode[3, :, 0] = tagcol.reshape(-1), idxcol.reshape(-1)
    bytecode[4, :, 0], bytecode[5, :, 0] = iscol.reshape(-1), valcol.reshape(-1)
    src = {"code": code.reshape(-1).copy(), "is_code_bits": np.packbits(is_code.reshape(-1), bitorder="little"),
           "code_offsets": (np.arange(C + 1, dtype=np.uint64) * np.uint64(code_len)),
           "hashes": H.copy()}

    # ---- per-transaction layout
    S_TX = 4 * G + 3                       # BeginTx + body + STOP + EndTx
    n_steps = T * S_TX + 1                  # + EndBlock
    steps = np.zeros((13, n_steps + 1, 4), dtype=np.uint64)   # + the dummy step of end_with_last_step
    GAS_PRICE, BASE_FEE, COINBASE, GAS_LIMIT = int(2e9), int(1e9), 0x10, 1 << 62
    body_gas = np.array([3 + 3 + GAS[o] + 2 for o in ops], dtype=np.int64).reshape(C, G).sum(axis=1)
    RW_TX_FIRST, RW_TX_REST = 24 + 6 * G + 1 + 9, 24 + 6 * G + 1 + 10   # rw rows of the first / another transaction
    n_real = RW_TX_FIRST + (T - 1) * RW_TX_REST + 2 - 1                  # last EndTx has no next-tx row; EndBlock adds 2
    nr = n_real + n_padding
    rw = np.zeros((14, nr, 4), dtype=np.uint64)
    rwf = np.zeros(nr, dtype=np.uint8)
    tx = np.zeros((5, 12 * T, 4), dtype=np.uint64)
    txf = np.zeros(12 * T, dtype=np.uint8)

    def put_rw(k, rw_, tag, id=0, addr=0, ft=0, val=0, prev=0, word=False, prev_word=False):
        rw[0, k, 0], rw[1, k, 0], rw[2, k, 0] = k + 1, rw_, tag
        rw[3, k, :], rw[4, k, :] = limbs4(id), limbs4(addr)
        rw[5, k, 0] = ft
        v, p = limbs4(val), limbs4(prev)
        rw[8, k, 0], rw[8, k, 1], rw[9, k, 0], rw[9, k, 1] = v[0], v[1], v[2], v[3]
        rw[10, k, 0], rw[10, k, 1], rw[11, k, 0], rw[11, k, 1] = p[0], p[1], p[2], p[3]
        rwf[k] = int(word) | (int(prev_word) << 1)

    def limbs4(v):
        return [(int(v) >> (64 * q)) & M64 for q in range(4)]

    TAG = {"acl": int(Target.TxAccessListAccount), "refund": int(Target.TxRefund), "acc": int(Target.Account),
           "cc": int(Target.CallContext), "stack": int(Target.Stack), "rcpt": int(Target.TxReceipt), "start": int(Target.Start)}
    k = 0          # next rw row (rw_counter = k + 1)
    cum_gas = 0
    coinbase_bal = 0
    grp_ar = np.arange(G, dtype=np.uint64)
    for t in range(T):
        tx_id, c, caller, callee = t + 1, t % C, 0xFE0000 + t, 0xC0DE0000 + (t % C)
        gas = 21000 + int(body_gas[c]) + 777
        h_lo = int(H[c, 0]) | (int(H[c, 1]) << 64)
        h_hi = int(H[c, 2]) | (int(H[c, 3]) << 64)
        code_hash = h_lo | (h_hi << 128)
        s0 = t * S_TX
        call_id = k + 1
        # tx table: twelve fixed rows
        fixed = [(TXF.Nonce, 0, 0), (TXF.Gas, gas, 0), (TXF.GasPrice, GAS_PRICE, 1), (TXF.CallerAddress, caller, 1),
                 (TXF.CalleeAddress, callee, 1), (TXF.IsCreate, 0, 0), (TXF.Value, 0, 1), (TXF.CallDataLength, 0, 0),
                 (TXF.CallDataGasCost, 0, 0), (TXF.TxInvalid, 0, 0), (TXF.AccessListGasCost, 0, 0), (TXF.TxSignHash, 1234, 0)]
        for q, (tg, v, w_) in enumerate(fixed):
            r_ = 12 * t + q
            tx[0, r_, 0], tx[1, r_, 0] = tx_id, int(tg)
            lv = limbs4(v)
            tx[3, r_, 0], tx[3, r_, 1], tx[4, r_, 0], tx[4, r_, 1] = lv[0], lv[1], lv[2], lv[3]
            txf[r_] = w_
        # ---- BeginTx
        steps[0, s0, 0], steps[1, s0, 0] = int(ExecutionState.BeginTx), k + 1
        if t:  # StepState of a BeginTx after an EndTx: call_id 0 .. (the reference's tests leave the defaults)
            pass
        steps[8, s0, 0] = 1024
        caller_bal = 10 ** 20
        put_rw(k, 0, TAG["cc"], call_id, int(CC.TxId), val=tx_id); k += 1
        put_rw(k, 0, TAG["cc"], call_id, int(CC.RwCounterEndOfReversion)); k += 1
        put_rw(k, 0, TAG["cc"], call_id, int(CC.IsPersistent), val=1); k += 1
        put_rw(k, 0, TAG["cc"], call_id, int(CC.IsSuccess), val=1); k += 1
        put_rw(k, 1, TAG["acc"], 0, caller, int(AF.Nonce), val=1, prev=0); k += 1
        for adr in (COINBASE, caller, callee):
            put_rw(k, 1, TAG["acl"], tx_id, adr, val=1, prev=0); k += 1
        put_rw(k, 1, TAG["acc"], 0, caller, int(AF.Balance), val=caller_bal - gas * GAS_PRICE, prev=caller_bal, word=True, prev_word=True); k += 1
        put_rw(k, 1, TAG["acc"], 0, callee, int(AF.Balance), val=0, prev=0, word=True, prev_word=True); k += 1
        put_rw(k, 0, TAG["acc"], 0, callee, int(AF.CodeHash), val=code_hash, prev=code_hash, word=True, prev_word=True); k += 1
        ctx_vals = [(CC.Depth, 1, 0), (CC.CallerAddress, caller, 1), (CC.CalleeAddress, callee, 1), (CC.CallDataOffset, 0, 0),
                    (CC.CallDataLength, 0, 0), (CC.Value, 0, 1), (CC.IsStatic, 0, 0), (CC.LastCalleeId, 0, 0),
                    (CC.LastCalleeReturnDataOffset, 0, 0), (CC.LastCalleeReturnDataLength, 0, 0), (CC.IsRoot, 1, 0),
                    (CC.IsCreate, 0, 0), (CC.CodeHash, code_hash, 1)]
        for tg, v, w_ in ctx_vals:
            put_rw(k, 0, TAG["cc"], call_id, int(tg), val=v, word=bool(w_)); k += 1
        # ---- body: 4 G steps, 6 G stack rows (vectorised)
        sb = s0 + 1
        st = np.empty((G, 4), dtype=np.uint64)
        st[:, 0] = st[:, 1] = int(ExecutionState.PUSH)
        opsl = ops[c * G:(c + 1) * G]
        st[:, 2] = np.array([int(ExecutionState.ADD) if o in ("ADD", "SUB") else int(ExecutionState.MUL) for o in opsl], dtype=np.uint64)
        st[:, 3] = int(ExecutionState.POP)
        body = slice(sb, sb + 4 * G)
        steps[0, body, 0] = st.reshape(-1)
        base_rwc = np.uint64(k + 1)
        steps[1, body, 0] = (np.stack([6 * grp_ar, 6 * grp_ar + 1, 6 * grp_ar + 2, 6 * grp_ar + 5], axis=1) + base_rwc).reshape(-1)
        steps[7, body, 0] = np.stack([68 * grp_ar, 68 * grp_ar + 33, 68 * grp_ar + 66, 68 * grp_ar + 67], axis=1).reshape(-1)
        steps[8, body, 0] = np.tile(np.array([1024, 1023, 1022, 1023], dtype=np.uint64), G)
        cost = np.stack([np.full(G, 3), np.full(G, 3), np.array([GAS[o] for o in opsl]), np.full(G, 2)], axis=1).reshape(-1)
        gas_after_begin = gas - 21000
        spent = np.concatenate([[0], np.cumsum(cost)])
        steps[9, sb:sb + 4 * G + 1, 0] = (gas_after_begin - spent).astype(np.uint64)   # body steps + STOP
        rs = slice(k, k + 6 * G)
        rw[0, rs, 0] = np.arange(k + 1, k + 6 * G + 1, dtype=np.uint64)
        rw[1, rs, 0] = np.tile(np.array([1, 1, 0, 0, 1, 0], dtype=np.uint64), G)
        rw[2, rs, 0] = TAG["stack"]
        rw[3, rs, 0] = call_id
        rw[4, rs, 0] = np.tile(np.array([1023, 1022, 1022, 1023, 1023, 1023], dtype=np.uint64), G)
        sl = slice(c * G, (c + 1) * G)
        vals = np.stack([B[sl], A[sl], A[sl], B[sl], Cv[sl], Cv[sl]], axis=1).reshape(6 * G, 4)
        rw[8, rs, 0], rw[8, rs, 1], rw[9, rs, 0], rw[9, rs, 1] = vals[:, 0], vals[:, 1], vals[:, 2], vals[:, 3]
        rwf[rs] = 1
        k += 6 * G
        # ---- STOP (root call): IsSuccess read, next = EndTx
        s_stop = sb + 4 * G
        steps[0, s_stop, 0], steps[1, s_stop, 0] = int(ExecutionState.STOP), k + 1
        steps[7, s_stop, 0], steps[8, s_stop, 0] = 68 * G, 1024
        put_rw(k, 0, TAG["cc"], call_id, int(CC.IsSuccess), val=1); k += 1
        # every step of the call: call_id, is_root, code hash, reversible_write_counter 2
        call = slice(sb, s_stop + 2)   # body, STOP and EndTx
        steps[2, call, 0], steps[3, call, 0] = call_id, 1
        steps[5, call, 0], steps[5, call, 1] = int(H[c, 0]), int(H[c, 1])
        steps[6, call, 0], steps[6, call, 1] = int(H[c, 2]), int(H[c, 3])
        steps[11, call, 0] = 2
        # ---- EndTx
        s_end = s_stop + 1
        gas_left = gas_after_begin - int(cost.sum())
        gas_used = gas - gas_left
        steps[0, s_end, 0], steps[1, s_end, 0], steps[9, s_end, 0] = int(ExecutionState.EndTx), k + 1, gas_left
        steps[7, s_end, 0], steps[8, s_end, 0] = 68 * G, 1024
        put_rw(k, 0, TAG["cc"], call_id, int(CC.TxId), val=tx_id); k += 1
        put_rw(k, 0, TAG["cc"], call_id, int(CC.IsPersistent), val=1); k += 1
        put_rw(k, 0, TAG["refund"], tx_id, val=0, prev=0); k += 1
        bal = caller_bal - gas * GAS_PRICE
        put_rw(k, 1, TAG["acc"], 0, caller, int(AF.Balance), val=bal + gas_left * GAS_PRICE, prev=bal, word=True, prev_word=True); k += 1
        reward = gas_used * (GAS_PRICE - BASE_FEE)
        put_rw(k, 1, TAG["acc"], 0, COINBASE, int(AF.Balance), val=coinbase_bal + reward, prev=coinbase_bal, word=True, prev_word=True); k += 1
        coinbase_bal += reward
        put_rw(k, 1, TAG["rcpt"], tx_id, 0, int(RF.PostStateOrStatus), val=1); k += 1
        put_rw(k, 1, TAG["rcpt"], tx_id, 0, int(RF.LogLength), val=0); k += 1
        if t:
            put_rw(k, 0, TAG["rcpt"], tx_id - 1, 0, int(RF.CumulativeGasUsed), val=cum_gas); k += 1
        cum_gas += gas_used
        put_rw(k, 1, TAG["rcpt"], tx_id, 0, int(RF.CumulativeGasUsed), val=cum_gas); k += 1
        if t + 1 < T:  # the next transaction's TxId, looked up with call_id = next.rw_counter
            put_rw(k, 0, TAG["cc"], k + 2, int(CC.TxId), val=tx_id + 1); k += 1
    # ---- EndBlock (the last step): TxId of the last call, cumulative gas of the last tx
    s_eb = T * S_TX
    last_call = int(steps[2, s_eb - 1, 0])
    steps[0, s_eb, 0], steps[1, s_eb, 0], steps[2, s_eb, 0], steps[8, s_eb, 0] = int(ExecutionState.EndBlock), k + 1, last_call, 1024
    put_rw(k, 0, TAG["cc"], last_call, int(CC.TxId), val=T); k += 1
    put_rw(k, 0, TAG["rcpt"], T, 0, int(RF.CumulativeGasUsed), val=cum_gas); k += 1
    assert k == n_real, (k, n_real)
    for q in range(n_padding):  # tail: Start rows, rw_counter 1 ..
        rw[0, n_real + q, 0], rw[2, n_real + q, 0] = q + 1, TAG["start"]
    # dummy step appended by end_with_last_step: StepState(EndBlock, rw_counter = -1)
    steps[0, n_steps, 0] = int(ExecutionState.EndBlock)
    steps[1, n_steps, :] = limbs4(P - 1)
    steps[8, n_steps, 0] = 1024
    # block table
    block = np.zeros((4, 8, 4), dtype=np.uint64)
    bf = np.zeros(8, dtype=np.uint8)
    for q, (v, w_) in enumerate([(COINBASE, 1), (GAS_LIMIT, 0), (0, 0), (0, 0), (0, 1), (BASE_FEE, 1), (1, 0), (0, 0)]):
        block[0, q, 0] = q + 1
        lv = limbs4(v)
        block[2, q, 0], block[2, q, 1], block[3, q, 0], block[3, q, 1] = lv[0], lv[1], lv[2], lv[3]
        bf[q] = w_
    return {"steps": steps, "n_steps": n_steps, "flags": 2 | 4, "bytecode": bytecode, "bytecode_src": src, "rw": rw, "rw_flags": rwf,
            "tx": tx, "tx_flags": txf, "block": block, "block_flags": bf, "wd": np.zeros((4, 0, 4), dtype=np.uint64),
            "copy": np.zeros((14, 0, 4), dtype=np.uint64), "keccak": np.zeros((5, 0, 4), dtype=np.uint64)}


def pi_public_data(n_txs: int, max_calldata: int, n_withdrawals: int, seed: int = 7):
    """seeded random PublicData for the public-inputs circuit, the recipe of the reference's
    tests/test_public_inputs.py:66-128 (rand_block / rand_tx / rand_withdrawal): `n_txs` transactions whose calldata
    (30 % zero bytes) shares `max_calldata` bytes, `n_withdrawals` withdrawals with ids 0.. and a non-zero amount"""
    from . import pi_circuit as pc

    rng = np.random.default_rng(seed)
    r256 = lambda: int.from_bytes(rng.bytes(32), "little")  # noqa: E731
    r160 = lambda: int.from_bytes(rng.bytes(20), "little")  # noqa: E731
    r64 = lambda: int(rng.integers(0, 1 << 63))  # noqa: E731
    block = pc.Block(hash=r256(), parent_hash=r256(), uncle_hash=r256(), coinbase=r160(), state_root=r256(), tx_hash=r256(),
                     receipt_hash=r256(), bloom=rng.bytes(256), prev_randao=r256(), number=r64(), gas_limit=r64(), gas_used=r64(),
                     time=r64(), extra=b"", mix_digest=r256(), nonce=r64(), base_fee=0, withdrawals_root=r256())
    txs = []
    for _ in range(n_txs):
        data = rng.integers(0, 256, int(rng.integers(0, max_calldata // max(1, n_txs) + 1)), dtype=np.uint8)
        data[rng.random(len(data)) < 0.3] = 0
        txs.append(pc.Transaction(r64(), r256(), r64(), r160(), r160(), r256(), bytes(data), r256()))
    wds = [pc.Withdrawal(k, r64(), r160(), 1 + r64()) for k in range(n_withdrawals)]
    return pc.PublicData(int(rng.integers(1, 128)), block, r256(), [r256() for _ in range(256)], txs, wds)


def withdrawals(n: int, max_withdrawals: int, seed: int = 0, ctx=None) -> Dict[str, np.ndarray]:
    """A seeded withdrawal-circuit witness of n withdrawals in a circuit of max_withdrawals rows, built like the
    reference's tests (tests/test_withdrawal_circuit.py: consecutive ids from a random u64, u64 validator ids and amounts,
    160-bit addresses, mock MPT rows with root = prev + 5, one WithdrawalRoot block row).  The rows and the keccak table
    are assigned on the device (Context.assign_withdrawal_circuit: hashes and RLCs from the device), the MPT and block
    tables are built here from the assigned hash cells and uploaded.  Returns the records and the three host matrices
    (rows as downloaded, mpt, block); the context is left with everything resident, ready for a check."""
    from . import native

    ctx = ctx or native.default_context()
    rng = np.random.default_rng(seed)
    rec = np.zeros((n, 5, 4), dtype=np.uint64)
    rec[:, 0, 0] = np.uint64(int(rng.integers(0, 1 << 62))) + np.arange(n, dtype=np.uint64)
    rec[:, 1, 0] = rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, n, dtype=np.uint64)
    rec[:, 2, 0] = rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2)
    rec[:, 2, 1] = rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    rec[:, 2, 2] = rng.integers(0, 1 << 32, n, dtype=np.uint64)
    rec[:, 3, 0] = rng.integers(1, 1 << 63, n, dtype=np.uint64)
    rec[:, 4, 0] = np.uint64(5) * (np.arange(n, dtype=np.uint64) + np.uint64(1))
    ctx.assign_withdrawal_circuit(rec, max_withdrawals)
    rows, _ = ctx.download_columns(native.CIRCUIT_WITHDRAWAL)
    mpt = np.zeros((12, n, 4), dtype=np.uint64)
    mpt[0] = rows[2, :n]
    mpt[1, :, 0] = 8  # MPTProofType.WithdrawalMod
    mpt[2, :, :2] = rows[0, :n, :2]  # Word(id): ids stay below 2^128
    mpt[4] = rows[6, :n]
    mpt[5] = rows[7, :n]
    mpt[6, 1:] = rows[6, :n - 1]
    mpt[7, 1:] = rows[7, :n - 1]
    mpt[8] = rows[4, :n]
    mpt[9] = rows[5, :n]
    block = np.zeros((4, 1, 4), dtype=np.uint64)
    block[0, 0, 0] = 9  # BlockContextFieldTag.WithdrawalRoot
    block[2, 0, 0] = 5 * n
    ctx.upload_table(native.TABLE_MPT, mpt)
    ctx.upload_table(native.TABLE_BLOCK, block)
    ctx.set_challenge(native.PARAM_WITHDRAWAL_MAX, max_withdrawals)
    return {"records": rec, "rows": rows, "mpt": mpt, "block": block, "max": max_withdrawals}
