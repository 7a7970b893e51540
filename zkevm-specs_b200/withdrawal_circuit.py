"""Withdrawal circuit, host side — /root/reference/src/zkevm_specs/withdrawal_circuit.py.

Same names and meaning as the reference: `Row` (:20-44), `MPTTable` (:47-76), `BlockTable` (:79-90),
`KeccakTable` (:93-117, with its all-zero row), `Witness` (:120-124) and
`verify_circuit(witness, MAX_WITHDRAWALS, keccak_randomness)` (:127-201).  The objects only build the witness;
every constraint of the loop, the RLP encoding of each row and its RLC included, is checked on the device by one
zk_check(ZK_CIRCUIT_WITHDRAWAL) (csrc/withdrawal.cu), and the first failure is raised with the reference's
exception class.  The two things the reference fails on before any constraint are Python list indexing: an empty
row list, and fewer rows than MAX_WITHDRAWALS (the next-id read of row len(rows) - 1).  Those raise IndexError here
too, after any failure the device finds on an earlier row."""
from __future__ import annotations

from typing import List, NamedTuple, Optional, Set, Tuple

import numpy as np

from . import native, packing
from .evm_circuit.main import raise_first_failure
from .evm_circuit.table import BlockTableRow, MPTTableRow  # noqa: F401  (re-exported like the reference)
from .state_circuit import mpt_row
from .util.arithmetic import FQ, RLC, Word
from .util.hash import keccak256

N_COLS = 8  # withdrawal_id, validator_id, address, amount, hash lo, hash hi, root lo, root hi (include/zkcheck.h)


class Row:
    """Withdrawal circuit row (withdrawal_circuit.py:20-44)"""

    def __init__(self, withdrawal_id: FQ, validator_id: FQ, address: FQ, amount: FQ, hash: Word, root: Word):
        self.withdrawal_id = withdrawal_id
        self.validator_id = validator_id
        self.address = address
        self.amount = amount
        self.hash = hash
        self.root = root


class MPTTable:
    def __init__(self, mpt_table: Set[MPTTableRow]):
        self.table = mpt_table


class BlockTable:
    def __init__(self, block_table: Set[BlockTableRow]):
        self.table = block_table


def rlp_encode_ints(values) -> bytes:
    """rlp.encode of a list of non-negative integers: each as its minimal big-endian bytes (0 -> 0x80, below 0x80 the
    byte itself, else 0x80 + length and the bytes), the list header 0xc0 + length, or 0xf8 + length from 56 bytes on
    (payloads here stay below 256 bytes)"""
    body = b""
    for v in values:
        v = int(v)
        b = v.to_bytes((v.bit_length() + 7) // 8, "big")
        body += b if len(b) == 1 and b[0] < 0x80 else bytes([0x80 + len(b)]) + b
    assert len(body) < 256
    return (bytes([0xC0 + len(body)]) if len(body) < 56 else bytes([0xF8, len(body)])) + body


def withdrawal_rlp(row: Row) -> bytes:
    return rlp_encode_ints([packing.cell_int(x) for x in (row.withdrawal_id, row.validator_id, row.address, row.amount)])


class KeccakTable:
    """columns (is_enabled, input_rlc, input_len, output) — withdrawal_circuit.py:93-117"""

    def __init__(self) -> None:
        self.table: Set[Tuple[FQ, FQ, FQ, Word]] = {(FQ(0), FQ(0), FQ(0), Word(0))}

    def add(self, input: bytes, keccak_randomness: FQ) -> None:
        self.table.add((FQ(1), RLC(bytes(reversed(input)), keccak_randomness, n_bytes=len(input)).expr(), FQ(len(input)),
                        Word(keccak256(input))))

    def matrix(self) -> np.ndarray:
        c = packing.cell_int
        return packing.matrix_from_ints([[c(a), c(b), c(n), c(o.lo), c(o.hi)] for a, b, n, o in self.table], 5)


class Witness(NamedTuple):
    rows: List[Row]
    mpt_table: MPTTable
    keccak_table: KeccakTable
    block_table: BlockTable


def row_cells(r: Row) -> List[int]:
    c = packing.cell_int
    return [c(r.withdrawal_id), c(r.validator_id), c(r.address), c(r.amount), c(r.hash.lo), c(r.hash.hi), c(r.root.lo),
            c(r.root.hi)]


def pack_rows(rows: List[Row]) -> np.ndarray:
    return packing.matrix_from_ints([row_cells(r) for r in rows], N_COLS)


def pack_tables(witness: Witness):
    """-> (keccak uint64[5][k][4], mpt uint64[12][m][4], block uint64[4][b][4])"""
    return (witness.keccak_table.matrix(), packing.matrix_from_ints([mpt_row(r) for r in witness.mpt_table.table], 12),
            packing.pack(witness.block_table.table, packing.block_table_row, 4))


def check_matrices(ctx: native.Context, rows, keccak, mpt, block, keccak_randomness, max_withdrawals: int, row_begin=0,
                   row_end=None, row_base=0):
    """upload everything and check rows [row_begin, row_end) of `rows` (global rows row_base + local)"""
    ctx.set_challenge(native.CHALLENGE_KECCAK, packing.cell_int(keccak_randomness))
    ctx.set_challenge(native.PARAM_WITHDRAWAL_MAX, int(max_withdrawals))
    ctx.upload_table(native.TABLE_KECCAK, keccak)
    ctx.upload_table(native.TABLE_MPT, mpt)
    ctx.upload_table(native.TABLE_BLOCK, block)
    ctx.upload_columns(native.CIRCUIT_WITHDRAWAL, rows)
    return ctx.check(native.CIRCUIT_WITHDRAWAL, row_begin, rows.shape[1] if row_end is None else row_end, row_base, 0)


def verify_circuit(witness: Witness, MAX_WITHDRAWALS: int, keccak_randomness: FQ,
                   ctx: Optional[native.Context] = None) -> None:
    """Reference signature (withdrawal_circuit.py:127); raises the exception the reference raises first."""
    ctx = ctx or native.default_context()
    rows = witness.rows
    if not rows:  # rows[0] in the loop, or rows[-1] in the block lookup of MAX == 0
        raise IndexError("list index out of range")
    short = 0 < MAX_WITHDRAWALS and len(rows) < MAX_WITHDRAWALS
    if MAX_WITHDRAWALS == 0:
        used, end = rows[-1:], 1  # an empty loop; the block lookup reads rows[-1].root, checked at global row 0
    elif short:
        used, end = rows, len(rows) - 1  # row len(rows) - 1 reads rows[len(rows)] for its next-id check
    else:
        used, end = rows[:MAX_WITHDRAWALS], MAX_WITHDRAWALS  # later rows are never read
    keccak, mpt, block = pack_tables(witness)
    ff, _ = check_matrices(ctx, pack_rows(used), keccak, mpt, block, keccak_randomness, MAX_WITHDRAWALS, 0, end)
    raise_first_failure(ff, native.CIRCUIT_WITHDRAWAL, "Constraints failed for withdrawal_index =")
    if short:
        raise IndexError(f"withdrawal_index = {len(rows) - 1}: rows[{len(rows)}] is out of range")
