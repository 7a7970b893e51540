"""Generate tests/golden/*.npz by running the REFERENCE itself (authoring container only).

    PYTHONPATH=oracle/pyshim:/root/reference/src python tests/golden/gen_golden.py [bytecode|state|copy|evm|all]

The reference (/root/reference, pure Python) is imported through oracle/pyshim (stand-ins
for its absent third-party deps).  For every case we store the witness matrix in the
column-major cell layout of include/zkcheck.h plus what the reference's own driver loop did
on it: pass, or (first failing row, exception class).  Negative cases are seeded single-cell
corruptions of a positive witness, the reference's own negative-test pattern
(tests/test_bytecode_circuit.py:113-313, tests/test_state_circuit.py:113-372).

/root/reference does not exist on the GPU box, so tests only ever read the .npz files.
"""
import dataclasses
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
P = 21888242871839275222246405745257275088548364400416034343698204186575808495617


def limbs(v: int):
    assert 0 <= v < (1 << 256)
    return [(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(4)]


def n_of(x) -> int:
    if hasattr(x, "expr"):
        return x.expr().n
    if hasattr(x, "n"):
        return x.n
    return int(x)


def to_matrix(rows_of_ints):
    """rows_of_ints: list of rows, each a list of python ints -> uint64[n_cols][n_rows][4]"""
    n_rows = len(rows_of_ints)
    n_cols = len(rows_of_ints[0]) if n_rows else 0
    out = np.zeros((n_cols, n_rows, 4), dtype=np.uint64)
    for i, row in enumerate(rows_of_ints):
        for c, v in enumerate(row):
            out[c, i, :] = limbs(v)
    return out


INTERESTING = [0, 1, 2, 3, 255, 256, 0x7F, 0x60, 1 << 64, (1 << 128) - 1, 1 << 128, P - 1]


def corrupt_value(rng: random.Random, old: int) -> int:
    while True:
        k = rng.randrange(6)
        if k == 0:
            v = (old + 1) % P
        elif k == 1:
            v = (old - 1) % P
        elif k == 2:
            v = rng.choice(INTERESTING)
        elif k == 3:
            v = rng.randrange(P)
        elif k == 4:
            v = old ^ (1 << rng.randrange(0, 16))
        else:
            v = rng.randrange(0, 1 << rng.choice([8, 16, 32, 64, 128]))
        if v != old and v < P:
            return v


# --------------------------------------------------------------------------- bytecode
def bytecode_cases():
    from zkevm_specs import bytecode_circuit as bc
    from zkevm_specs.evm_circuit import Bytecode, Opcode, is_push_with_data
    from zkevm_specs.util import FQ, Word

    r = FQ(0x1234567890ABCDEF1122334455667788990011223344556677889900AABBCCDD % P)

    def unroll(code: bytes):
        return bc.UnrolledBytecode(code, list(Bytecode(bytearray(code)).table_assignments()))

    def row_ints(row):
        return [n_of(row.q_first), n_of(row.q_last), n_of(row.hash.lo), n_of(row.hash.hi),
                n_of(row.tag), n_of(row.index), n_of(row.value), n_of(row.is_code),
                n_of(row.push_data_left), n_of(row.value_rlc), n_of(row.length),
                n_of(row.push_data_size)]

    FIELDS = ["q_first", "q_last", "hash.lo", "hash.hi", "tag", "index", "value", "is_code",
              "push_data_left", "value_rlc", "length", "push_data_size"]

    def set_cell(row, col, v):
        f = FIELDS[col]
        if f == "hash.lo":
            return dataclasses.replace(row, hash=Word((FQ(v), row.hash.hi), check=False))
        if f == "hash.hi":
            return dataclasses.replace(row, hash=Word((row.hash.lo, FQ(v)), check=False))
        return dataclasses.replace(row, **{f: FQ(v)})

    def run(rows, push_table, keccak_table):
        """the reference driver loop, tests/test_bytecode_circuit.py:26-47"""
        for idx, row in enumerate(rows):
            try:
                bc.check_bytecode_row(row, rows[(idx + 1) % len(rows)], push_table, keccak_table, r)
            except Exception as e:  # noqa: BLE001
                return idx, type(e).__name__
        return -1, ""

    all_bytes = []
    for b in range(256):
        if not is_push_with_data(b):
            all_bytes.append(b)
    for n in range(1, 33):
        all_bytes.append(int(Opcode.PUSH0) + n)
        all_bytes.extend([int(Opcode.PUSH32)] * n)

    rng = random.Random(1)
    cfg1_code = bytes(np.random.default_rng(1).integers(0, 256, 32, dtype=np.uint8))
    positives = {
        "unrolling_all_bytes": (10, [bytes(all_bytes)]),
        "empty": (6, [b""]),
        "full": (6, [bytes([7] * (2**6 - 2)), b""]),
        "incomplete": (6, [bytes([7] * (2**6 + 1))]),
        "multiple": (6, [b"", bytes([0x7F]), bytes([0x7F, 1]), bytes([1, 0x7F]), bytes([1, 0x7F, 1])]),
        "small": (5, [bytes([8, 2, 3, 8, 9, 7, 128])]),
        "is_code": (5, [bytes([0x01, 0x60, 0x60, 0x03, 0x66, 0x01, 0x65])]),
        "cfg1_32byte_contract": (10, [cfg1_code]),
        "truncated_push": (5, [bytes([0x61, 0xAA]), bytes([0x7F] * 5)]),
    }
    cases = []
    for name, (k, codes) in positives.items():
        unrolled = [unroll(c) for c in codes]
        rows = bc.assign_bytecode_circuit(k, unrolled, r)
        push_table = bc.assign_push_table()
        keccak_table = bc.assign_keccak_table(codes, r)
        push_m = to_matrix([[n_of(a), n_of(b)] for a, b in push_table])
        kec_m = to_matrix([[n_of(x.state_tag), n_of(x.input_rlc), n_of(x.input_len),
                            n_of(x.output.lo), n_of(x.output.hi)] for x in keccak_table])
        base = to_matrix([row_ints(x) for x in rows])
        fail_row, exc = run(rows, push_table, keccak_table)
        muts = [(-1, -1, 0, fail_row, exc)]
        n_mut = 60 if len(rows) <= 64 else 40
        live = max(2, sum(len(c) + 1 for c in codes) + 2)
        for _ in range(n_mut):
            i = rng.randrange(min(len(rows), live)) if rng.random() < 0.8 else rng.randrange(len(rows))
            c = rng.randrange(12)
            old = row_ints(rows[i])[c]
            v = corrupt_value(rng, old)
            bad = list(rows)
            bad[i] = set_cell(rows[i], c, v)
            fr_, ex_ = run(bad, push_table, keccak_table)
            muts.append((i, c, v, fr_, ex_))
        # corrupting the tables instead of the witness
        for _ in range(6):
            kt = list(keccak_table)
            if kt:
                j = rng.randrange(len(kt))
                kt[j] = dataclasses.replace(kt[j], input_len=FQ(n_of(kt[j].input_len) + 1))
                fr_, ex_ = run(rows, push_table, set(kt))
                # encode a table mutation as col = 100 + table col, row = table row (keccak col 2)
                # the stored keccak table is the ORIGINAL; the loader re-applies the mutation
                muts.append((1000 + j, 102, n_of(kt[j].input_len), fr_, ex_))
                break
        cases.append((name, base, push_m, kec_m, muts))
    out = {"r": np.array(limbs(r.n), dtype=np.uint64), "names": np.array([c[0] for c in cases])}
    for name, base, push_m, kec_m, muts in cases:
        out[f"{name}/cols"] = base
        out[f"{name}/push"] = push_m
        out[f"{name}/keccak"] = kec_m
        out[f"{name}/mut_row"] = np.array([m[0] for m in muts], dtype=np.int64)
        out[f"{name}/mut_col"] = np.array([m[1] for m in muts], dtype=np.int64)
        out[f"{name}/mut_val"] = np.array([limbs(m[2]) for m in muts], dtype=np.uint64)
        out[f"{name}/exp_row"] = np.array([m[3] for m in muts], dtype=np.int64)
        out[f"{name}/exp_exc"] = np.array([m[4] for m in muts])
    np.savez_compressed(os.path.join(HERE, "bytecode.npz"), **out)
    n_fail = sum(1 for c in cases for m in c[4] if m[3] >= 0)
    n_all = sum(len(c[4]) for c in cases)
    print(f"bytecode: {len(cases)} witnesses, {n_all} vectors ({n_fail} failing)")


# --------------------------------------------------------------------------- evm
def evm_cases():
    """cfg2-style straight-line traces `PUSH32 b, PUSH32 a, OP, POP` (+ final STOP as the last
    `next`), verified by the reference's verify_step loop (main.py:34-46), plus seeded
    corruptions of step cells, rw-table cells and bytecode-table cells."""
    import copy

    from zkevm_specs.evm_circuit import (Bytecode, ExecutionState, Opcode, RWDictionary, StepState,
                                         Tables, Block, RWTableRow, BytecodeTableRow)
    from zkevm_specs.evm_circuit.instruction import Instruction
    from zkevm_specs.evm_circuit.main import verify_step
    from zkevm_specs.util import FQ, Word, WordOrValue

    sys.path.insert(0, os.path.join(HERE, "..", ".."))
    from zkevm_specs_b200.evm_circuit.table import fixed_table_matrix

    # our arithmetic fixed-table generator must reproduce the reference's set exactly
    ours = fixed_table_matrix()
    ours_set = set(tuple(sum(int(ours[c, i, k]) << (64 * k) for k in range(4)) for c in range(4))
                   for i in range(ours.shape[1]))
    ref_set = set((n_of(r.tag), n_of(r.value0), n_of(r.value1), n_of(r.value2)) for r in Tables.fixed_table)
    assert ours_set == ref_set and len(ours_set) == ours.shape[1], "fixed table mismatch"
    print("fixed table: ours == reference,", len(ref_set), "rows")

    M256 = (1 << 256) - 1
    NASTY = [(0, 0), (1, 0), (0, 1), (255, 256), (260, 513), (65535, 65536), (M256, M256 - 1),
             (M256 - 1, M256), (M256, 0), (0, M256), (1 << 128, (1 << 128) - 1), (7, 3), (M256, 2)]

    def build_trace(ops, rng):
        """returns (steps, bytecode_rows, rw_rows)"""
        bc = Bytecode()
        groups = []
        for op in ops:
            if rng.random() < 0.5:
                a, b = rng.choice(NASTY)
            elif rng.random() < 0.5:
                a, b = rng.randrange(1 << 64), rng.randrange(1, 1 << 64)
            else:
                a, b = rng.randrange(1 << 256), rng.randrange(1 << 256)
            bc.push32(b).push32(a)
            getattr(bc, op.lower())()
            bc.pop()
            groups.append((op, a, b))
        bc.stop()
        code_hash = Word(bc.hash())
        rw = RWDictionary(1)
        steps = []
        pc, sp, gas = 0, 1024, 3 * 2 * len(ops) + 5 * len(ops) + 2 * len(ops) + 40
        call_id = 1

        def step(state):
            steps.append(StepState(execution_state=state, rw_counter=rw.rw_counter, call_id=call_id,
                                   is_root=True, is_create=False, code_hash=code_hash,
                                   program_counter=pc, stack_pointer=sp, gas_left=gas))

        for op, a, b in groups:
            step(ExecutionState.PUSH); rw.stack_write(call_id, sp - 1, Word(b)); pc += 33; sp -= 1; gas -= 3
            step(ExecutionState.PUSH); rw.stack_write(call_id, sp - 1, Word(a)); pc += 33; sp -= 1; gas -= 3
            if op == "ADD":
                c, st, g = (a + b) & M256, ExecutionState.ADD, 3
            elif op == "SUB":
                c, st, g = (a - b) & M256, ExecutionState.ADD, 3
            elif op == "MUL":
                c, st, g = (a * b) & M256, ExecutionState.MUL, 5
            elif op == "DIV":
                c, st, g = (0 if b == 0 else a // b), ExecutionState.MUL, 5
            else:
                c, st, g = (0 if b == 0 else a % b), ExecutionState.MUL, 5
            step(st)
            rw.stack_read(call_id, sp, Word(a)); rw.stack_read(call_id, sp + 1, Word(b))
            rw.stack_write(call_id, sp + 1, Word(c)); pc += 1; sp += 1; gas -= g
            step(ExecutionState.POP); rw.stack_read(call_id, sp, Word(c)); pc += 1; sp += 1; gas -= 2
        step(ExecutionState.STOP)
        return steps, list(bc.table_assignments()), list(rw.rws)

    def step_ints(s):
        return [int(s.execution_state), n_of(s.rw_counter), n_of(s.call_id), int(s.is_root), int(s.is_create),
                n_of(s.code_hash.lo), n_of(s.code_hash.hi), n_of(s.program_counter), n_of(s.stack_pointer),
                n_of(s.gas_left), n_of(s.memory_word_size), n_of(s.reversible_write_counter), n_of(s.log_id)]

    def bc_ints(r):
        return [n_of(r.bytecode_hash.lo), n_of(r.bytecode_hash.hi), n_of(r.field_tag), n_of(r.index),
                n_of(r.is_code), n_of(r.value)]

    def rw_ints(r):
        return [n_of(r.rw_counter), n_of(r.rw), n_of(r.key0), n_of(r.id), n_of(r.address), n_of(r.field_tag),
                n_of(r.storage_key.lo), n_of(r.storage_key.hi), n_of(r.value.lo), n_of(r.value.hi),
                n_of(r.value_prev.lo), n_of(r.value_prev.hi), n_of(r.aux0.lo), n_of(r.aux0.hi)]

    def step_from_ints(v):
        s = StepState(execution_state=ExecutionState(v[0]), rw_counter=0)
        s.rw_counter, s.call_id = FQ(v[1]), FQ(v[2])
        s.is_root, s.is_create = v[3], v[4]  # ints: the reference wraps ints with FQ() (instruction.py:233)
        s.code_hash = Word((FQ(v[5]), FQ(v[6])), check=False)
        s.program_counter, s.stack_pointer, s.gas_left = FQ(v[7]), FQ(v[8]), FQ(v[9])
        s.memory_word_size, s.reversible_write_counter, s.log_id = FQ(v[10]), FQ(v[11]), FQ(v[12])
        return s

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def rw_from_ints(v):
        return RWTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), FQ(v[3]), FQ(v[4]), FQ(v[5]), W(v[6], v[7]),
                          WordOrValue(W(v[8], v[9])), WordOrValue(W(v[10], v[11])), W(v[12], v[13]))

    def bc_from_ints(v):
        return BytecodeTableRow(W(v[0], v[1]), FQ(v[2]), FQ(v[3]), FQ(v[4]), FQ(v[5]))

    def run(step_rows, bc_rows, rw_rows, first=False, last=False):
        steps = [step_from_ints(v) for v in step_rows]
        tables = Tables(block_table=set(Block().table_assignments()), tx_table=set(), withdrawal_table=set(),
                        bytecode_table=set(bc_from_ints(v) for v in bc_rows),
                        rw_table=set(rw_from_ints(v) for v in rw_rows))
        for idx, (curr, nxt) in enumerate(zip(steps, steps[1:])):
            try:
                verify_step(Instruction(tables=tables, curr=curr, next=nxt,
                                        is_first_step=first and idx == 0,
                                        is_last_step=last and idx == len(steps) - 2))
            except Exception as e:  # noqa: BLE001
                return idx, type(e).__name__
        return -1, ""

    valid_states = [int(s) for s in ExecutionState]
    rng = random.Random(2)
    traces = {
        "add_sub": ["ADD", "SUB", "ADD"],
        "mul_div_mod": ["MUL", "DIV", "MOD"],
        "mixed5": ["ADD", "SUB", "MUL", "DIV", "MOD"],
        "divmod_nasty": ["DIV", "MOD", "DIV", "MOD"],
    }
    out = {"names": np.array(list(traces.keys()))}
    tot = nfail = 0
    for name, ops in traces.items():
        steps, bcs, rws = build_trace(ops, rng)
        S = [step_ints(s) for s in steps]
        B = [bc_ints(r) for r in bcs]
        R = [rw_ints(r) for r in rws]
        assert run(S, B, R) == (-1, ""), (name, run(S, B, R))
        muts = [(0, -1, -1, 0, -1, "")]
        n_mut = 70
        for k in range(n_mut):
            which = rng.choice([0, 0, 0, 1, 1, 2])
            S2, B2, R2 = [list(x) for x in S], [list(x) for x in B], [list(x) for x in R]
            if which == 0:
                i, c = rng.randrange(len(S)), rng.randrange(13)
                old = S[i][c]
                if c == 0:
                    v = rng.choice([x for x in valid_states if x != old] if rng.random() < 0.5 else
                                   [int(ExecutionState.ADD), int(ExecutionState.MUL), int(ExecutionState.PUSH),
                                    int(ExecutionState.POP), int(ExecutionState.STOP), int(ExecutionState.EndTx),
                                    int(ExecutionState.BeginTx), int(ExecutionState.EndBlock)])
                    if v == old:
                        continue
                elif c in (3, 4):
                    v = 1 - old
                else:
                    v = corrupt_value(rng, old)
                S2[i][c] = v
            elif which == 1:
                i, c = rng.randrange(len(R)), rng.randrange(14)
                v = corrupt_value(rng, R[i][c])
                R2[i][c] = v
            else:
                i = rng.randrange(len(B)) if rng.random() < 0.5 else rng.choice(
                    [0, 1, 34, 67, 68, 69, len(B) - 1])
                i = min(i, len(B) - 1)
                c = rng.randrange(6)
                v = corrupt_value(rng, B[i][c])
                B2[i][c] = v
            fr_, ex_ = run(S2, B2, R2)
            muts.append((which, i, c, v, fr_, ex_))
            tot += 1
            nfail += fr_ >= 0
        # duplicate-row ambiguity: add a second rw row equal on the queried key, different value
        for i in (0, 2, 5):
            if i < len(R):
                dup = list(R[i]); dup[8] = (dup[8] + 1) % (1 << 128)
                fr_, ex_ = run(S, B, R + [dup])
                muts.append((3, i, 8, dup[8], fr_, ex_))
        dupb = list(B[1]); dupb[5] = (dupb[5] + 1) % 256
        fr_, ex_ = run(S, B + [dupb], R)
        muts.append((4, 1, 5, dupb[5], fr_, ex_))
        # first / last step flags
        fr_, ex_ = run(S, B, R, first=True)
        muts.append((5, 0, 0, 0, fr_, ex_))
        out[f"{name}/steps"] = to_matrix(S)
        out[f"{name}/bytecode"] = to_matrix(B)
        out[f"{name}/rw"] = to_matrix(R)
        out[f"{name}/mut_kind"] = np.array([m[0] for m in muts], dtype=np.int64)
        out[f"{name}/mut_row"] = np.array([m[1] for m in muts], dtype=np.int64)
        out[f"{name}/mut_col"] = np.array([m[2] for m in muts], dtype=np.int64)
        out[f"{name}/mut_val"] = np.array([limbs(m[3]) for m in muts], dtype=np.uint64)
        out[f"{name}/exp_row"] = np.array([m[4] for m in muts], dtype=np.int64)
        out[f"{name}/exp_exc"] = np.array([m[5] for m in muts])
        print(name, len(S), "steps", len(B), "bytecode rows", len(R), "rw rows", len(muts), "vectors")
    np.savez_compressed(os.path.join(HERE, "evm.npz"), **out)
    print(f"evm: {tot} corruptions, {nfail} failing")


# --------------------------------------------------------------------------- copy
def copy_cases():
    """Copy-circuit events built with the reference's CopyCircuit (typing.py:996-1150) and checked
    by the reference's verify_copy_table (copy_circuit.py:92-130); the failing row is recovered
    by tracking the row iterator.  Corruptions: copy rows, rw / tx / bytecode table cells."""
    from zkevm_specs import copy_circuit as cc
    from zkevm_specs.evm_circuit import (Bytecode, Block, CopyCircuit, CopyCircuitRow, CopyDataTypeTag,
                                         RWDictionary, RWTableRow, BytecodeTableRow, Tables, TxTableRow,
                                         TxContextFieldTag)
    from zkevm_specs.util import FQ, Word, WordOrValue

    r = FQ(0x0FEDCBA9876543210FEDCBA9876543210FEDCBA9876543210FEDCBA987654321 % P)
    rng = random.Random(4)

    class Tracking(list):
        def __iter__(self):
            for idx in range(len(self)):
                self.last = idx
                yield list.__getitem__(self, idx)

    class FakeCircuit:
        def __init__(self, rows):
            self.rows = Tracking(rows)

        def table(self):
            return self.rows

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def wov(lo, hi, is_word):
        return WordOrValue(W(lo, hi)) if is_word else WordOrValue(FQ(lo))

    # ---- row <-> ints -------------------------------------------------------------------
    def copy_ints(x):
        return [n_of(x.q_step), n_of(x.is_first), n_of(x.is_last), n_of(x.id.lo), n_of(x.id.hi), n_of(x.tag),
                n_of(x.addr), n_of(x.src_addr_end), n_of(x.bytes_left), n_of(x.value), n_of(x.rlc_acc),
                n_of(x.is_code), n_of(x.is_pad), n_of(x.rw_counter), n_of(x.rwc_inc_left), n_of(x.is_memory),
                n_of(x.is_bytecode), n_of(x.is_tx_calldata), n_of(x.is_tx_log), n_of(x.is_rlc_acc)]

    def copy_from(v, flag):
        f = [FQ(x) for x in v]
        return CopyCircuitRow(f[0], f[1], f[2], wov(v[3], v[4], flag & 1), *f[5:])

    def rw_ints(x):
        return [n_of(x.rw_counter), n_of(x.rw), n_of(x.key0), n_of(x.id), n_of(x.address), n_of(x.field_tag),
                n_of(x.storage_key.lo), n_of(x.storage_key.hi), n_of(x.value.lo), n_of(x.value.hi),
                n_of(x.value_prev.lo), n_of(x.value_prev.hi), n_of(x.aux0.lo), n_of(x.aux0.hi)]

    def rw_from(v, flag):
        return RWTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), FQ(v[3]), FQ(v[4]), FQ(v[5]), W(v[6], v[7]),
                          wov(v[8], v[9], flag & 1), wov(v[10], v[11], (flag >> 1) & 1), W(v[12], v[13]))

    def tx_ints(x):
        return [n_of(x.tx_id), n_of(x.field_tag), n_of(x.call_data_index_or_zero), n_of(x.value.lo), n_of(x.value.hi)]

    def tx_from(v, flag):
        return TxTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), wov(v[3], v[4], flag & 1))

    def bc_ints(x):
        return [n_of(x.bytecode_hash.lo), n_of(x.bytecode_hash.hi), n_of(x.field_tag), n_of(x.index),
                n_of(x.is_code), n_of(x.value)]

    def bc_from(v):
        return BytecodeTableRow(W(v[0], v[1]), FQ(v[2]), FQ(v[3]), FQ(v[4]), FQ(v[5]))

    def run(C, CF, RW, RWF, TX, TXF, BC):
        fake = FakeCircuit([copy_from(v, f) for v, f in zip(C, CF)])
        tables = Tables(block_table=set(Block().table_assignments()),
                        tx_table=set(tx_from(v, f) for v, f in zip(TX, TXF)), withdrawal_table=set(),
                        bytecode_table=set(bc_from(v) for v in BC),
                        rw_table=set(rw_from(v, f) for v, f in zip(RW, RWF)))
        try:
            cc.verify_copy_table(fake, tables, r)
        except Exception as e:  # noqa: BLE001
            return fake.rows.last, type(e).__name__
        return -1, ""

    def scenario(kind):
        circ, rw = CopyCircuit(), RWDictionary(10)
        code = Bytecode().push32(0x1234).push1(7).add().stop()
        bc_rows = list(code.table_assignments())
        tx_rows = []
        if kind in ("sha3", "mix"):
            data = {100 + k: rng.randrange(256) for k in range(6)}
            for a, b in data.items():
                rw.memory_write(1, a, b)
            circ.copy(r, rw, 1, CopyDataTypeTag.Memory, 1, CopyDataTypeTag.RlcAcc, 100, 106, 0, 6, data)
        if kind in ("calldata", "mix"):
            calldata = [rng.randrange(256) for _ in range(5)]
            tx_rows = [TxTableRow(FQ(3), FQ(TxContextFieldTag.CallData), FQ(k), WordOrValue(FQ(b)))
                       for k, b in enumerate(calldata)]
            # 7 bytes requested from offset 1, only 4 exist -> 3 padded reads
            circ.copy(r, rw, 3, CopyDataTypeTag.TxCalldata, 1, CopyDataTypeTag.Memory, 1, 5, 32, 7,
                      {k: b for k, b in enumerate(calldata)})
        if kind in ("codecopy", "mix"):
            src = {k: (code.code[k], code.is_code[k]) for k in range(len(code.code))}
            circ.copy(r, rw, Word(code.hash()), CopyDataTypeTag.Bytecode, 1, CopyDataTypeTag.Memory, 30,
                      len(code.code), 64, 8, src)
        if kind in ("log", "mix"):
            data = {200 + k: rng.randrange(256) for k in range(4)}
            for a, b in data.items():
                rw.memory_write(1, a, b)
            circ.copy(r, rw, 1, CopyDataTypeTag.Memory, 2, CopyDataTypeTag.TxLog, 200, 204, 0, 4, data, log_id=1)
        return list(circ.table()), list(rw.rws), tx_rows, bc_rows

    out = {"r": np.array(limbs(r.n), dtype=np.uint64), "names": np.array(["sha3", "calldata", "codecopy", "log", "mix"])}
    tot = nfail = 0
    for name in ["sha3", "calldata", "codecopy", "log", "mix"]:
        rows, rws, txs, bcs = scenario(name)
        C = [copy_ints(x) for x in rows]
        CF = [int(x.id.is_word) for x in rows]
        RW = [rw_ints(x) for x in rws]
        RWF = [int(x.value.is_word) | (int(x.value_prev.is_word) << 1) for x in rws]
        TX = [tx_ints(x) for x in txs]
        TXF = [int(x.value.is_word) for x in txs]
        BC = [bc_ints(x) for x in bcs]
        assert run(C, CF, RW, RWF, TX, TXF, BC) == (-1, ""), (name, run(C, CF, RW, RWF, TX, TXF, BC))
        muts = [(-1, 0, 0, 0, -1, "")]
        for k in range(90 if name == "mix" else 45):
            which = rng.choice([0, 0, 0, 0, 1, 1, 2, 3, 4, 5])
            C2, CF2, RW2, RWF2, TX2, TXF2, BC2 = ([list(x) for x in C], list(CF), [list(x) for x in RW], list(RWF),
                                                  [list(x) for x in TX], list(TXF), [list(x) for x in BC])
            if which == 0:
                i, c = rng.randrange(len(C)), rng.randrange(20)
                if c == 4 and not CF[i]:
                    continue  # a value-typed id has no hi cell in the reference (WordOrValue.hi is FQ(0))
                v = (1 - C[i][c]) if (C[i][c] in (0, 1) and rng.random() < 0.5) else corrupt_value(rng, C[i][c])
                C2[i][c] = v
            elif which == 1 and RW:
                i, c = rng.randrange(len(RW)), rng.randrange(10)
                v = corrupt_value(rng, RW[i][c]); RW2[i][c] = v
            elif which == 2 and TX:
                i, c = rng.randrange(len(TX)), rng.randrange(5)
                v = corrupt_value(rng, TX[i][c]); TX2[i][c] = v
            elif which == 3:
                i, c = rng.randrange(len(BC)), rng.randrange(6)
                v = corrupt_value(rng, BC[i][c]); BC2[i][c] = v
            elif which == 4:  # flip the is_word type flag of a copy row id
                i, c, v = rng.randrange(len(C)), 100, 0
                CF2[i] ^= 1
                if not CF2[i]:
                    C2[i][4] = 0  # Word -> value: the hi half disappears with the type
            elif which == 5 and RW:  # flip the is_word flag of an rw value, or duplicate an rw row
                i = rng.randrange(len(RW))
                if rng.random() < 0.5:
                    c, v = 101, 0
                    RWF2[i] ^= 1
                else:
                    c, v = 102, (RW[i][8] + 1) % 256
                    dup = list(RW[i]); dup[8] = v
                    RW2.append(dup); RWF2.append(RWF[i])
            else:
                continue
            fr_, ex_ = run(C2, CF2, RW2, RWF2, TX2, TXF2, BC2)
            muts.append((which, i, c, v, fr_, ex_))
            tot += 1
            nfail += fr_ >= 0
        out[f"{name}/copy"] = to_matrix(C)
        out[f"{name}/copy_flags"] = np.array(CF, dtype=np.uint8)
        out[f"{name}/rw"] = to_matrix(RW) if RW else np.zeros((14, 0, 4), dtype=np.uint64)
        out[f"{name}/rw_flags"] = np.array(RWF, dtype=np.uint8)
        out[f"{name}/tx"] = to_matrix(TX) if TX else np.zeros((5, 0, 4), dtype=np.uint64)
        out[f"{name}/tx_flags"] = np.array(TXF, dtype=np.uint8)
        out[f"{name}/bytecode"] = to_matrix(BC)
        out[f"{name}/mut_kind"] = np.array([m[0] for m in muts], dtype=np.int64)
        out[f"{name}/mut_row"] = np.array([m[1] for m in muts], dtype=np.int64)
        out[f"{name}/mut_col"] = np.array([m[2] for m in muts], dtype=np.int64)
        out[f"{name}/mut_val"] = np.array([limbs(m[3]) for m in muts], dtype=np.uint64)
        out[f"{name}/exp_row"] = np.array([m[4] for m in muts], dtype=np.int64)
        out[f"{name}/exp_exc"] = np.array([m[5] for m in muts])
        print(name, len(C), "copy rows", len(RW), "rw", len(TX), "tx", len(BC), "bytecode", len(muts), "vectors")
    np.savez_compressed(os.path.join(HERE, "copy.npz"), **out)
    print(f"copy: {tot} corruptions, {nfail} failing")


# --------------------------------------------------------------------------- state
def state_cases():
    """State-circuit rows assigned by the reference (assign_state_circuit, state_circuit.py:861-889)
    from operation lists modelled on tests/test_state_circuit.py:41-110, checked by the reference's
    check_state_row under its own driver loop (tests/test_state_circuit.py:17-38)."""
    import zkevm_specs.state_circuit as sc
    from zkevm_specs.evm_circuit import (RW, AccountFieldTag, CallContextFieldTag, TxLogFieldTag,
                                         TxReceiptFieldTag, MPTTableRow)
    from zkevm_specs.util import FQ, Word, WordOrValue

    rng = random.Random(3)
    R_, W_ = RW.Read, RW.Write

    def ops_all():
        return [
            sc.StartOp(rw_counter=1, rw=R_, lexicographic_ordering_selector=0),
            sc.StartOp(rw_counter=2, rw=R_),
            sc.StartOp(rw_counter=3, rw=R_),
            sc.MemoryOp(rw_counter=1, rw=R_, call_id=1, mem_addr=0, value=FQ(0)),
            sc.MemoryOp(rw_counter=2, rw=W_, call_id=1, mem_addr=0, value=FQ(42)),
            sc.MemoryOp(rw_counter=3, rw=R_, call_id=1, mem_addr=0, value=FQ(42)),
            sc.MemoryOp(rw_counter=40, rw=W_, call_id=1, mem_addr=7, value=FQ(255)),
            sc.StackOp(rw_counter=4, rw=W_, call_id=1, stack_ptr=1022, value=Word(4321)),
            sc.StackOp(rw_counter=5, rw=W_, call_id=1, stack_ptr=1023, value=Word(533)),
            sc.StackOp(rw_counter=6, rw=R_, call_id=1, stack_ptr=1023, value=Word(533)),
            sc.StorageOp(rw_counter=7, rw=R_, tx_id=1, addr=0x12345678, key=0x1516, value=Word(789), committed_value=Word(789)),
            sc.StorageOp(rw_counter=8, rw=W_, tx_id=1, addr=0x12345678, key=0x4959, value=Word(38491), committed_value=Word(98765)),
            sc.CallContextOp(rw_counter=9, rw=R_, call_id=1, field_tag=CallContextFieldTag.IsStatic, value=FQ(0)),
            sc.CallContextOp(rw_counter=10, rw=R_, call_id=2, field_tag=CallContextFieldTag.IsStatic, value=FQ(0)),
            sc.AccountOp(rw_counter=12, rw=W_, addr=0x12345678, field_tag=AccountFieldTag.Nonce, value=FQ(1), committed_value=FQ(0)),
            sc.AccountOp(rw_counter=13, rw=R_, addr=0x12345678, field_tag=AccountFieldTag.Nonce, value=FQ(1), committed_value=FQ(0)),
            sc.AccountOp(rw_counter=42, rw=R_, addr=0x12345678, field_tag=AccountFieldTag.Balance, value=Word(3), committed_value=Word(0)),
            sc.TxRefundOp(rw_counter=14, rw=W_, tx_id=1, value=FQ(1)),
            sc.TxRefundOp(rw_counter=15, rw=W_, tx_id=1, value=FQ(1)),
            sc.TxAccessListAccountOp(rw_counter=16, rw=R_, tx_id=1, addr=0x12345678, value=FQ(0)),
            sc.TxAccessListAccountOp(rw_counter=17, rw=W_, tx_id=1, addr=0x12345678, value=FQ(1)),
            sc.TxAccessListAccountStorageOp(rw_counter=18, rw=R_, tx_id=1, addr=0x12345678, key=0x1516, value=FQ(0)),
            sc.TxAccessListAccountStorageOp(rw_counter=19, rw=W_, tx_id=1, addr=0x12345678, key=0x1516, value=FQ(1)),
            sc.TxLogOp(rw_counter=20, rw=W_, tx_id=1, log_id=1, field_tag=TxLogFieldTag.Address, index=0, value=FQ(124)),
            sc.TxLogOp(rw_counter=21, rw=W_, tx_id=1, log_id=1, field_tag=TxLogFieldTag.Topic, index=0, value=Word(10)),
            sc.TxLogOp(rw_counter=22, rw=W_, tx_id=1, log_id=1, field_tag=TxLogFieldTag.Topic, index=1, value=Word(5)),
            sc.TxLogOp(rw_counter=25, rw=W_, tx_id=1, log_id=1, field_tag=TxLogFieldTag.Data, index=0, value=FQ(10)),
            sc.TxLogOp(rw_counter=27, rw=W_, tx_id=1, log_id=2, field_tag=TxLogFieldTag.Address, index=0, value=FQ(255)),
            sc.TxLogOp(rw_counter=29, rw=W_, tx_id=2, log_id=1, field_tag=TxLogFieldTag.Address, index=0, value=FQ(210)),
            sc.TxReceiptOp(rw_counter=32, rw=R_, tx_id=1, field_tag=TxReceiptFieldTag.PostStateOrStatus, value=FQ(1)),
            sc.TxReceiptOp(rw_counter=33, rw=R_, tx_id=1, field_tag=TxReceiptFieldTag.CumulativeGasUsed, value=FQ(200)),
            sc.TxReceiptOp(rw_counter=34, rw=R_, tx_id=2, field_tag=TxReceiptFieldTag.PostStateOrStatus, value=FQ(1)),
            sc.TxReceiptOp(rw_counter=35, rw=R_, tx_id=2, field_tag=TxReceiptFieldTag.CumulativeGasUsed, value=FQ(500)),
        ]

    def ops_mem_stack():
        ops = [sc.StartOp(rw_counter=1, rw=R_, lexicographic_ordering_selector=0), sc.StartOp(rw_counter=2, rw=R_)]
        rwc = 1
        for call in (1, 2):
            for a in range(6):
                ops.append(sc.MemoryOp(rw_counter=rwc, rw=W_, call_id=call, mem_addr=a * 3, value=FQ(rng.randrange(256)))); rwc += 1
                ops.append(sc.MemoryOp(rw_counter=rwc, rw=R_, call_id=call, mem_addr=a * 3, value=ops[-1].value.lo)); rwc += 1
        for call in (1, 2):
            for sp in (1021, 1022, 1023):
                v = Word(rng.randrange(1 << 256))
                ops.append(sc.StackOp(rw_counter=rwc, rw=W_, call_id=call, stack_ptr=sp, value=v)); rwc += 1
                ops.append(sc.StackOp(rw_counter=rwc, rw=R_, call_id=call, stack_ptr=sp, value=v)); rwc += 1
        return ops

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def wov(lo, hi, is_word):
        return WordOrValue(W(lo, hi)) if is_word else WordOrValue(FQ(lo))

    def row_ints(x):
        return ([n_of(x.rw_counter), n_of(x.is_write)] + [n_of(k) for k in x.keys[:4]] +
                [n_of(x.keys[4].lo), n_of(x.keys[4].hi)] + [n_of(l) for l in x.key2_limbs] +
                [n_of(b) for b in x.key45_bytes] + [n_of(x.value.lo), n_of(x.value.hi), n_of(x.initial_value.lo),
                                                    n_of(x.initial_value.hi), n_of(x.root.lo), n_of(x.root.hi),
                                                    n_of(x.lexicographic_ordering_selector)])

    def row_from(v, flag):
        f = [FQ(x) for x in v]
        return sc.Row(f[0], f[1], (f[2], f[3], f[4], f[5], W(v[6], v[7])), tuple(f[8:18]), tuple(f[18:50]),
                      wov(v[50], v[51], flag & 1), wov(v[52], v[53], (flag >> 1) & 1), W(v[54], v[55]), f[56])

    def mpt_ints(x):
        return [n_of(x.address), n_of(x.proof_type), n_of(x.storage_key.lo), n_of(x.storage_key.hi), n_of(x.root.lo),
                n_of(x.root.hi), n_of(x.root_prev.lo), n_of(x.root_prev.hi), n_of(x.value.lo), n_of(x.value.hi),
                n_of(x.value_prev.lo), n_of(x.value_prev.hi)]

    def mpt_from(v):
        return MPTTableRow(FQ(v[0]), FQ(v[1]), W(v[2], v[3]), W(v[4], v[5]), W(v[6], v[7]), W(v[8], v[9]), W(v[10], v[11]))

    def run(S, SF, M):
        rows = [row_from(v, f) for v, f in zip(S, SF)]
        tables = sc.Tables(set(mpt_from(v) for v in M))
        for idx, row in enumerate(rows):
            try:
                sc.check_state_row(row, rows[(idx - 1) % len(rows)], rows[(idx + 1) % len(rows)], tables)
            except Exception as e:  # noqa: BLE001
                return idx, type(e).__name__
        return -1, ""

    out = {"names": np.array(["all_tags", "mem_stack"])}
    tot = nfail = 0
    for name, ops in (("all_tags", ops_all()), ("mem_stack", ops_mem_stack())):
        ops = sorted(ops, key=lambda o: (0 if isinstance(o, sc.StartOp) else 1, int(o.tag), int(o.id), int(o.address),
                                         int(o.field_tag), int(o.storage_key), o.rw_counter)) if name == "mem_stack" else ops
        rows = sc.assign_state_circuit(ops)
        mpt = list(sc.mpt_table_from_ops(ops))
        S = [row_ints(x) for x in rows]
        SF = [int(x.value.is_word) | (int(x.initial_value.is_word) << 1) for x in rows]
        M = [mpt_ints(x) for x in mpt]
        assert run(S, SF, M) == (-1, ""), (name, run(S, SF, M))
        muts = [(-1, 0, 0, 0, -1, "")]
        for k in range(260 if name == "all_tags" else 120):
            which = rng.choice([0, 0, 0, 0, 0, 0, 1, 2, 3])
            S2, SF2, M2 = [list(x) for x in S], list(SF), [list(x) for x in M]
            targeted = None
            if k < 12:  # targeted corruptions for the rarely hit Python-runtime error paths
                acc = [j for j, x in enumerate(S) if x[2] == 6]
                targeted = [(rng.randrange(len(S)), 2, 12), (len(S) - 1, 18 + rng.randrange(32), 300),
                            (acc[0] if acc else 0, 5, rng.choice([0, 5, 7])), (rng.randrange(len(S)), 18 + rng.randrange(32), 256)][k % 4]
            if targeted is not None:
                which = 0
                i, c, v = targeted
                S2[i][c] = v
            elif which == 0:
                i = rng.randrange(len(S))
                c = rng.choice([0, 1, 2, 3, 4, 5, 6, 7, 50, 51, 52, 53, 54, 55, 56]) if rng.random() < 0.7 else rng.randrange(57)
                if c == 51 and not (SF[i] & 1) or c == 53 and not (SF[i] & 2):
                    continue  # a value-typed cell has no hi half in the reference
                old = S[i][c]
                if c == 2:
                    v = rng.randrange(0, 14)
                elif c == 5:
                    v = rng.randrange(0, 27)
                else:
                    v = corrupt_value(rng, old)
                if v == old:
                    continue
                S2[i][c] = v
            elif which == 1:  # flip a type flag
                i, c, v = rng.randrange(len(S)), 100 + rng.randrange(2), 0
                SF2[i] ^= 1 << (c - 100)
                if not (SF2[i] >> (c - 100)) & 1:
                    S2[i][51 if c == 100 else 53] = 0
            elif which == 2 and M:
                i, c = rng.randrange(len(M)), rng.randrange(12)
                v = corrupt_value(rng, M[i][c]); M2[i][c] = v
            elif which == 3:  # swap two adjacent rows (ordering)
                i, c, v = rng.randrange(len(S) - 1), 200, 0
                S2[i], S2[i + 1] = S2[i + 1], S2[i]
                SF2[i], SF2[i + 1] = SF2[i + 1], SF2[i]
            else:
                continue
            fr_, ex_ = run(S2, SF2, M2)
            muts.append((which, i, c, v, fr_, ex_))
            tot += 1
            nfail += fr_ >= 0
        out[f"{name}/rows"] = to_matrix(S)
        out[f"{name}/flags"] = np.array(SF, dtype=np.uint8)
        out[f"{name}/mpt"] = to_matrix(M) if M else np.zeros((12, 0, 4), dtype=np.uint64)
        out[f"{name}/mut_kind"] = np.array([m[0] for m in muts], dtype=np.int64)
        out[f"{name}/mut_row"] = np.array([m[1] for m in muts], dtype=np.int64)
        out[f"{name}/mut_col"] = np.array([m[2] for m in muts], dtype=np.int64)
        out[f"{name}/mut_val"] = np.array([limbs(m[3]) for m in muts], dtype=np.uint64)
        out[f"{name}/exp_row"] = np.array([m[4] for m in muts], dtype=np.int64)
        out[f"{name}/exp_exc"] = np.array([m[5] for m in muts])
        print(name, len(S), "rows", len(M), "mpt rows", len(muts), "vectors")
    np.savez_compressed(os.path.join(HERE, "state.npz"), **out)
    print(f"state: {tot} corruptions, {nfail} failing")


# --------------------------------------------------------------------------- synthetic generators
def synth_cases():
    """The numpy generators of zkevm-specs_b200/synth.py (used at scale by tests and bench.py) are run
    through the REFERENCE at small sizes: the reference must accept them."""
    import zkevm_specs.state_circuit as sc
    from zkevm_specs.evm_circuit import (Block, BytecodeTableRow, ExecutionState, RWTableRow, StepState, Tables,
                                         MPTTableRow)
    from zkevm_specs.evm_circuit.main import verify_steps
    from zkevm_specs.util import FQ, Word, WordOrValue

    sys.path.insert(0, os.path.join(HERE, "..", ".."))
    from zkevm_specs_b200 import synth

    def cell(m, c, i):
        return sum(int(m[c, i, k]) << (64 * k) for k in range(4))

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    # EVM trace, 10 groups = 40 steps (all five ops twice)
    w = synth.evm_trace(10, seed=2)
    S, B, R = w["steps"], w["bytecode"], w["rw"]
    steps = []
    for i in range(S.shape[1]):
        s = StepState(ExecutionState(cell(S, 0, i)), rw_counter=cell(S, 1, i), call_id=cell(S, 2, i),
                      is_root=bool(cell(S, 3, i)), is_create=bool(cell(S, 4, i)), code_hash=W(cell(S, 5, i), cell(S, 6, i)),
                      program_counter=cell(S, 7, i), stack_pointer=cell(S, 8, i), gas_left=cell(S, 9, i))
        steps.append(s)
    tables = Tables(block_table=set(Block().table_assignments()), tx_table=set(), withdrawal_table=set(),
                    bytecode_table=set(BytecodeTableRow(W(cell(B, 0, i), cell(B, 1, i)), FQ(cell(B, 2, i)), FQ(cell(B, 3, i)),
                                                        FQ(cell(B, 4, i)), FQ(cell(B, 5, i))) for i in range(B.shape[1])),
                    rw_table=set(RWTableRow(FQ(cell(R, 0, i)), FQ(cell(R, 1, i)), FQ(cell(R, 2, i)), FQ(cell(R, 3, i)),
                                            FQ(cell(R, 4, i)), FQ(0), Word(0), WordOrValue(W(cell(R, 8, i), cell(R, 9, i))))
                                 for i in range(R.shape[1])))
    verify_steps(tables, steps)
    print("synth.evm_trace(10): accepted by the reference's verify_steps,", len(steps) - 1, "steps")

    # state rows, 256 rows incl. Storage / Account groups with the mock MPT table
    w = synth.state_rows(256, seed=3, n_start=16)
    M, F, T = w["rows"], w["flags"], w["mpt"]

    def wov(lo, hi, is_word):
        return WordOrValue(W(lo, hi)) if is_word else WordOrValue(FQ(lo))

    rows = []
    for i in range(M.shape[1]):
        v = [cell(M, c, i) for c in range(57)]
        f = [FQ(x) for x in v]
        rows.append(sc.Row(f[0], f[1], (f[2], f[3], f[4], f[5], W(v[6], v[7])), tuple(f[8:18]), tuple(f[18:50]),
                           wov(v[50], v[51], F[i] & 1), wov(v[52], v[53], (F[i] >> 1) & 1), W(v[54], v[55]), f[56]))
    mpt = set(MPTTableRow(FQ(cell(T, 0, i)), FQ(cell(T, 1, i)), W(cell(T, 2, i), cell(T, 3, i)), W(cell(T, 4, i), cell(T, 5, i)),
                          W(cell(T, 6, i), cell(T, 7, i)), W(cell(T, 8, i), cell(T, 9, i)), W(cell(T, 10, i), cell(T, 11, i)))
              for i in range(T.shape[1]))
    tb = sc.Tables(mpt)
    for idx, row in enumerate(rows):
        sc.check_state_row(row, rows[(idx - 1) % len(rows)], rows[(idx + 1) % len(rows)], tb)
    print("synth.state_rows(256): accepted by the reference's check_state_row,", len(rows), "rows,", len(mpt), "mpt rows")

    # copy events: 2 SHA3-style + 2 CALLDATACOPY-style, 20 bytes each
    from zkevm_specs import copy_circuit as cc
    from zkevm_specs.evm_circuit import CopyCircuitRow, TxTableRow

    w = synth.copy_events(4, 20, seed=4)
    Cm, RWm, TXm = w["copy"], w["rw"], w["tx"]
    r_int = sum(int(w["r"][k]) << (64 * k) for k in range(4))

    class Fake:
        def __init__(self, rows):
            self.rows = rows

        def table(self):
            return self.rows

    crow = []
    for i in range(Cm.shape[1]):
        v = [cell(Cm, c, i) for c in range(20)]
        f = [FQ(x) for x in v]
        crow.append(CopyCircuitRow(f[0], f[1], f[2], WordOrValue(FQ(v[3])), *f[5:]))
    tables = Tables(block_table=set(), withdrawal_table=set(), bytecode_table=set(),
                    tx_table=set(TxTableRow(FQ(cell(TXm, 0, i)), FQ(cell(TXm, 1, i)), FQ(cell(TXm, 2, i)),
                                            WordOrValue(FQ(cell(TXm, 3, i)))) for i in range(TXm.shape[1])),
                    rw_table=set(RWTableRow(FQ(cell(RWm, 0, i)), FQ(cell(RWm, 1, i)), FQ(cell(RWm, 2, i)), FQ(cell(RWm, 3, i)),
                                            FQ(cell(RWm, 4, i)), FQ(0), Word(0), WordOrValue(FQ(cell(RWm, 8, i))))
                                 for i in range(RWm.shape[1])))
    cc.verify_copy_table(Fake(crow), tables, FQ(r_int))
    print("synth.copy_events(4, 20): accepted by the reference's verify_copy_table,", len(crow), "rows")

    # bytecode circuit rows: 2^9 rows, 3 contracts + Header padding
    import zkevm_specs.bytecode_circuit as bcc
    from zkevm_specs.evm_circuit import KeccakTableRow

    w = synth.bytecode_circuit_rows(9, 3, seed=5)
    Bm, Km = w["rows"], w["keccak"]
    r_int = sum(int(w["r"][k]) << (64 * k) for k in range(4))
    brows = []
    for i in range(Bm.shape[1]):
        v = [cell(Bm, c, i) for c in range(12)]
        brows.append(bcc.Row(FQ(v[0]), FQ(v[1]), W(v[2], v[3]), *[FQ(x) for x in v[4:]]))
    push_table = bcc.assign_push_table()
    kt = set(KeccakTableRow(FQ(cell(Km, 0, i)), FQ(cell(Km, 1, i)), FQ(cell(Km, 2, i)), W(cell(Km, 3, i), cell(Km, 4, i)))
             for i in range(Km.shape[1]))
    for idx, row in enumerate(brows):
        bcc.check_bytecode_row(row, brows[(idx + 1) % len(brows)], push_table, kt, FQ(r_int))
    print("synth.bytecode_circuit_rows(9, 3): accepted by the reference's check_bytecode_row,", len(brows), "rows")

    # whole-block trace: 3 transactions over 2 contracts, BeginTx .. STOP, EndTx per transaction, EndBlock last;
    # verify_steps with begin_with_first_step and end_with_last_step (it appends the dummy step itself)
    from zkevm_specs.evm_circuit import BlockTableRow, WithdrawalTableRow

    w = synth.block_trace(3, 2, 2, seed=6)
    S, B, R, RF, TX, TXF, BL, BF = (w[k] for k in ("steps", "bytecode", "rw", "rw_flags", "tx", "tx_flags", "block", "block_flags"))
    steps = []
    for i in range(w["n_steps"]):  # without the dummy step
        s = StepState(ExecutionState(cell(S, 0, i)), rw_counter=cell(S, 1, i), call_id=cell(S, 2, i),
                      is_root=bool(cell(S, 3, i)), is_create=bool(cell(S, 4, i)), code_hash=W(cell(S, 5, i), cell(S, 6, i)),
                      program_counter=cell(S, 7, i), stack_pointer=cell(S, 8, i), gas_left=cell(S, 9, i),
                      memory_word_size=cell(S, 10, i), reversible_write_counter=cell(S, 11, i), log_id=cell(S, 12, i))
        steps.append(s)
    tables = Tables(
        block_table=set(BlockTableRow(FQ(cell(BL, 0, i)), FQ(cell(BL, 1, i)), wov(cell(BL, 2, i), cell(BL, 3, i), BF[i])) for i in range(BL.shape[1])),
        tx_table=set(TxTableRow(FQ(cell(TX, 0, i)), FQ(cell(TX, 1, i)), FQ(cell(TX, 2, i)), wov(cell(TX, 3, i), cell(TX, 4, i), TXF[i])) for i in range(TX.shape[1])),
        withdrawal_table=set(),
        bytecode_table=set(BytecodeTableRow(W(cell(B, 0, i), cell(B, 1, i)), FQ(cell(B, 2, i)), FQ(cell(B, 3, i)),
                                            FQ(cell(B, 4, i)), FQ(cell(B, 5, i))) for i in range(B.shape[1])),
        rw_table=set(RWTableRow(FQ(cell(R, 0, i)), FQ(cell(R, 1, i)), FQ(cell(R, 2, i)), FQ(cell(R, 3, i)), FQ(cell(R, 4, i)), FQ(cell(R, 5, i)),
                                W(cell(R, 6, i), cell(R, 7, i)), wov(cell(R, 8, i), cell(R, 9, i), RF[i] & 1),
                                wov(cell(R, 10, i), cell(R, 11, i), (RF[i] >> 1) & 1), W(cell(R, 12, i), cell(R, 13, i)))
                     for i in range(R.shape[1])))
    verify_steps(tables, steps, begin_with_first_step=True, end_with_last_step=True)
    print("synth.block_trace(3, 2, 2): accepted by the reference's verify_steps(begin_with_first_step, end_with_last_step),",
          len(steps) - 1, "steps,", R.shape[1], "rw rows")


# --------------------------------------------------------------------------- evm2: SHA3 / CALLDATACOPY
def evm2_cases(part="evm2"):
    """SHA3 and CALLDATACOPY steps built like the reference's tests (tests/evm/test_sha3.py:35-141,
    tests/evm/test_calldatacopy.py:42-164) with their copy-table and keccak-table rows, verified by the
    reference's verify_step; corruptions of step cells, rw rows (+ type flags), copy-table and
    keccak-table cells."""
    from zkevm_specs.evm_circuit import (Block, Bytecode, CallContextFieldTag, CopyCircuit, CopyDataTypeTag,
                                         CopyTableRow, ExecutionState, KeccakCircuit, KeccakTableRow, Opcode,
                                         RWDictionary, RWTableRow, BytecodeTableRow, StepState, Tables)
    from zkevm_specs.evm_circuit.instruction import Instruction
    from zkevm_specs.evm_circuit.main import verify_step
    from zkevm_specs.util import FQ, Word, WordOrValue, keccak256, GAS_COST_COPY, GAS_COST_COPY_SHA3

    r = FQ(0x0BADC0FFEE0DDF00D0BADC0FFEE0DDF00D0BADC0FFEE0DDF00D0BADC0FFEE % P)
    rng = random.Random({"evm2": 5, "evm3": 7, "evm4": 9, "evm5": 11, "evm6": 13, "evm7": 15, "evm8": 17, "evm9": 19, "evm10": 21, "evm12": 23, "evm13": 25, "evm14": 27, "evm15": 29, "evm16": 31, "evm17": 33, "evm18": 35, "evm19": 37, "evm20": 39, "evm21": 41, "evm22": 43, "evm23": 45, "evm24": 47, "evm25": 49, "evm26": 51, "evm27": 53, "evm28": 55}[part])

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def wov(lo, hi, is_word):
        return WordOrValue(W(lo, hi)) if is_word else WordOrValue(FQ(lo))

    def stop_case(root, with_stop, caller=(False, False, 232, 1023, 10, 3, 5)):
        """tests/evm/test_stop.py:27-139: STOP in the root call (-> EndTx) and in an internal call
        (restores the caller's context from 12 call-context rows)."""
        bc = Bytecode().push(0, n_bytes=1)
        if with_stop:
            bc = bc.stop()
        h = Word(bc.hash())
        if root:
            rw = RWDictionary(24).call_context_read(1, CallContextFieldTag.IsSuccess, 1)
            steps = [StepState(ExecutionState.STOP, rw_counter=24, call_id=1, is_root=True, is_create=False, code_hash=h,
                               program_counter=2, stack_pointer=1023, gas_left=0, reversible_write_counter=2),
                     StepState(ExecutionState.EndTx, rw_counter=25, call_id=1)]
            return steps, list(bc.table_assignments()), list(rw.rws), [], []
        c_root, c_create, c_pc, c_sp, c_gas, c_mem, c_rev = caller
        cbc = Bytecode().call(0, 0xFF, 0, 0, 0, 0, 0).stop()
        ch = Word(cbc.hash())
        rw = (RWDictionary(69).call_context_read(24, CallContextFieldTag.IsSuccess, 1)
              .call_context_read(24, CallContextFieldTag.CallerId, 1)
              .call_context_read(1, CallContextFieldTag.IsRoot, c_root)
              .call_context_read(1, CallContextFieldTag.IsCreate, c_create)
              .call_context_read(1, CallContextFieldTag.CodeHash, ch)
              .call_context_read(1, CallContextFieldTag.ProgramCounter, c_pc)
              .call_context_read(1, CallContextFieldTag.StackPointer, c_sp)
              .call_context_read(1, CallContextFieldTag.GasLeft, c_gas)
              .call_context_read(1, CallContextFieldTag.MemorySize, c_mem)
              .call_context_read(1, CallContextFieldTag.ReversibleWriteCounter, c_rev)
              .call_context_write(1, CallContextFieldTag.LastCalleeId, 24)
              .call_context_write(1, CallContextFieldTag.LastCalleeReturnDataOffset, 0)
              .call_context_write(1, CallContextFieldTag.LastCalleeReturnDataLength, 0))
        steps = [StepState(ExecutionState.STOP, rw_counter=69, call_id=24, is_root=False, is_create=False, code_hash=h,
                           program_counter=2, stack_pointer=1023, gas_left=400, reversible_write_counter=2),
                 StepState(ExecutionState.STOP, rw_counter=82, call_id=1, is_root=c_root, is_create=c_create, code_hash=ch,
                           program_counter=c_pc, stack_pointer=c_sp, gas_left=c_gas + 400, memory_word_size=c_mem,
                           reversible_write_counter=c_rev + 2)]
        return steps, list(bc.table_assignments()) + list(cbc.table_assignments()), list(rw.rws), [], []

    def memory_case(opcode, offset, value, cur_mem=0):
        """tests/evm/test_memory.py:55-150: MLOAD / MSTORE / MSTORE8 with their 32 (1) memory rows"""
        is_mload, is_mstore8 = opcode == Opcode.MLOAD, opcode == Opcode.MSTORE8
        ow, vw = Word(offset), Word(value)
        bc = (Bytecode().mload(ow).stop() if is_mload else
              Bytecode().mstore8(ow, vw).stop() if is_mstore8 else Bytecode().mstore(ow, vw).stop())
        h = Word(bc.hash())
        rw = (RWDictionary(1).stack_read(1, 1022, ow).stack_write(1, 1022, vw) if is_mload else
              RWDictionary(1).stack_read(1, 1022, ow).stack_read(1, 1023, vw))
        data = value.to_bytes(32, "big")
        if is_mstore8:
            rw.memory_write(1, offset, value & 0xFF)
        else:
            for idx in range(32):
                (rw.memory_read if is_mload else rw.memory_write)(1, offset + idx, data[idx])
        # memory_expansion(offset = curr.memory_word_size, length = address + 1 + 31 * not8), as written
        size = (offset + (1 if is_mstore8 else 32) + cur_mem + 31) // 32
        nxt = max(cur_mem, size)
        gas = Opcode.MLOAD.constant_gas_cost() + (nxt - cur_mem) * 3 + (nxt * nxt // 512 - cur_mem * cur_mem // 512)
        steps = [StepState(ExecutionState.MEMORY, rw_counter=1, call_id=1, is_root=True, is_create=False, code_hash=h,
                           program_counter=33 if is_mload else 66, stack_pointer=1022, memory_word_size=cur_mem, gas_left=gas),
                 StepState(ExecutionState.STOP, rw_counter=4 if is_mstore8 else 35, call_id=1, is_root=True, is_create=False,
                           code_hash=h, program_counter=34 if is_mload else 67, stack_pointer=1022 if is_mload else 1024,
                           memory_word_size=nxt, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], []

    def simple_case(kind, a=0, b=0):
        """tests/evm/test_{msize,gas,iszero,comparator,jump,jumpi}.py: one step + STOP"""
        A, B = Word(a), Word(b)
        if kind == "msize":
            bc, rw = Bytecode().msize().stop(), RWDictionary(9).stack_write(1, 1023, Word(a * 32))
            cur = dict(program_counter=0, stack_pointer=1024, memory_word_size=a, gas_left=2)
            nxt = dict(program_counter=1, stack_pointer=1023, memory_word_size=a, gas_left=0)
            state = ExecutionState.MSIZE
        elif kind == "gas":
            bc, rw = Bytecode().gas().stop(), RWDictionary(9).stack_write(1, 1023, Word(a - 2))
            cur = dict(program_counter=0, stack_pointer=1024, gas_left=a)
            nxt = dict(program_counter=1, stack_pointer=1023, gas_left=a - 2)
            state = ExecutionState.GAS
        elif kind == "iszero":
            bc = Bytecode().push(a, n_bytes=32).iszero().stop()
            rw = RWDictionary(9).stack_read(1, 1023, A).stack_write(1, 1023, Word(int(a == 0)))
            cur = dict(program_counter=33, stack_pointer=1023, gas_left=3)
            nxt = dict(program_counter=34, stack_pointer=1023, gas_left=0)
            state = ExecutionState.ISZERO
        elif kind in ("lt", "gt", "eq"):
            bc = getattr(Bytecode().push(b, n_bytes=32).push(a, n_bytes=32), kind)().stop()
            res = {"lt": a < b, "gt": a > b, "eq": a == b}[kind]
            rw = RWDictionary(9).stack_read(1, 1022, A).stack_read(1, 1023, B).stack_write(1, 1023, Word(int(res)))
            cur = dict(program_counter=66, stack_pointer=1022, gas_left=3)
            nxt = dict(program_counter=67, stack_pointer=1023, gas_left=0)
            state = ExecutionState.CMP
        elif kind == "jump":
            bc = Bytecode().push(a, n_bytes=32).jump()
            while len(bc.code) < a:
                bc = bc.stop()
            bc = bc.jumpdest().stop()
            rw = RWDictionary(9).stack_read(1, 1023, A)
            cur = dict(program_counter=33, stack_pointer=1023, gas_left=8)
            nxt = dict(program_counter=a, stack_pointer=1024, gas_left=0)
            state = ExecutionState.JUMP
        else:  # jumpi: a = dest, b = cond
            bc = Bytecode().push(b, n_bytes=32).push(a, n_bytes=32).jumpi()
            while len(bc.code) < a:
                bc = bc.stop()
            bc = bc.jumpdest().stop()
            rw = RWDictionary(9).stack_read(1, 1022, A).stack_read(1, 1023, B)
            cur = dict(program_counter=66, stack_pointer=1022, gas_left=10)
            nxt = dict(program_counter=67, stack_pointer=1024, gas_left=0)  # see oracle/evm.c:gadget_jumpi
            state = ExecutionState.JUMPI
        h = Word(bc.hash())
        steps = [StepState(state, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h, **cur),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False,
                           code_hash=h, **nxt)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], []

    def cc_push_case(kind, value):
        """tests/evm/test_{caller,callvalue,calldatasize,address,returndatasize,codesize}.py"""
        tag = {"caller": CallContextFieldTag.CallerAddress, "callvalue": CallContextFieldTag.Value,
               "calldatasize": CallContextFieldTag.CallDataLength, "address": CallContextFieldTag.CalleeAddress,
               "returndatasize": CallContextFieldTag.LastCalleeReturnDataLength}.get(kind)
        state = {"caller": ExecutionState.CALLER, "callvalue": ExecutionState.CALLVALUE,
                 "calldatasize": ExecutionState.CALLDATASIZE, "address": ExecutionState.ADDRESS,
                 "returndatasize": ExecutionState.RETURNDATASIZE, "codesize": ExecutionState.CODESIZE}[kind]
        bc = getattr(Bytecode(), kind)().stop()
        if kind == "codesize":
            bc = Bytecode().push(value, n_bytes=32).codesize().stop()
            rw = RWDictionary(9).stack_write(1, 1022, Word(len(bc.code)))
            pc, sp = 33, 1023
        else:
            as_word = kind in ("caller", "callvalue", "address")
            rw = RWDictionary(9).call_context_read(1, tag, Word(value) if as_word else value).stack_write(1, 1023, Word(value))
            pc, sp = 0, 1024
        h = Word(bc.hash())
        steps = [StepState(state, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h, program_counter=pc,
                           stack_pointer=sp, gas_left=2),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False,
                           code_hash=h, program_counter=pc + 1, stack_pointer=sp - 1, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], []

    def bit_case(kind, a, b=0):
        """tests/evm/test_{bitwise,not,byte}.py"""
        A, B = Word(a), Word(b)
        if kind == "not":
            bc = Bytecode().push(a, n_bytes=32).not_().stop()
            rw = RWDictionary(9).stack_read(1, 1023, A).stack_write(1, 1023, Word(a ^ ((1 << 256) - 1)))
            state, pc, sp, nsp, gas = ExecutionState.NOT, 33, 1023, 1023, 3
        else:
            if kind == "byte":
                res = (b >> (8 * (31 - a))) & 0xFF if a < 32 else 0
                state = ExecutionState.BYTE
            else:
                res = {"and": a & b, "or": a | b, "xor": a ^ b}[kind]
                state = ExecutionState.BITWISE
            bc = getattr(Bytecode().push(b, n_bytes=32).push(a, n_bytes=32), kind + ("_" if kind in ("and", "or", "not") else ""))().stop()
            rw = RWDictionary(9).stack_read(1, 1022, A).stack_read(1, 1023, B).stack_write(1, 1023, Word(res))
            pc, sp, nsp, gas = 66, 1022, 1023, 3
        h = Word(bc.hash())
        steps = [StepState(state, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h, program_counter=pc,
                           stack_pointer=sp, gas_left=gas),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False,
                           code_hash=h, program_counter=pc + 1, stack_pointer=nsp, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], []

    def signed_case(kind, a, b):
        """tests/evm/test_{slt_sgt,signextend}.py"""
        A, B = Word(a), Word(b)
        M = (1 << 256)

        def sgn(x):
            return x - M if x >> 255 else x

        if kind == "signextend":  # a = index, b = value
            if a < 31:
                bits = 8 * (a + 1)
                low = b & ((1 << bits) - 1)
                res = (low | (M - (1 << bits))) % M if (low >> (bits - 1)) & 1 else low
            else:
                res = b
            state = ExecutionState.SIGNEXTEND
        else:
            res = int(sgn(a) < sgn(b)) if kind == "slt" else int(sgn(a) > sgn(b))
            state = ExecutionState.SCMP
        bc = getattr(Bytecode().push(b, n_bytes=32).push(a, n_bytes=32), kind)().stop()
        rw = RWDictionary(9).stack_read(1, 1022, A).stack_read(1, 1023, B).stack_write(1, 1023, Word(res))
        h = Word(bc.hash())
        steps = [StepState(state, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h, program_counter=66,
                           stack_pointer=1022, gas_left=5 if kind == "signextend" else 3),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False,
                           code_hash=h, program_counter=67, stack_pointer=1023, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], []

    def ctx_case(kind, value):
        """tests/evm/test_{block_ctx,origin,gasprice}.py: a block-table / tx-table word pushed on the stack"""
        from zkevm_specs.evm_circuit import BlockContextFieldTag, BlockTableRow, TxContextFieldTag, TxTableRow
        txs, blocks = [], []
        if kind in ("origin", "gasprice"):
            bc = getattr(Bytecode(), kind)().stop()
            tag = TxContextFieldTag.CallerAddress if kind == "origin" else TxContextFieldTag.GasPrice
            rw = RWDictionary(9).call_context_read(1, CallContextFieldTag.TxId, 3).stack_write(1, 1023, Word(value))
            txs = [TxTableRow(FQ(3), FQ(tag), FQ(0), WordOrValue(Word(value))),
                   TxTableRow(FQ(3), FQ(TxContextFieldTag.Nonce), FQ(0), WordOrValue(FQ(7))),
                   TxTableRow(FQ(4), FQ(tag), FQ(0), WordOrValue(Word(value + 1)))]
            state = ExecutionState.ORIGIN if kind == "origin" else ExecutionState.GASPRICE
        else:
            bc = getattr(Bytecode(), kind)().stop()
            tag = {"coinbase": BlockContextFieldTag.Coinbase, "timestamp": BlockContextFieldTag.Timestamp,
                   "number": BlockContextFieldTag.Number, "gaslimit": BlockContextFieldTag.GasLimit,
                   "prevrandao": BlockContextFieldTag.PrevRandao, "basefee": BlockContextFieldTag.BaseFee,
                   "chainid": BlockContextFieldTag.ChainId}[kind]
            rw = RWDictionary(9).stack_write(1, 1023, Word(value))
            blocks = [BlockTableRow(FQ(tag), FQ(0), WordOrValue(Word(value))),
                      BlockTableRow(FQ(BlockContextFieldTag.HistoryHash), FQ(5), WordOrValue(Word(99)))]
            state = ExecutionState.BlockCtx
        h = Word(bc.hash())
        steps = [StepState(state, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h, program_counter=0,
                           stack_pointer=1024, gas_left=2),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False,
                           code_hash=h, program_counter=1, stack_pointer=1023, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], [], txs, blocks

    def shift_case(kind, shift, value):
        """tests/evm/test_shl_shr.py"""
        M = 1 << 256
        res = ((value << shift) % M if shift < 256 else 0) if kind == "shl" else (value >> shift if shift < 256 else 0)
        bc = getattr(Bytecode().push(value, n_bytes=32).push(shift, n_bytes=32), kind)().stop()
        rw = RWDictionary(9).stack_read(1, 1022, Word(shift)).stack_read(1, 1023, Word(value)).stack_write(1, 1023, Word(res))
        h = Word(bc.hash())
        steps = [StepState(ExecutionState.SHL_SHR, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h,
                           program_counter=66, stack_pointer=1022, gas_left=3),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False,
                           code_hash=h, program_counter=67, stack_pointer=1023, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], []

    def arith_case(kind, a, b, n=0, res=None):
        """tests/evm/test_{addmod,mulmod,sdiv_smod,sar}.py (res: a pushed result other than the EVM's, for the cases the
        reference leaves unconstrained)"""
        M = 1 << 256

        def sgn(x):
            return x - M if x >> 255 else x

        if kind in ("addmod", "mulmod"):
            r = 0 if n == 0 else ((a + b) % n if kind == "addmod" else (a * b) % n)
            bc = getattr(Bytecode().push32(n).push32(b).push32(a), kind)().stop()
            rw = (RWDictionary(9).stack_read(1, 1021, Word(a)).stack_read(1, 1022, Word(b)).stack_read(1, 1023, Word(n))
                  .stack_write(1, 1023, Word(r if res is None else res)))
            state, pc, sp, nsp, gas = (ExecutionState.ADDMOD if kind == "addmod" else ExecutionState.MULMOD), 99, 1021, 1023, 8
        else:
            if kind == "sar":  # a = shift, b = value
                r = (sgn(b) >> a) % M if a < 256 else (M - 1 if b >> 255 else 0)
                state, gas = ExecutionState.SAR, 3
            else:
                sa, sb = sgn(a), sgn(b)
                if b == 0:
                    r = 0
                elif kind == "sdiv":
                    q = abs(sa) // abs(sb)
                    r = (q if (sa < 0) == (sb < 0) else -q) % M
                else:
                    m = abs(sa) % abs(sb)
                    r = (-m if sa < 0 else m) % M
                state, gas = ExecutionState.SDIV_SMOD, 5
            bc = getattr(Bytecode().push32(b).push32(a), kind)().stop()
            rw = RWDictionary(9).stack_read(1, 1022, Word(a)).stack_read(1, 1023, Word(b)).stack_write(1, 1023, Word(r if res is None else res))
            pc, sp, nsp = 66, 1022, 1023
        h = Word(bc.hash())
        steps = [StepState(state, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h, program_counter=pc,
                           stack_pointer=sp, gas_left=gas),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False,
                           code_hash=h, program_counter=pc + 1, stack_pointer=nsp, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], []

    def storage_case(kind, value=2, value_prev=0, original=0, warm=False, persistent=True, rev0=0, refund_prev=15000):
        """tests/evm/test_sload.py, test_sstore.py"""
        from zkevm_specs.util import COLD_SLOAD_COST, SLOAD_GAS, SSTORE_CLEARS_SCHEDULE, SSTORE_RESET_GAS, SSTORE_SET_GAS, WARM_STORAGE_READ_COST
        callee = 0xCAFE0000000000000000000000000000BEEF1234
        key = Word(int.from_bytes(bytes(range(32, 0, -1)), "big"))
        rev_end = 0 if persistent else 40
        if kind == "sload":
            bc = Bytecode().push32(key.int_value()).sload().stop()
            rw = (RWDictionary(9).call_context_read(1, CallContextFieldTag.TxId, 3)
                  .call_context_read(1, CallContextFieldTag.RwCounterEndOfReversion, rev_end)
                  .call_context_read(1, CallContextFieldTag.IsPersistent, persistent)
                  .call_context_read(1, CallContextFieldTag.CalleeAddress, Word(callee))
                  .stack_read(1, 1023, key).account_storage_read(callee, key, Word(value), 3, Word(original)).stack_write(1, 1023, Word(value))
                  .tx_access_list_account_storage_write(3, callee, key, 1, 1 if warm else 0,
                                                        rw_counter_of_reversion=None if persistent else rev_end - rev0))
            gas, pc, sp, nsp, d_rev, state = (WARM_STORAGE_READ_COST if warm else COLD_SLOAD_COST), 33, 1023, 1023, 1, ExecutionState.SLOAD
        else:
            bc = Bytecode().push32(value).push32(key.int_value()).sstore().stop()
            if value_prev == value:
                gas = SLOAD_GAS
            elif original == value_prev:
                gas = SSTORE_SET_GAS if original == 0 else SSTORE_RESET_GAS
            else:
                gas = SLOAD_GAS
            if not warm:
                gas += COLD_SLOAD_COST
            refund = refund_prev
            if value_prev != value:
                if original == value_prev:
                    if original != 0 and value == 0:
                        refund += SSTORE_CLEARS_SCHEDULE
                else:
                    if original != 0:
                        if value_prev == 0:
                            refund -= SSTORE_CLEARS_SCHEDULE
                        if value == 0:
                            refund += SSTORE_CLEARS_SCHEDULE
                    if original == value:
                        refund += (SSTORE_SET_GAS if original == 0 else SSTORE_RESET_GAS) - SLOAD_GAS
            rw = (RWDictionary(9).call_context_read(1, CallContextFieldTag.TxId, 3).call_context_read(1, CallContextFieldTag.IsStatic, 0)
                  .call_context_read(1, CallContextFieldTag.RwCounterEndOfReversion, rev_end)
                  .call_context_read(1, CallContextFieldTag.IsPersistent, persistent)
                  .call_context_read(1, CallContextFieldTag.CalleeAddress, Word(callee))
                  .stack_read(1, 1022, key).stack_read(1, 1023, Word(value))
                  .account_storage_write(callee, key, Word(value), Word(value_prev), 3, Word(original),
                                         rw_counter_of_reversion=None if persistent else rev_end - rev0)
                  .tx_access_list_account_storage_write(3, callee, key, True, warm, rw_counter_of_reversion=None if persistent else rev_end - rev0 - 1)
                  .tx_refund_write(3, refund, refund_prev, rw_counter_of_reversion=None if persistent else rev_end - rev0 - 2))
            pc, sp, nsp, d_rev, state = 66, 1022, 1024, 3, ExecutionState.SSTORE
        h = Word(bc.hash())
        steps = [StepState(state, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h, program_counter=pc,
                           stack_pointer=sp, gas_left=gas, reversible_write_counter=rev0),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False, code_hash=h,
                           program_counter=pc + 1, stack_pointer=nsp, gas_left=0, reversible_write_counter=rev0 + d_rev)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], []

    def calldataload_case(call_data, cd_len, offset, is_root, cd_off=0):
        """tests/evm/test_calldataload.py: 32 bytes of the tx call data (tx table) or of the caller's memory"""
        from zkevm_specs.evm_circuit import Transaction
        tx = Transaction(id=1, call_data=bytes(call_data) if is_root else bytes())
        bc = Bytecode().push32(offset).calldataload().stop()
        h = Word(bc.hash())
        call_id = 1 if is_root else 2
        word = bytearray(32)
        rw = RWDictionary(9).stack_read(call_id, 1023, Word(offset))
        if is_root:
            rw.call_context_read(call_id, CallContextFieldTag.TxId, 1).call_context_read(call_id, CallContextFieldTag.CallDataLength, cd_len)
            for k in range(32):
                if offset + k < cd_len:
                    word[k] = call_data[offset + k]
        else:
            (rw.call_context_read(call_id, CallContextFieldTag.CallerId, 1).call_context_read(call_id, CallContextFieldTag.CallDataLength, cd_len)
             .call_context_read(call_id, CallContextFieldTag.CallDataOffset, cd_off))
            for k in range(32):
                if offset + k < cd_len:
                    word[k] = call_data[cd_off + offset + k]
                    rw.memory_read(1, cd_off + offset + k, word[k])
        rw.stack_write(call_id, 1023, Word(bytes(word)))
        steps = [StepState(ExecutionState.CALLDATALOAD, rw_counter=9, call_id=call_id, is_root=is_root, is_create=False, code_hash=h,
                           program_counter=33, stack_pointer=1023, gas_left=3),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=call_id, is_root=is_root, is_create=False, code_hash=h,
                           program_counter=34, stack_pointer=1023, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], [], list(tx.table_assignments()), []

    def log_case(topics, mstart, msize, persistent, cur_mem=0, log_id=0):
        """tests/evm/test_logs.py: LOG0..LOG4 (tx-log rows for the address and the topics, the data through the copy table)"""
        from zkevm_specs.evm_circuit import TxLogFieldTag
        from zkevm_specs.util.param import GAS_COST_LOG, GAS_COST_LOGDATA
        callee = 0xCAFE0000000000000000000000000000BEEF1234
        bc = Bytecode()
        for t in reversed(topics):
            bc.push32(t)
        bc.push32(msize).push32(mstart)
        getattr(bc, "log%d" % len(topics))()
        bc.stop()
        h = Word(bc.hash())
        sp = 1024 - 2 - len(topics)
        nxt, exp = mem_exp(cur_mem, mstart + msize)
        if msize == 0:  # memory_expansion_dynamic_length still counts the offset (instruction.py:1164-1166)
            nxt = max(cur_mem, mws(mstart)); exp = (nxt - cur_mem) * 3 + (nxt * nxt // 512 - cur_mem * cur_mem // 512)
        gas = GAS_COST_LOG * (1 + len(topics)) + GAS_COST_LOGDATA * msize + exp
        rw = (RWDictionary(9).stack_read(1, sp, Word(mstart)).stack_read(1, sp + 1, Word(msize))
              .call_context_read(1, CallContextFieldTag.TxId, 3).call_context_read(1, CallContextFieldTag.IsStatic, 0)
              .call_context_read(1, CallContextFieldTag.CalleeAddress, Word(callee))
              .call_context_read(1, CallContextFieldTag.IsPersistent, persistent))
        if persistent:
            rw.tx_log_write(3, log_id + 1, TxLogFieldTag.Address, 0, Word(callee))
        for k_, t in enumerate(topics):
            rw.stack_read(1, sp + 2 + k_, Word(t))
            if persistent:
                rw.tx_log_write(3, log_id + 1, TxLogFieldTag.Topic, k_, Word(t))
        cc = CopyCircuit()
        if persistent and msize:
            data = {mstart + k_: rng.randrange(256) for k_ in range(msize)}
            cc.copy(r, rw, 1, CopyDataTypeTag.Memory, 3, CopyDataTypeTag.TxLog, mstart, mstart + msize, 0, msize, data, log_id=log_id + 1)
        pc = 33 * (2 + len(topics))
        steps = [StepState(ExecutionState.LOG, rw_counter=9, call_id=1, is_root=False, is_create=False, code_hash=h, program_counter=pc,
                           stack_pointer=sp, memory_word_size=cur_mem, gas_left=gas, log_id=log_id),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=False, is_create=False, code_hash=h,
                           program_counter=pc + 1, stack_pointer=1024, memory_word_size=nxt, gas_left=0, log_id=log_id + int(persistent))]
        t = Tables(block_table=set(), tx_table=set(), withdrawal_table=set(), bytecode_table=set(bc.table_assignments()),
                   rw_table=set(rw.rws), copy_circuit=cc.rows)
        return steps, list(bc.table_assignments()), list(rw.rws), list(t.copy_table), []

    def ewp_case(op, root, value=100):
        """tests/evm/test_error_write_protection.py: a state-modifying opcode in a static call"""
        bc = Bytecode()
        if op == "call":
            bc = bc.call(0x2000, 0xFF, value, 0, 0, 0, 0)
            state_pc, sp = 231, 1017
        elif op == "sstore":
            bc = bc.push32(5).push32(7).sstore(); state_pc, sp = 66, 1022
        else:
            bc = bc.push32(5).push32(7).log0(); state_pc, sp = 66, 1022
        bc.stop()
        h = Word(bc.hash())
        call_id, rev = (1 if root else 2), 2
        rw = RWDictionary(24 if root else 69)
        rwc0 = rw.rw_counter
        rw.call_context_read(call_id, CallContextFieldTag.IsStatic, 1)
        if op == "call":
            rw.stack_read(call_id, sp + 2, Word(value))
        rw.call_context_read(call_id, CallContextFieldTag.IsSuccess, 0)
        cur = StepState(ExecutionState.ErrorWriteProtection, rw_counter=rwc0, call_id=call_id, is_root=root, is_create=False, code_hash=h,
                        program_counter=state_pc, stack_pointer=sp, gas_left=100, reversible_write_counter=rev)
        if root:
            return [cur, StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter + rev, call_id=1, gas_left=0)], list(bc.table_assignments()), list(rw.rws), [], []
        cbc = Bytecode().call(0, 0xFF, 0, 0, 0, 0, 0).stop()
        ch = Word(cbc.hash())
        ctx = (True, False, 232, 1023, 10, 3, 5)
        caller_ctx_rws(rw, 1, ch, ctx, 2)
        nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter + rev, call_id=1, is_root=ctx[0], is_create=ctx[1], code_hash=ch,
                        program_counter=ctx[2], stack_pointer=ctx[3], gas_left=ctx[4], memory_word_size=ctx[5],
                        reversible_write_counter=ctx[6])
        return [cur, nxt], list(bc.table_assignments()) + list(cbc.table_assignments()), list(rw.rws), [], []

    def eopc_case(address, cd_len, gas_left, root=False):
        """ErrorOutOfGasPrecompile (execution/precompiles/error_oog_precompile.py; the reference has no test of its own for
        it): a precompile call's context (callee address 1..9, call-data length) with less gas than the precompile costs"""
        bc = Bytecode().stop()
        h = Word(bc.hash())
        call_id, rev = (1 if root else 2), 2
        rw = RWDictionary(24 if root else 69)
        rwc0 = rw.rw_counter
        rw.call_context_read(call_id, CallContextFieldTag.CalleeAddress, Word(address))
        rw.call_context_read(call_id, CallContextFieldTag.CallDataLength, cd_len)
        rw.call_context_read(call_id, CallContextFieldTag.IsSuccess, 0)
        cur = StepState(ExecutionState.ErrorOutOfGasPrecompile, rw_counter=rwc0, call_id=call_id, is_root=root, is_create=False, code_hash=h,
                        program_counter=0, stack_pointer=1024, gas_left=gas_left, reversible_write_counter=rev)
        if root:
            return [cur, StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter + rev, call_id=1, gas_left=0)], list(bc.table_assignments()), list(rw.rws), [], []
        cbc = Bytecode().call(0, address, 0, 0, cd_len & 0xFFFF, 0, 0).stop()
        ch = Word(cbc.hash())
        ctx = (True, False, 232, 1023, 10, 3, 5)
        caller_ctx_rws(rw, 1, ch, ctx, 2)
        nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter + rev, call_id=1, is_root=ctx[0], is_create=ctx[1], code_hash=ch,
                        program_counter=ctx[2], stack_pointer=ctx[3], gas_left=ctx[4], memory_word_size=ctx[5],
                        reversible_write_counter=ctx[6])
        return [cur, nxt], list(bc.table_assignments()) + list(cbc.table_assignments()), list(rw.rws), [], []

    def eguo_mem_case(op, offset, root=False):
        """ErrorGasUintOverflow on MLOAD / MSTORE / MSTORE8 (error_gas_uint_overflow.py; the reference's test returns early for
        these three): the memory offset alone overflows"""
        from zkevm_specs.evm_circuit import Transaction
        bc = getattr(Bytecode(), op)()
        h = Word(bc.hash())
        call_id = 1 if root else 2
        tx = Transaction(id=1, call_data=bytes([0x7f]))
        rw = RWDictionary(25)
        rw.call_context_read(call_id, CallContextFieldTag.CallDataLength, 1)
        rw.call_context_read(call_id, CallContextFieldTag.TxId, 1)
        rw.call_context_read(call_id, CallContextFieldTag.IsRoot, FQ(root))
        if op == "mload":
            rw.stack_read(call_id, 1023, Word(offset)); sp = 1023
        else:
            rw.stack_read(call_id, 1022, Word(offset)).stack_read(call_id, 1023, Word(7)); sp = 1022
        rw.call_context_read(call_id, CallContextFieldTag.IsSuccess, 0)
        cur = StepState(ExecutionState.ErrorGasUintOverflow, rw_counter=25, call_id=call_id, is_root=root, is_create=False, code_hash=h,
                        program_counter=0, stack_pointer=sp, gas_left=0, reversible_write_counter=0)
        if root:
            nxt = StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter, call_id=1, gas_left=0)
        else:
            ctx = (False, False, 232, 1023, 100, 100, 0)
            caller_ctx_rws(rw, 1, h, ctx, 2)
            nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=ctx[0], is_create=ctx[1], code_hash=h,
                            program_counter=ctx[2], stack_pointer=ctx[3], gas_left=ctx[4], memory_word_size=ctx[5],
                            reversible_write_counter=ctx[6])
        return [cur, nxt], list(bc.table_assignments()), list(rw.rws), [], [], list(tx.table_assignments())

    def blockhash_case(current, number, res=None):
        """tests/evm/test_blockhash.py: the hash of one of the 256 previous blocks, else zero"""
        from zkevm_specs.evm_circuit import BlockContextFieldTag, BlockTableRow
        hashes = {n_: rng.randrange(1, 1 << 256) for n_ in range(max(0, current - 255), current)}
        want = hashes.get(number, 0) if res is None else res
        bc = Bytecode().push32(number).blockhash().stop()
        h = Word(bc.hash())
        rw = RWDictionary(9).stack_read(1, 1023, Word(number)).stack_write(1, 1023, Word(want))
        blocks = [BlockTableRow(FQ(BlockContextFieldTag.Number), FQ(0), WordOrValue(FQ(current))),
                  BlockTableRow(FQ(BlockContextFieldTag.Coinbase), FQ(0), WordOrValue(Word(0x77)))]
        blocks += [BlockTableRow(FQ(BlockContextFieldTag.HistoryHash), FQ(n_), WordOrValue(Word(v_))) for n_, v_ in list(hashes.items())[-6:] + ([(number, hashes[number])] if number in hashes else [])]
        steps = [StepState(ExecutionState.BLOCKHASH, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h, program_counter=33,
                           stack_pointer=1023, gas_left=20),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False, code_hash=h,
                           program_counter=34, stack_pointer=1023, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], [], [], list(set(blocks))

    def exp_case(base, exponent, res=None):
        """tests/evm/test_exp.py: the exponentiation read from the exp table (first and last step rows of the exp circuit)"""
        from zkevm_specs.evm_circuit import ExpCircuit
        from zkevm_specs.util import GAS_COST_EXP_PER_BYTE, byte_size
        want = pow(base, exponent, 1 << 256) if res is None else res
        bc = Bytecode().push32(exponent).push32(base).exp().stop()
        h = Word(bc.hash())
        rw = RWDictionary(9).stack_read(1, 1022, Word(base)).stack_read(1, 1023, Word(exponent)).stack_write(1, 1023, Word(want))
        ec = ExpCircuit(max_exp_steps=4).add_event(base, exponent, rw.rw_counter)
        if rng.random() < 0.5:
            ec.add_event(3, 5, 77)
        t = Tables(block_table=set(), tx_table=set(), withdrawal_table=set(), bytecode_table=set(bc.table_assignments()),
                   rw_table=set(rw.rws), exp_circuit=ec.rows)
        gas = Opcode.EXP.constant_gas_cost() + byte_size(exponent) * GAS_COST_EXP_PER_BYTE
        steps = [StepState(ExecutionState.EXP, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h, program_counter=66,
                           stack_pointer=1022, gas_left=gas),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False, code_hash=h,
                           program_counter=67, stack_pointer=1023, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], [], [], [], list(t.exp_table)

    def code_store_case(kind, root, size=200, gas_left=39999, first_byte=0xEF):
        """tests/evm/test_error_code_store.py, test_error_invalid_creation_code.py: RETURN from a CREATE / CREATE2 that cannot
        store its code (too long / not enough gas for the deposit / first byte 0xEF)"""
        bc = Bytecode().push32(size).push32(32).return_()
        h = Word(bc.hash())
        call_id, rev = (1 if root else 2), 2
        rw = RWDictionary(24 if root else 69)
        rwc0 = rw.rw_counter
        if kind == "invalid":
            state = ExecutionState.ErrorInvalidCreationCode
            rw.stack_read(call_id, 1022, Word(32)).memory_read(call_id, 32, first_byte)
        else:
            state = ExecutionState.ErrorMaxCodeSizeExceeded if kind == "max" else ExecutionState.ErrorOutOfGasCodeStore
            rw.stack_read(call_id, 1023, Word(size)).call_context_read(call_id, CallContextFieldTag.IsStatic, 0)
        rw.call_context_read(call_id, CallContextFieldTag.IsSuccess, 0)
        cur = StepState(state, rw_counter=rwc0, call_id=call_id, is_root=root, is_create=True, code_hash=h, program_counter=66,
                        stack_pointer=1022, gas_left=gas_left, reversible_write_counter=rev)
        if root:
            return [cur, StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter + rev, call_id=1, gas_left=0)], list(bc.table_assignments()), list(rw.rws), [], []
        cbc = Bytecode().call(0, 0xFF, 0, 0, 0, 0, 0).stop()
        ch = Word(cbc.hash())
        ctx = (True, False, 232, 1023, 10, 3, 5)
        caller_ctx_rws(rw, 1, ch, ctx, 2)
        nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter + rev, call_id=1, is_root=ctx[0], is_create=ctx[1], code_hash=ch,
                        program_counter=ctx[2], stack_pointer=ctx[3], gas_left=ctx[4], memory_word_size=ctx[5],
                        reversible_write_counter=ctx[6])
        return [cur, nxt], list(bc.table_assignments()) + list(cbc.table_assignments()), list(rw.rws), [], []

    def return_case(kind, is_return, offset, length, caller_len=10, cur_mem=2, gas=1000000):
        """tests/evm/test_return_revert.py: RETURN / REVERT in the root call, in an internal call (return data copied to the
        caller's memory, caller context restored) and at the end of a CREATE (memory -> deployed bytecode)"""
        from zkevm_specs.evm_circuit import AccountFieldTag
        from zkevm_specs.util.hash import EMPTY_CODE_HASH
        from zkevm_specs.util.param import GAS_COST_CODE_DEPOSIT
        bc = Bytecode().push32(0x2222222222222222222222222222222222222222222222222222222222222222).push1(4).mstore().push1(length).push1(offset)
        bc = bc.return_() if is_return else bc.revert()
        h = Word(bc.hash())
        pc = 40
        root = kind in ("root", "create_root")
        create = kind.startswith("create")
        callee = 1 if root else 2
        if create:
            length = len(bc.code)  # the deployed code is the running (init) code itself, as in the reference's test
        rw = RWDictionary(24).call_context_read(callee, CallContextFieldTag.IsSuccess, int(is_return))
        rw.stack_read(callee, 1022, Word(offset)).stack_read(callee, 1023, Word(length))
        cc = CopyCircuit()
        gas_left = gas
        if create:
            A = 0xFE
            rw.call_context_read(callee, CallContextFieldTag.CalleeAddress, Word(A)).account_write(A, AccountFieldTag.CodeHash, h, Word(EMPTY_CODE_HASH))
            src = {offset + k_: (bc.code[k_], bc.is_code[k_]) for k_ in range(length)}
            cc.copy(r, rw, callee, CopyDataTypeTag.Memory, h, CopyDataTypeTag.Bytecode, offset, offset + length, 0, length, src)
            gas_left -= length * GAS_COST_CODE_DEPOSIT
        elif not root:
            rw.call_context_read(callee, CallContextFieldTag.ReturnDataOffset, 0x40).call_context_read(callee, CallContextFieldTag.ReturnDataLength, caller_len)
            n_copy = min(length, caller_len)
            mem = [0] * 4 + [0x22] * 32 + [0] * 200
            src = {k_: mem[k_] for k_ in range(offset, offset + n_copy)}
            cc.copy(r, rw, callee, CopyDataTypeTag.Memory, 1, CopyDataTypeTag.Memory, offset, offset + length, 0x40, n_copy, src)
        rev = 2
        cur = StepState(ExecutionState.RETURN, rw_counter=24, call_id=callee, is_root=root, is_create=create, code_hash=h, program_counter=pc,
                        stack_pointer=1022, gas_left=gas, memory_word_size=cur_mem, reversible_write_counter=rev)
        bcs = list(bc.table_assignments())
        if root:
            rw.call_context_read(callee, CallContextFieldTag.IsPersistent, int(is_return))
            # (the CREATE branch's two lookups are not counted in rwc_delta, return_revert.py:37-45: the next step starts 2 early)
            nxt = StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter - (2 if create else 0), call_id=callee, gas_left=gas_left)
        else:
            nxt_mem, exp = mem_exp(cur_mem, offset + length)
            if length == 0:
                nxt_mem = max(cur_mem, mws(offset)); exp = (nxt_mem - cur_mem) * 3 + (nxt_mem * nxt_mem // 512 - cur_mem * cur_mem // 512)
            cbc = Bytecode().call(0, 0xFF, 0, 0, 0, 0, 0).stop()
            ch = Word(cbc.hash())
            ctx = (True, False, 232, 1023, 77, 3, 5)
            c_root, c_create, c_pc, c_sp, c_gas, c_mem, c_rev = ctx
            (rw.call_context_read(callee, CallContextFieldTag.CallerId, 1).call_context_read(1, CallContextFieldTag.IsRoot, c_root)
             .call_context_read(1, CallContextFieldTag.IsCreate, c_create).call_context_read(1, CallContextFieldTag.CodeHash, ch)
             .call_context_read(1, CallContextFieldTag.ProgramCounter, c_pc).call_context_read(1, CallContextFieldTag.StackPointer, c_sp)
             .call_context_read(1, CallContextFieldTag.GasLeft, c_gas).call_context_read(1, CallContextFieldTag.MemorySize, c_mem)
             .call_context_read(1, CallContextFieldTag.ReversibleWriteCounter, c_rev)
             .call_context_write(1, CallContextFieldTag.LastCalleeId, callee)
             .call_context_write(1, CallContextFieldTag.LastCalleeReturnDataOffset, offset)
             .call_context_write(1, CallContextFieldTag.LastCalleeReturnDataLength, length))
            nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter - (2 if create else 0), call_id=1, is_root=c_root, is_create=c_create, code_hash=ch,
                            program_counter=c_pc, stack_pointer=c_sp, gas_left=c_gas + gas_left - exp, memory_word_size=c_mem,
                            reversible_write_counter=c_rev + rev)
            bcs += list(cbc.table_assignments())
        t = Tables(block_table=set(), tx_table=set(), withdrawal_table=set(), bytecode_table=set(bcs), rw_table=set(rw.rws), copy_circuit=cc.rows)
        return [cur, nxt], bcs, list(rw.rws), list(t.copy_table), []

    def oog_call_case(op, root, is_warm, gas_left, value=0, cd=(64, 320), rd=(0, 32), cur_mem=0):
        """tests/evm/test_error_oog_call.py: CALL / CALLCODE / DELEGATECALL / STATICCALL without the gas for the call itself"""
        from zkevm_specs.evm_circuit import AccountFieldTag
        callee_code = Bytecode().stop()
        A = 0xFF
        has_value = op in ("call", "callcode")
        bc = Bytecode()
        if has_value:
            bc = getattr(bc, op)(100, A, value, cd[0], cd[1], rd[0], rd[1]).stop()
        else:
            bc = getattr(bc, op)(100, A, cd[0], cd[1], rd[0], rd[1]).stop()
        h = Word(bc.hash())
        call_id, rev = (1 if root else 2), 2
        sp = 1018 - int(has_value)
        rw = RWDictionary(24 if root else 69)
        rwc0 = rw.rw_counter
        rw.call_context_read(call_id, CallContextFieldTag.TxId, 1).stack_read(call_id, sp, Word(100)).stack_read(call_id, sp + 1, Word(A))
        if has_value:
            rw.stack_read(call_id, 1019, Word(value))
        (rw.stack_read(call_id, 1020, Word(cd[0])).stack_read(call_id, 1021, Word(cd[1])).stack_read(call_id, 1022, Word(rd[0]))
         .stack_read(call_id, 1023, Word(rd[1])).stack_write(call_id, 1023, Word(0))
         .account_read(A, AccountFieldTag.CodeHash, Word(callee_code.hash())).tx_access_list_account_read(1, A, is_warm)
         .call_context_read(call_id, CallContextFieldTag.IsSuccess, 0))
        cur = StepState(ExecutionState.ErrorOutOfGasCall, rw_counter=rwc0, call_id=call_id, is_root=root, is_create=False, code_hash=h,
                        program_counter=231 if has_value else 198, stack_pointer=sp, gas_left=gas_left, memory_word_size=cur_mem,
                        reversible_write_counter=rev)
        bcs = list(bc.table_assignments()) + list(callee_code.table_assignments())
        if root:
            return [cur, StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter + rev, call_id=1, gas_left=0)], bcs, list(rw.rws), [], []
        cbc = Bytecode().call(0, 0xFE, 0, 0, 0, 0, 0).stop()
        ch = Word(cbc.hash())
        ctx = (True, False, 232, 1023, 10, 3, 5)
        caller_ctx_rws(rw, 1, ch, ctx, 2)
        nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter + rev, call_id=1, is_root=ctx[0], is_create=ctx[1], code_hash=ch,
                        program_counter=ctx[2], stack_pointer=ctx[3], gas_left=ctx[4], memory_word_size=ctx[5],
                        reversible_write_counter=ctx[6])
        return [cur, nxt], bcs + list(cbc.table_assignments()), list(rw.rws), [], []

    def callop_case(idx):
        """tests/evm/test_callop.py: case `idx` of the reference test's own TESTING_DATA, built with its template
        (callop_test_template / expected are imported from the reference's test module; nothing of it is copied here)"""
        import importlib
        tdir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(sys.modules["zkevm_specs"].__file__))), "..", "tests", "evm")
        tdir = os.path.normpath(tdir)
        for d_ in (tdir, os.path.dirname(tdir)):  # tests/evm and tests/ (common.py)
            if d_ not in sys.path:
                sys.path.insert(0, d_)
        tc = importlib.import_module("test_callop")
        opcode, callee, caller_ctx, stack, is_warm, depth, exp = tc.TESTING_DATA[idx]
        (_, caller_bc, callee_bc, call_id, next_pc, sp, rw, precheck_ok, empty_hash) = tc.callop_test_template(
            opcode, callee, caller_ctx, stack, is_warm, depth, False, exp)
        h = Word(caller_bc.hash())
        callee_h = Word(callee_bc.hash() if not callee.is_empty() else 0)
        cur = StepState(ExecutionState.CALL_OP, rw_counter=call_id, call_id=1, is_root=True, is_create=False, code_hash=h,
                        program_counter=next_pc - 1, stack_pointer=sp, gas_left=caller_ctx.gas_left, memory_word_size=caller_ctx.memory_word_size,
                        reversible_write_counter=caller_ctx.reversible_write_counter)
        if empty_hash or precheck_ok is False:
            nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False, code_hash=h,
                            program_counter=next_pc, stack_pointer=1023, gas_left=exp.caller_gas_left, memory_word_size=exp.next_memory_size,
                            reversible_write_counter=caller_ctx.reversible_write_counter + 3)
        else:
            nxt = StepState(ExecutionState.STOP if callee.code == tc.STOP_BYTECODE else ExecutionState.PUSH, rw_counter=rw.rw_counter, call_id=call_id,
                            is_root=False, is_create=False, code_hash=callee_h, program_counter=0, stack_pointer=1024,
                            gas_left=exp.callee_gas_left, reversible_write_counter=2)
        return [cur, nxt], list(caller_bc.table_assignments()) + list(callee_bc.table_assignments()), list(rw.rws), [], []

    def recorded_case(module, fn, args):
        """Run one of the reference's OWN test functions (tests/evm/<module>.py) with its verify_steps / verify_copy_table
        replaced by a recorder: yields the tables and the steps it would have verified.  A step's aux_data (a Word: the
        init code's hash of CREATE / CREATE2; an int: the committed value of ErrorOutOfGasSloadSstore) rides along as a
        side table keyed by the step row"""
        import importlib
        tdir = os.path.normpath(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(sys.modules["zkevm_specs"].__file__))), "..", "tests", "evm"))
        for d_ in (tdir, os.path.dirname(tdir)):
            if d_ not in sys.path:
                sys.path.insert(0, d_)
        tc = importlib.import_module(module)
        got = {}
        keep = (tc.verify_steps, getattr(tc, "verify_copy_table", None))
        tc.verify_steps = lambda tables, steps, **kw: got.update(tables=tables, steps=steps)
        if keep[1] is not None:
            tc.verify_copy_table = lambda *a, **kw: None
        try:
            getattr(tc, fn)(*args)
        finally:
            tc.verify_steps = keep[0]
            if keep[1] is not None:
                tc.verify_copy_table = keep[1]
        if not got:
            return None  # the reference test skipped this case
        t, steps = got["tables"], got["steps"]
        aux = []
        for k_, st_ in enumerate(steps):
            a_ = st_.aux_data
            if isinstance(a_, int):
                aux.append((k_, a_ & ((1 << 128) - 1), a_ >> 128))
            elif a_ is not None:
                aux.append((k_, a_.lo.n, a_.hi.n))
        return (steps, list(t.bytecode_table), list(t.rw_table), list(getattr(t, "copy_table", [])), [], list(t.tx_table),
                list(t.block_table), [], aux)

    def create_case(idx):
        """tests/evm/test_create.py: case `idx` of the reference test's own TESTING_DATA"""
        import importlib
        tdir = os.path.normpath(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(sys.modules["zkevm_specs"].__file__))), "..", "tests", "evm"))
        for d_ in (tdir, os.path.dirname(tdir)):
            if d_ not in sys.path:
                sys.path.insert(0, d_)
        data = importlib.import_module("test_create").TESTING_DATA[idx]
        sc_ = recorded_case("test_create", "test_create_create2", data)
        return sc_[:5] + ([], [], [], sc_[8])  # the creation gadget reads neither the tx nor the block table

    def mws(a):
        return (a + 31) // 32

    def mem_exp(cur, addr):
        nxt = max(mws(addr), cur)
        return nxt, (nxt - cur) * 3 + (nxt * nxt // 512 - cur * cur // 512)

    def sha3_case(offset, length):
        mem = bytes(rng.randrange(256) for _ in range(offset + length))
        src = {i: mem[i] for i in range(offset, offset + length)}
        bc = Bytecode().push(offset, n_bytes=32).push(length, n_bytes=32).sha3().stop()
        h = Word(bc.hash())
        out = Word(int.from_bytes(keccak256(mem[offset:offset + length]), "big"))
        nxt, exp = mem_exp(mws(offset + length), offset + length)
        gas = Opcode.SHA3.constant_gas_cost() + exp + mws(length) * GAS_COST_COPY_SHA3
        rw = (RWDictionary(1).stack_write(1, 1023, Word(length)).stack_write(1, 1022, Word(offset))
              .stack_read(1, 1022, Word(offset)).stack_read(1, 1023, Word(length)).stack_write(1, 1023, out))
        cc = CopyCircuit().copy(r, rw, 1, CopyDataTypeTag.Memory, 1, CopyDataTypeTag.RlcAcc, offset, offset + length,
                                FQ.zero(), length, src)
        kc = KeccakCircuit().add(mem[offset:offset + length], r)
        steps = [StepState(ExecutionState.SHA3, rw_counter=3, call_id=1, is_root=True, code_hash=h, program_counter=66,
                           stack_pointer=1022, memory_word_size=nxt, gas_left=gas),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, code_hash=h,
                           program_counter=67, stack_pointer=1023, memory_word_size=nxt, gas_left=0)]
        t = Tables(block_table=set(), tx_table=set(), withdrawal_table=set(), bytecode_table=set(bc.table_assignments()),
                   rw_table=set(rw.rws), copy_circuit=cc.rows, keccak_table=kc.rows)
        return steps, list(bc.table_assignments()), list(rw.rws), list(t.copy_table), list(kc.rows)

    def cdc_case(cd_len, data_off, mem_off, length, from_tx, cd_off):
        bc = Bytecode().calldatacopy(mem_off, data_off, length)
        h = Word(bc.hash())
        call_data = bytes(rng.randrange(256) for _ in range(cd_len))
        cur = mws(0 if from_tx else cd_off + cd_len)
        nxt, exp = mem_exp(cur, mem_off + length if length else 0)
        gas = Opcode.CALLDATACOPY.constant_gas_cost() + exp + mws(length) * GAS_COST_COPY
        rw = (RWDictionary(1).stack_read(1, 1021, Word(mem_off)).stack_read(1, 1022, Word(data_off))
              .stack_read(1, 1023, Word(length)))
        if from_tx:
            rw.call_context_read(1, CallContextFieldTag.TxId, 13).call_context_read(1, CallContextFieldTag.CallDataLength, cd_len)
        else:
            (rw.call_context_read(1, CallContextFieldTag.CallerId, 0).call_context_read(1, CallContextFieldTag.CallDataLength, cd_len)
             .call_context_read(1, CallContextFieldTag.CallDataOffset, cd_off))
        src = {cd_off + i: call_data[i] for i in range(data_off, min(data_off + length, len(call_data)))}
        cc = CopyCircuit().copy(r, rw, 13 if from_tx else 0, CopyDataTypeTag.TxCalldata if from_tx else CopyDataTypeTag.Memory,
                                1, CopyDataTypeTag.Memory, data_off + cd_off, cd_len + cd_off, mem_off, length, src)
        steps = [StepState(ExecutionState.CALLDATACOPY, rw_counter=1, call_id=1, is_root=from_tx, code_hash=h,
                           program_counter=99, stack_pointer=1021, memory_word_size=cur, gas_left=gas),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=from_tx, code_hash=h,
                           program_counter=100, stack_pointer=1024, memory_word_size=nxt, gas_left=0)]
        t = Tables(block_table=set(), tx_table=set(), withdrawal_table=set(), bytecode_table=set(bc.table_assignments()),
                   rw_table=set(rw.rws), copy_circuit=cc.rows)
        return steps, list(bc.table_assignments()), list(rw.rws), list(t.copy_table), []

    def step_ints(s):
        return [int(s.execution_state), n_of(s.rw_counter), n_of(s.call_id), int(s.is_root), int(s.is_create),
                n_of(s.code_hash.lo), n_of(s.code_hash.hi), n_of(s.program_counter), n_of(s.stack_pointer),
                n_of(s.gas_left), n_of(s.memory_word_size), n_of(s.reversible_write_counter), n_of(s.log_id)]

    def step_from(v):
        s = StepState(ExecutionState(v[0]), rw_counter=0)
        s.rw_counter, s.call_id, s.is_root, s.is_create = FQ(v[1]), FQ(v[2]), v[3], v[4]
        s.code_hash = W(v[5], v[6])
        s.program_counter, s.stack_pointer, s.gas_left = FQ(v[7]), FQ(v[8]), FQ(v[9])
        s.memory_word_size, s.reversible_write_counter, s.log_id = FQ(v[10]), FQ(v[11]), FQ(v[12])
        return s

    def bc_ints(x):
        return [n_of(x.bytecode_hash.lo), n_of(x.bytecode_hash.hi), n_of(x.field_tag), n_of(x.index), n_of(x.is_code), n_of(x.value)]

    def rw_ints(x):
        return [n_of(x.rw_counter), n_of(x.rw), n_of(x.key0), n_of(x.id), n_of(x.address), n_of(x.field_tag),
                n_of(x.storage_key.lo), n_of(x.storage_key.hi), n_of(x.value.lo), n_of(x.value.hi),
                n_of(x.value_prev.lo), n_of(x.value_prev.hi), n_of(x.aux0.lo), n_of(x.aux0.hi)]

    def copy_ints(x):
        return [n_of(x.is_first), n_of(x.src_id.lo), n_of(x.src_id.hi), n_of(x.src_tag), n_of(x.dst_id.lo), n_of(x.dst_id.hi),
                n_of(x.dst_tag), n_of(x.src_addr), n_of(x.src_addr_end), n_of(x.dst_addr), n_of(x.length), n_of(x.rlc_acc),
                n_of(x.rw_counter), n_of(x.rwc_inc)]

    def kec_ints(x):
        return [n_of(x.state_tag), n_of(x.input_rlc), n_of(x.input_len), n_of(x.output.lo), n_of(x.output.hi)]

    def tx_ints(x):
        return [n_of(x.tx_id), n_of(x.field_tag), n_of(x.call_data_index_or_zero), n_of(x.value.lo), n_of(x.value.hi)]

    def blk_ints(x):
        return [n_of(x.field_tag), n_of(x.block_number_or_zero), n_of(x.value.lo), n_of(x.value.hi)]

    def caller_ctx_rws(rw, caller_id, ch, ctx, callee_id):
        """the 12 call-context rows of step_state_transition_to_restored_context (instruction.py:293-363)"""
        c_root, c_create, c_pc, c_sp, c_gas, c_mem, c_rev = ctx
        return (rw.call_context_read(callee_id, CallContextFieldTag.CallerId, caller_id)
                .call_context_read(caller_id, CallContextFieldTag.IsRoot, c_root)
                .call_context_read(caller_id, CallContextFieldTag.IsCreate, c_create)
                .call_context_read(caller_id, CallContextFieldTag.CodeHash, ch)
                .call_context_read(caller_id, CallContextFieldTag.ProgramCounter, c_pc)
                .call_context_read(caller_id, CallContextFieldTag.StackPointer, c_sp)
                .call_context_read(caller_id, CallContextFieldTag.GasLeft, c_gas)
                .call_context_read(caller_id, CallContextFieldTag.MemorySize, c_mem)
                .call_context_read(caller_id, CallContextFieldTag.ReversibleWriteCounter, c_rev)
                .call_context_write(caller_id, CallContextFieldTag.LastCalleeId, callee_id)
                .call_context_write(caller_id, CallContextFieldTag.LastCalleeReturnDataOffset, 0)
                .call_context_write(caller_id, CallContextFieldTag.LastCalleeReturnDataLength, 0))

    def error_case(kind, root, arg=None):
        """tests/evm/test_error_{stack,invalid_opcode,oog_constant,invalid_jump}.py: an error state in the root call
        (-> EndTx) or in an internal call (restores the caller's context), reversible_write_counter 2"""
        from zkevm_specs.evm_circuit import AccountFieldTag  # noqa: F401
        rev, pops = 2, []
        if kind == "stack_underflow":
            bc, state, pc, sp, gas = Bytecode().pop(), ExecutionState.ErrorStack, 0, 1024, 2
        elif kind == "stack_overflow":
            bc, state, pc, sp, gas = Bytecode().push1(0x10).push1(0x20), ExecutionState.ErrorStack, 2, 0, 10
        elif kind == "invalid_opcode":
            bc = Bytecode(bytearray(arg), [True] * len(arg)).stop()
            state, pc, sp, gas = ExecutionState.ErrorInvalidOpcode, 0, 1024, 2
        elif kind == "oog_constant":
            bc, state, pc, sp, gas = Bytecode().push1(0x40), ExecutionState.ErrorOutOfGasConstant, 0, 1023, 2
        else:  # invalid_jump: arg = (opcode name, dest, cond)
            op, dest, cond = arg
            bc = Bytecode().push1(0x80).push1(cond).push1(dest)
            bc = (bc.jump() if op == "jump" else bc.jumpi()).jumpdest().stop()
            state, pc, sp, gas, rev = ExecutionState.ErrorInvalidJump, 6, 1021, 8, 0
            pops = [Word(dest)] + ([Word(cond)] if op == "jumpi" else [])
        h = Word(bc.hash())
        call_id = 1 if root else 2
        rw = RWDictionary(24 if root else 69)
        rwc0 = rw.rw_counter
        for k, wd in enumerate(pops):
            rw.stack_read(call_id, sp + k, wd)
        rw.call_context_read(call_id, CallContextFieldTag.IsSuccess, 0)
        cur = StepState(state, rw_counter=rwc0, call_id=call_id, is_root=root, is_create=False, code_hash=h,
                        program_counter=pc, stack_pointer=sp, gas_left=gas, reversible_write_counter=rev)
        if root:
            nxt = StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter + rev, call_id=1, gas_left=0)
            return [cur, nxt], list(bc.table_assignments()), list(rw.rws), [], []
        cbc = Bytecode().call(0, 0xFF, 0, 0, 0, 0, 0).stop()
        ch = Word(cbc.hash())
        ctx = (True, False, 232, 1023, 10, 3, 5)
        caller_ctx_rws(rw, 1, ch, ctx, 2)
        nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter + rev, call_id=1, is_root=ctx[0], is_create=ctx[1], code_hash=ch,
                        program_counter=ctx[2], stack_pointer=ctx[3], gas_left=ctx[4], memory_word_size=ctx[5],
                        reversible_write_counter=ctx[6])
        return [cur, nxt], list(bc.table_assignments()) + list(cbc.table_assignments()), list(rw.rws), [], []

    def selfbalance_case(callee, balance):
        """tests/evm/test_selfbalance.py"""
        from zkevm_specs.evm_circuit import AccountFieldTag
        bc = Bytecode().selfbalance().stop()
        h = Word(bc.hash())
        rw = (RWDictionary(9).call_context_read(1, CallContextFieldTag.CalleeAddress, Word(callee))
              .account_read(callee, AccountFieldTag.Balance, Word(balance)).stack_write(1, 1023, Word(balance)))
        steps = [StepState(ExecutionState.SELFBALANCE, rw_counter=9, call_id=1, is_root=True, is_create=False, code_hash=h,
                           program_counter=0, stack_pointer=1024, gas_left=5),
                 StepState(ExecutionState.STOP, rw_counter=12, call_id=1, is_root=True, is_create=False, code_hash=h,
                           program_counter=1, stack_pointer=1023, gas_left=0)]
        return steps, list(bc.table_assignments()), list(rw.rws), [], []

    def oog_case(kind, root, a=0, b=0, gas_left=0, cur_mem=0, op=None):
        """tests/evm/test_error_oog_{sha3,static_memory_expansion,dynamic_memory_expansion,log,exp}.py and
        test_error_return_data_out_of_bound.py: one error step, then EndTx (root) or the restored caller"""
        rev, extra_cc = 2, []
        if kind == "sha3":       # a = offset, b = size
            bc, state, pc, sp = Bytecode().push32(b).push32(a).sha3().stop(), ExecutionState.ErrorOutOfGasSHA3, 66, 1022
            pops = [(0, Word(a)), (1, Word(b))]
        elif kind == "static":   # a = offset
            bc = Bytecode().push32(7).push32(a)
            bc = {Opcode.MLOAD: bc.mload, Opcode.MSTORE: bc.mstore, Opcode.MSTORE8: bc.mstore8}[op]().stop()
            state, pc, sp, pops = ExecutionState.ErrorOutOfGasStaticMemoryExpansion, 66, 1022, [(0, Word(a))]
        elif kind == "dynamic":  # a = offset, b = size
            bc = Bytecode().push32(b).push32(a)
            bc = (bc.return_() if op == Opcode.RETURN else bc.revert()).stop()
            state, pc, sp, pops = ExecutionState.ErrorOutOfGasDynamicMemoryExpansion, 66, 1022, [(0, Word(a)), (1, Word(b))]
        elif kind == "log":      # a = mstart, b = msize, op = LOGn
            bc = Bytecode().push32(b).push32(a)
            bc.code.append(int(op)); bc.is_code.append(True)
            bc = bc.stop()
            state, pc, sp, pops = ExecutionState.ErrorOutOfGasLOG, 66, 1022, [(0, Word(a)), (1, Word(b))]
        elif kind == "exp":      # a = exponent
            bc = Bytecode().push32(a).push32(3).exp().stop()
            state, pc, sp, pops = ExecutionState.ErrorOutOfGasEXP, 66, 1022, [(1, Word(a))]
        else:                    # return data: a = data_offset, b = length, cur_mem reused as return_data_length
            bc = Bytecode().push32(b).push32(a).push32(32).returndatacopy().stop()
            state, pc, sp, pops = ExecutionState.ErrorReturnDataOutOfBound, 99, 1021, [(1, Word(a)), (2, Word(b))]
            extra_cc = [(CallContextFieldTag.LastCalleeReturnDataLength, cur_mem)]
            cur_mem = 0
        h = Word(bc.hash())
        call_id = 1 if root else 2
        rw = RWDictionary(15 if root else 40)
        rwc0 = rw.rw_counter
        for off, wd in pops:
            rw.stack_read(call_id, sp + off, wd)
        for tag, val in extra_cc:
            rw.call_context_read(call_id, tag, val)
        rw.call_context_read(call_id, CallContextFieldTag.IsSuccess, 0)
        cur = StepState(state, rw_counter=rwc0, call_id=call_id, is_root=root, is_create=False, code_hash=h, program_counter=pc,
                        stack_pointer=sp, gas_left=gas_left, memory_word_size=cur_mem, reversible_write_counter=rev)
        if root:
            nxt = StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter + rev, call_id=1, gas_left=0)
            return [cur, nxt], list(bc.table_assignments()), list(rw.rws), [], []
        cbc = Bytecode().call(0, 0xFF, 0, 0, 0, 0, 0).stop()
        ch = Word(cbc.hash())
        ctx = (False, False, 232, 1023, 77, 3, 5)
        caller_ctx_rws(rw, 1, ch, ctx, 2)
        nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter + rev, call_id=1, is_root=ctx[0], is_create=ctx[1], code_hash=ch,
                        program_counter=ctx[2], stack_pointer=ctx[3], gas_left=ctx[4], memory_word_size=ctx[5],
                        reversible_write_counter=ctx[6])
        return [cur, nxt], list(bc.table_assignments()) + list(cbc.table_assignments()), list(rw.rws), [], []

    def account_case(kind, address, exists, is_warm, is_persistent, balance=0, code=b"", rev0=0):
        """tests/evm/test_{balance,extcodehash,extcodesize}.py: pop an address, add it to the tx access list (with its
        reversion row when the call is not persistent), read the account, push the result"""
        from zkevm_specs.evm_circuit import AccountFieldTag
        from zkevm_specs.util import EMPTY_CODE_HASH
        bc = {"balance": Bytecode().balance, "extcodehash": Bytecode().extcodehash, "extcodesize": Bytecode().extcodesize}[kind]().stop()
        h = Word(bc.hash())
        code_hash = int.from_bytes(keccak256(code), "big") if kind != "balance" else EMPTY_CODE_HASH
        rev_end = 0 if is_persistent else 40
        rw = (RWDictionary(1).stack_read(1, 1023, Word(address)).call_context_read(1, CallContextFieldTag.TxId, 1)
              .call_context_read(1, CallContextFieldTag.RwCounterEndOfReversion, rev_end)
              .call_context_read(1, CallContextFieldTag.IsPersistent, is_persistent)
              .tx_access_list_account_write(1, address, True, is_warm, rw_counter_of_reversion=rev_end - rev0))
        rw.account_read(address, AccountFieldTag.CodeHash, Word(code_hash if exists else 0))
        if kind == "balance":
            if exists:
                rw.account_read(address, AccountFieldTag.Balance, Word(balance))
            result = balance if exists else 0
        elif kind == "extcodehash":
            result = code_hash if exists else 0
        else:
            result = len(code) if exists else 0
        rw.stack_write(1, 1023, Word(result))
        state = {"balance": ExecutionState.BALANCE, "extcodehash": ExecutionState.EXTCODEHASH, "extcodesize": ExecutionState.EXTCODESIZE}[kind]
        steps = [StepState(state, rw_counter=1, call_id=1, is_root=True, is_create=False, code_hash=h, program_counter=0,
                           stack_pointer=1023, gas_left=100 + (not is_warm) * 2500, reversible_write_counter=rev0),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, is_create=False, code_hash=h,
                           program_counter=1, stack_pointer=1023, gas_left=0,
                           reversible_write_counter=rev0 + (1 if kind == "extcodesize" else 0))]
        bcs = list(bc.table_assignments()) + (list(Bytecode(bytearray(code)).table_assignments()) if kind == "extcodesize" else [])
        return steps, bcs, list(rw.rws), [], []

    def oog_account_case(op, is_warm, root):
        """tests/evm/test_error_oog_account_access.py"""
        address = 0xCAFECAFE
        bc = Bytecode().push32(address)
        bc = {Opcode.BALANCE: bc.balance, Opcode.EXTCODESIZE: bc.extcodesize, Opcode.EXTCODEHASH: bc.extcodehash}[op]().stop()
        h = Word(bc.hash())
        call_id, rev = (1 if root else 2), 2
        rw = RWDictionary(14).stack_read(call_id, 1023, Word(address)).call_context_read(call_id, CallContextFieldTag.TxId, 1)
        rw.tx_access_list_account_read(1, address, is_warm)
        rw.call_context_read(call_id, CallContextFieldTag.IsSuccess, 0)
        cur = StepState(ExecutionState.ErrorOutOfGasAccountAccess, rw_counter=14, call_id=call_id, is_root=root, is_create=False,
                        code_hash=h, program_counter=33, stack_pointer=1023, gas_left=(99 if is_warm else 2599), reversible_write_counter=rev)
        if root:
            return [cur, StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter + rev, call_id=1, gas_left=0)], list(bc.table_assignments()), list(rw.rws), [], []
        cbc = Bytecode().call(0, 0xFF, 0, 0, 0, 0, 0).stop()
        ch = Word(cbc.hash())
        ctx = (False, False, 232, 1023, 77, 3, 5)
        caller_ctx_rws(rw, 1, ch, ctx, 2)
        nxt = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter + rev, call_id=1, is_root=ctx[0], is_create=ctx[1], code_hash=ch,
                        program_counter=ctx[2], stack_pointer=ctx[3], gas_left=ctx[4], memory_word_size=ctx[5], reversible_write_counter=ctx[6])
        return [cur, nxt], list(bc.table_assignments()) + list(cbc.table_assignments()), list(rw.rws), [], []

    def codecopy_case(code_off, mem_off, length, cur_mem=0):
        """tests/evm/test_codecopy.py: the running contract's code -> memory (padding beyond the code end)"""
        bc = Bytecode().push32(length).push32(code_off).push32(mem_off).codecopy().stop()
        h = Word(bc.hash())
        nxt, exp = mem_exp(cur_mem, mem_off + length if length else 0)
        gas = Opcode.CODECOPY.constant_gas_cost() + exp + mws(length) * GAS_COST_COPY
        rw = RWDictionary(4).stack_read(1, 1021, Word(mem_off)).stack_read(1, 1022, Word(code_off)).stack_read(1, 1023, Word(length))
        src = {i: (b, int(c)) for i, (b, c) in enumerate(zip(bc.code, bc.is_code))}
        cc = CopyCircuit().copy(r, rw, h, CopyDataTypeTag.Bytecode, 1, CopyDataTypeTag.Memory, code_off, len(bc.code), mem_off, length, src)
        steps = [StepState(ExecutionState.CODECOPY, rw_counter=4, call_id=1, is_root=True, code_hash=h, program_counter=99,
                           stack_pointer=1021, memory_word_size=cur_mem, gas_left=gas),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, code_hash=h, program_counter=100,
                           stack_pointer=1024, memory_word_size=nxt, gas_left=0)]
        t = Tables(block_table=set(), tx_table=set(), withdrawal_table=set(), bytecode_table=set(bc.table_assignments()),
                   rw_table=set(rw.rws), copy_circuit=cc.rows)
        return steps, list(bc.table_assignments()), list(rw.rws), list(t.copy_table), []

    def returndatacopy_case(rd_len, rd_off, data_off, mem_off, length, cur_mem=8):
        """tests/evm/test_returndatacopy.py: the last callee's return data (its memory) -> memory"""
        bc = Bytecode().push32(length).push32(data_off).push32(mem_off).returndatacopy().stop()
        h = Word(bc.hash())
        nxt, exp = mem_exp(cur_mem, mem_off + length if length else 0)
        gas = Opcode.RETURNDATACOPY.constant_gas_cost() + exp + mws(length) * GAS_COST_COPY
        callee = 7
        rw = (RWDictionary(9).stack_read(1, 1021, Word(mem_off)).stack_read(1, 1022, Word(data_off)).stack_read(1, 1023, Word(length))
              .call_context_read(1, CallContextFieldTag.LastCalleeId, callee)
              .call_context_read(1, CallContextFieldTag.LastCalleeReturnDataLength, rd_len)
              .call_context_read(1, CallContextFieldTag.LastCalleeReturnDataOffset, rd_off))
        data = bytes(rng.randrange(256) for _ in range(rd_off + rd_len + 40))
        src = {i: data[i] for i in range(len(data))}
        cc = CopyCircuit().copy(r, rw, callee, CopyDataTypeTag.Memory, 1, CopyDataTypeTag.Memory, rd_off, rd_off + length, mem_off, length, src)
        steps = [StepState(ExecutionState.RETURNDATACOPY, rw_counter=9, call_id=1, is_root=True, code_hash=h, program_counter=99,
                           stack_pointer=1021, memory_word_size=cur_mem, gas_left=gas),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, code_hash=h, program_counter=100,
                           stack_pointer=1024, memory_word_size=nxt, gas_left=0)]
        t = Tables(block_table=set(), tx_table=set(), withdrawal_table=set(), bytecode_table=set(bc.table_assignments()),
                   rw_table=set(rw.rws), copy_circuit=cc.rows)
        return steps, list(bc.table_assignments()), list(rw.rws), list(t.copy_table), []

    def extcodecopy_case(code, exists, is_warm, is_persistent, code_off, mem_off, length, rev0=0):
        """tests/evm/test_extcodecopy.py"""
        from zkevm_specs.evm_circuit import AccountFieldTag
        address = 0xCAFE0000000000000000000000000000BEEF1234
        ext = Bytecode(bytearray(code))
        ext_hash = ext.hash() if exists else 0
        bc = Bytecode().push32(length).push32(code_off).push32(mem_off).push32(address).extcodecopy().stop()
        h = Word(bc.hash())
        nxt, exp = mem_exp(0, mem_off + length if length else 0)
        gas = Opcode.EXTCODECOPY.constant_gas_cost() + exp + mws(length) * GAS_COST_COPY + (0 if is_warm else 2500)
        rev_end = 0 if is_persistent else 60
        rw = (RWDictionary(5).stack_read(1, 1020, Word(address)).stack_read(1, 1021, Word(mem_off)).stack_read(1, 1022, Word(code_off))
              .stack_read(1, 1023, Word(length)).call_context_read(1, CallContextFieldTag.TxId, 1)
              .call_context_read(1, CallContextFieldTag.RwCounterEndOfReversion, rev_end)
              .call_context_read(1, CallContextFieldTag.IsPersistent, is_persistent)
              .tx_access_list_account_write(1, address, True, is_warm, rw_counter_of_reversion=rev_end - rev0)
              .account_read(address, AccountFieldTag.CodeHash, Word(ext_hash)))
        src = {i: (b, int(c)) for i, (b, c) in enumerate(zip(ext.code, ext.is_code))} if exists else {}
        cc = CopyCircuit()
        if length:
            cc.copy(r, rw, Word(ext_hash), CopyDataTypeTag.Bytecode, 1, CopyDataTypeTag.Memory, code_off, len(ext.code) if exists else 0,
                    mem_off, length, src)
        steps = [StepState(ExecutionState.EXTCODECOPY, rw_counter=5, call_id=1, is_root=True, code_hash=h, program_counter=132,
                           stack_pointer=1020, memory_word_size=0, gas_left=gas, reversible_write_counter=rev0),
                 StepState(ExecutionState.STOP, rw_counter=rw.rw_counter, call_id=1, is_root=True, code_hash=h, program_counter=133,
                           stack_pointer=1024, memory_word_size=nxt, gas_left=0, reversible_write_counter=rev0)]
        bcs = list(bc.table_assignments()) + (list(ext.table_assignments()) if exists else [])
        t = Tables(block_table=set(), tx_table=set(), withdrawal_table=set(), bytecode_table=set(bcs), rw_table=set(rw.rws), copy_circuit=cc.rows)
        return steps, bcs, list(rw.rws), list(t.copy_table), []

    def oog_copy_case(op, root, mem_off, length, is_warm=True):
        """tests/evm/test_error_oog_memory_copy.py"""
        ext = op == Opcode.EXTCODECOPY
        bc = Bytecode().push32(length).push32(0).push32(mem_off)
        if ext:
            bc = bc.push32(0x1234)
        bc.code.append(int(op)); bc.is_code.append(True)
        bc = bc.stop()
        h = Word(bc.hash())
        call_id, rev, sp = (1 if root else 2), 2, (1020 if ext else 1021)
        rw = RWDictionary(20)
        k = 0
        if ext:
            rw.stack_read(call_id, sp, Word(0x1234)); k = 1
        rw.stack_read(call_id, sp + k, Word(mem_off)).stack_read(call_id, sp + k + 2, Word(length))
        if ext:
            rw.call_context_read(call_id, CallContextFieldTag.TxId, 1).tx_access_list_account_read(1, 0x1234, is_warm)
        rw.call_context_read(call_id, CallContextFieldTag.IsSuccess, 0)
        nxt, exp = mem_exp(0, mem_off + length if length else 0)
        need = ((100 if is_warm else 2600) if ext else 3) + exp + mws(length) * GAS_COST_COPY
        cur = StepState(ExecutionState.ErrorOutOfGasMemoryCopy, rw_counter=20, call_id=call_id, is_root=root, is_create=False, code_hash=h,
                        program_counter=132 if ext else 99, stack_pointer=sp, gas_left=need - 1, reversible_write_counter=rev)
        if root:
            return [cur, StepState(ExecutionState.EndTx, rw_counter=rw.rw_counter + rev, call_id=1, gas_left=0)], list(bc.table_assignments()), list(rw.rws), [], []
        cbc = Bytecode().call(0, 0xFF, 0, 0, 0, 0, 0).stop()
        ch = Word(cbc.hash())
        ctx = (False, False, 232, 1023, 77, 3, 5)
        caller_ctx_rws(rw, 1, ch, ctx, 2)
        nxt_s = StepState(ExecutionState.STOP, rw_counter=rw.rw_counter + rev, call_id=1, is_root=ctx[0], is_create=ctx[1], code_hash=ch,
                          program_counter=ctx[2], stack_pointer=ctx[3], gas_left=ctx[4], memory_word_size=ctx[5], reversible_write_counter=ctx[6])
        return [cur, nxt_s], list(bc.table_assignments()) + list(cbc.table_assignments()), list(rw.rws), [], []

    def exp_ints(x):
        return [n_of(x.is_step), n_of(x.identifier), n_of(x.is_last), n_of(x.base_limb0), n_of(x.base_limb1), n_of(x.base_limb2), n_of(x.base_limb3),
                n_of(x.exponent.lo), n_of(x.exponent.hi), n_of(x.exponentiation.lo), n_of(x.exponentiation.hi)]

    def run(S, B, R, RF, C, K, T=(), BL=(), TF=None, BF=None, EX=(), AUX=()):
        from zkevm_specs.evm_circuit import BlockTableRow, TxTableRow
        steps = [step_from(v) for v in S]
        for a_ in AUX:  # StepState.aux_data of step a_[0] (a Word)
            if 0 <= a_[0] < len(steps):
                steps[a_[0]].aux_data = W(a_[1], a_[2]) if part == "evm24" else a_[1] + (a_[2] << 128)
        t = Tables(block_table=set(BlockTableRow(FQ(v[0]), FQ(v[1]), wov(v[2], v[3], 1 if BF is None else BF[k_])) for k_, v in enumerate(BL)),
                   tx_table=set(TxTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), wov(v[3], v[4], 1 if TF is None else TF[k_])) for k_, v in enumerate(T)),
                   withdrawal_table=set(),
                   bytecode_table=set(BytecodeTableRow(W(v[0], v[1]), FQ(v[2]), FQ(v[3]), FQ(v[4]), FQ(v[5])) for v in B),
                   rw_table=set(RWTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), FQ(v[3]), FQ(v[4]), FQ(v[5]), W(v[6], v[7]),
                                           wov(v[8], v[9], f & 1), wov(v[10], v[11], (f >> 1) & 1), W(v[12], v[13]))
                                for v, f in zip(R, RF)))
        t.copy_table = set(CopyTableRow(FQ(v[0]), WordOrValue(W(v[1], v[2])), FQ(v[3]), WordOrValue(W(v[4], v[5])), FQ(v[6]),
                                        FQ(v[7]), FQ(v[8]), FQ(v[9]), FQ(v[10]), FQ(v[11]), FQ(v[12]), FQ(v[13])) for v in C)
        t.keccak_table = set(KeccakTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), W(v[3], v[4])) for v in K)
        if EX or part == "evm19":  # (Tables() defines exp_table only when it is given an exp circuit)
            from zkevm_specs.evm_circuit.table import ExpTableRow
            t.exp_table = set(ExpTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), FQ(v[3]), FQ(v[4]), FQ(v[5]), FQ(v[6]), W(v[7], v[8]), W(v[9], v[10])) for v in EX)
        for idx, (cur, nxt) in enumerate(zip(steps, steps[1:])):
            try:
                verify_step(Instruction(tables=t, curr=cur, next=nxt, is_first_step=False, is_last_step=False))
            except Exception as e:  # noqa: BLE001
                return idx, type(e).__name__
        return -1, ""

    if part == "evm28":
        # every case of tests/evm/test_error_gas_uint_overflow.py that the test itself runs (it returns early where an
        # overflowing call data would be needed) + the three memory opcodes it always skips
        import importlib
        tdir = os.path.normpath(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(sys.modules["zkevm_specs"].__file__))), "..", "tests", "evm"))
        for d_ in (tdir, os.path.dirname(tdir)):
            if d_ not in sys.path:
                sys.path.insert(0, d_)
        data = importlib.import_module("test_error_gas_uint_overflow").TESTING_DATA
        scenarios = {}
        for k_, d_ in enumerate(data):
            sc_ = recorded_case("test_error_gas_uint_overflow", "test_error_gas_uint_overflow_root", d_)
            if sc_ is not None:
                scenarios["eguo_%03d" % k_] = sc_
        for k_, (op_, off_, root_) in enumerate([("mload", 1 << 64, False), ("mstore", (1 << 64) + 5, False), ("mstore8", 1 << 200, False),
                                                   ("mload", (1 << 70) + 3, True), ("mstore8", 1 << 64, True)]):
            try:
                scenarios["eguo_mem_%d" % k_] = eguo_mem_case(op_, off_, root_)
                S_ = scenarios["eguo_mem_%d" % k_]
            except Exception:
                raise
    elif part == "evm27":
        # only DATACOPY and BN254PAIRING can verify: for the other seven precompiles gas_cost stays a Python int and
        # compare() raises AttributeError on it (error_oog_precompile.py:19-30) - reached here through the corruptions of the
        # callee-address cell; a root call cannot end in this state (it does not count as halting, execution_state.py:364-390)
        scenarios = {}
        scenarios["eopc_copy_0"] = eopc_case(4, 0, 14)
        scenarios["eopc_copy_33"] = eopc_case(4, 33, 15 + 6 - 1)
        scenarios["eopc_copy_640"] = eopc_case(4, 640, 15 + 60 - 1)
        scenarios["eopc_copy_1"] = eopc_case(4, 1, 0)
        scenarios["eopc_pair_0"] = eopc_case(8, 0, 44999)
        scenarios["eopc_pair_2"] = eopc_case(8, 384, 45000 + 68000 - 1)
        scenarios["eopc_pair_5"] = eopc_case(8, 960, 100)
    elif part == "evm26":
        # every case of tests/evm/test_error_oog_create.py (two of them walk 320 bytes of tx call data)
        import importlib
        tdir = os.path.normpath(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(sys.modules["zkevm_specs"].__file__))), "..", "tests", "evm"))
        for d_ in (tdir, os.path.dirname(tdir)):
            if d_ not in sys.path:
                sys.path.insert(0, d_)
        data = importlib.import_module("test_error_oog_create").TESTING_DATA_IS_ROOT
        scenarios = {"eocr_%d" % k_: recorded_case("test_error_oog_create", "test_error_oog_create", d_) for k_, d_ in enumerate(data)}
    elif part == "evm25":
        import itertools
        # every case of tests/evm/test_error_oog_sload_store.py
        scenarios = {"eoss_sload_%d" % int(w_): recorded_case("test_error_oog_sload_store", "test_error_oog_sload", (w_,)) for w_ in (False, True)}
        for o_, p_, v_, w_, c_ in itertools.product((0, 1), (1, 2), (1, 2), (True, False), (True, False)):
            scenarios["eoss_sstore_%d%d%d%d%d" % (o_, p_, v_, int(w_), int(c_))] = recorded_case(
                "test_error_oog_sload_store", "test_error_oog_sstore", (o_, p_, v_, w_, c_))
    elif part == "evm24":
        # 52 of the reference test's 1,152 cases: 3-4 of each of its 14 outcome classes (CREATE / CREATE2 x pre-check failure,
        # address collision, creation without init code (reverting or not), creation with init code = a new call context)
        picks = [0, 72, 75, 78, 97, 103, 106, 145, 216, 219, 222, 241, 247, 250, 297, 372, 377, 378, 397, 403, 516, 521, 522,
                 541, 547, 575, 576, 648, 651, 654, 673, 679, 682, 721, 792, 795, 798, 817, 823, 826, 873, 948, 953, 954, 973,
                 979, 1092, 1097, 1098, 1117, 1123, 1151]
        scenarios = {"create_%04d" % k_: create_case(k_) for k_ in picks}
    elif part == "evm23":
        # 36 of the reference test's 768 cases: every opcode x callee kind, both reversion settings, the four stack shapes,
        # warm / cold, depth 1 / 1024 / 1025 (index = a mixed-radix number over the test's product order)
        picks = []
        for op_i in range(4):
            for callee_i in range(4):
                for v in range(2):
                    ctx_i, stack_i = (op_i + callee_i + v) % 2, (op_i * 2 + callee_i + v) % 4
                    warm_i, depth_i = (callee_i + v) % 2, (0 if v == 0 else (op_i + callee_i) % 3)
                    picks.append((((((op_i * 4 + callee_i) * 2 + ctx_i) * 4 + stack_i) * 2 + warm_i) * 3) + depth_i)
        picks += [5, 100, 300, 700]
        scenarios = {"callop_%03d" % k_: callop_case(k_) for k_ in sorted(set(picks))}
    elif part == "evm22":
        scenarios = {
            "call_warm_root": oog_call_case("call", True, True, 50), "call_cold_internal": oog_call_case("call", False, False, 100),
            "call_value_root": oog_call_case("call", True, True, 9100, value=5), "callcode_cold_root": oog_call_case("callcode", True, False, 2600),
            "callcode_value_internal": oog_call_case("callcode", False, True, 9000, value=1 << 200),
            "delegatecall_warm_root": oog_call_case("delegatecall", True, True, 50), "delegatecall_cold_internal": oog_call_case("delegatecall", False, False, 2000, cur_mem=20),
            "staticcall_warm_internal": oog_call_case("staticcall", False, True, 100, cd=(0, 0), rd=(0x400, 0x40)),
            "staticcall_cold_root": oog_call_case("staticcall", True, False, 2599, cd=(0, 0), rd=(0, 0)),
        }
    elif part == "evm21":
        scenarios = {
            "ret_root": return_case("root", True, 4, 10), "rev_root": return_case("root", False, 4, 10), "ret_root_expand": return_case("root", True, 4, 100),
            "ret_internal_short": return_case("internal", True, 4, 8), "rev_internal_short": return_case("internal", False, 4, 8),
            "ret_internal_equal": return_case("internal", True, 4, 10), "ret_internal_long": return_case("internal", True, 4, 20),
            "rev_internal_expand": return_case("internal", False, 4, 100), "ret_internal_one": return_case("internal", True, 0, 1),  # (a zero-length return to a caller cannot verify: the copy lookup is unconditional)
            "ret_create_root": return_case("create_root", True, 4, 0), "rev_create_root": return_case("create_root", False, 4, 0),
            "ret_create_internal": return_case("create_internal", True, 4, 0), "rev_create_internal": return_case("create_internal", False, 4, 0),
        }
    elif part == "evm20":
        scenarios = {
            "oog_store_root": code_store_case("oog", True), "oog_store_internal": code_store_case("oog", False),
            "oog_store_max_size": code_store_case("oog", True, size=24576, gas_left=24576 * 200 - 1),
            "max_size_root": code_store_case("max", True, size=24577, gas_left=5000000), "max_size_internal": code_store_case("max", False, size=24577, gas_left=2000000),
            "max_size_both": code_store_case("max", True, size=60000, gas_left=100),
            "invalid_code_root": code_store_case("invalid", True), "invalid_code_internal": code_store_case("invalid", False),
        }
    elif part == "evm19":
        MX = (1 << 256) - 1
        scenarios = {
            "exp_0_0": exp_case(0, 0), "exp_0_max": exp_case(0, MX), "exp_1_max": exp_case(1, MX), "exp_cafe_0": exp_case(0xCAFE, 0),
            "exp_max_1": exp_case(MX, 1), "exp_cafe_1": exp_case(0xCAFE, 1), "exp_2_5": exp_case(2, 5), "exp_3_101": exp_case(3, 101),
            "exp_5_259": exp_case(5, 259), "exp_7_1023": exp_case(7, 1023), "exp_max_2": exp_case(MX, 2), "exp_max_3": exp_case(MX, 3),
            "exp_max_max": exp_case(MX, MX), "exp_big_base": exp_case(rng.randrange(1 << 256), 6), "exp_2_256": exp_case(2, 256),
            "exp_wide_exponent": exp_case(3, (1 << 200) + 12345),
        }
    elif part == "evm18":
        scenarios = {
            "log0_empty": log_case([], 10, 0, True), "log1": log_case([0x030201], 10, 2, True), "log2": log_case([0x030201, 0x0F0E0D], 100, 20, True, cur_mem=2),
            "log3": log_case([0x030201, 0x0F0E0D, 0x0D8F01], 180, 50, True, log_id=4), "log4": log_case([(1 << 255) + 5, 2, 3, (1 << 200) + 9], 0x40, 33, True),
            "log0_data": log_case([], 0, 70, True, cur_mem=8), "log2_reverted": log_case([0x030201, 0x0F0E0D], 100, 20, False),
            "log0_reverted_empty": log_case([], 5, 0, False, log_id=2), "log4_reverted": log_case([9, 8, 7, 6], 0x100, 5, False, cur_mem=1),
            "ewp_call_root": ewp_case("call", True), "ewp_call_internal": ewp_case("call", False, value=(1 << 130)),
            "ewp_sstore_internal": ewp_case("sstore", False), "ewp_log_root": ewp_case("log0", True),
            "bh_prev": blockhash_case(1000, 999), "bh_oldest": blockhash_case(1000, 745), "bh_too_old": blockhash_case(1000, 744),
            "bh_current": blockhash_case(1000, 1000), "bh_future": blockhash_case(300, 40000), "bh_genesis": blockhash_case(5, 0),
            "bh_edge": blockhash_case(70, 65279),
        }
    elif part == "evm17":
        cd = bytes(rng.randrange(1, 256) for _ in range(80))
        scenarios = {
            "sload_cold": storage_case("sload"), "sload_warm": storage_case("sload", warm=True, value=(1 << 255) + 7, original=5),
            "sload_cold_reverted": storage_case("sload", persistent=False, rev0=3), "sload_warm_reverted": storage_case("sload", warm=True, persistent=False, rev0=1),
            "sstore_same": storage_case("sstore", value=0x1F2E3D, value_prev=0x1F2E3D, original=0x1F2E3D), "sstore_set": storage_case("sstore", 1, 0, 0, warm=True),
            "sstore_reset": storage_case("sstore", 2, 1, 1), "sstore_clear": storage_case("sstore", 0, 1, 1, warm=True),
            "sstore_dirty": storage_case("sstore", 3, 2, 1), "sstore_dirty_restore": storage_case("sstore", 1, 2, 1, warm=True),
            "sstore_dirty_from_zero": storage_case("sstore", 7, 0, 1), "sstore_dirty_to_zero": storage_case("sstore", 0, 2, 1),
            "sstore_restore_zero": storage_case("sstore", 0, 2, 0, warm=True),
            "sstore_reverted": storage_case("sstore", 2, 1, 1, persistent=False, rev0=0), "sstore_reverted_warm": storage_case("sstore", 9, 0, 0, warm=True, persistent=False, rev0=2),
            "cdl_root_full": calldataload_case(cd, 0x20, 0, True), "cdl_root_tail": calldataload_case(cd, 0x20, 0x1F, True),
            "cdl_root_mid": calldataload_case(cd, 0x30, 0x10, True), "cdl_root_beyond": calldataload_case(cd, 0x20, 0x40, True),
            "cdl_internal": calldataload_case(cd, 0x20, 0x10, False), "cdl_internal_off": calldataload_case(cd, 0x21, 0x10, False, cd_off=1),
            "cdl_internal_full": calldataload_case(cd, 0x40, 0x08, False, cd_off=3),
        }
    elif part == "evm16":
        MX, NEG = (1 << 256) - 1, 1 << 255
        big1, big2, big3 = rng.randrange(1 << 256), rng.randrange(1 << 256), rng.randrange(1 << 200)
        scenarios = {
            "addmod_max": arith_case("addmod", MX, MX, MX), "addmod_n1": arith_case("addmod", MX, MX, 1), "addmod_n0": arith_case("addmod", MX, 1, 0),
            "addmod_rand": arith_case("addmod", big1, big2, big3), "addmod_small": arith_case("addmod", 10, 7, 6), "addmod_wrap": arith_case("addmod", MX, 5, MX - 1),
            "mulmod_max": arith_case("mulmod", MX, MX, MX - 4), "mulmod_n0": arith_case("mulmod", 7, 9, 0), "mulmod_rand": arith_case("mulmod", big1, big2, big3),
            "mulmod_small": arith_case("mulmod", 10, 7, 6), "mulmod_n1": arith_case("mulmod", big2, big1, 1),
            "sdiv_pos": arith_case("sdiv", 0xFFFFFF, 0xABC), "sdiv_neg": arith_case("sdiv", NEG + (7 << 128), 0x1234), "sdiv_m1": arith_case("sdiv", MX, 0xABCDEF),
            "sdiv_by_m1": arith_case("sdiv", 0xABCDEF, MX), "sdiv_overflow": arith_case("sdiv", NEG, MX), "sdiv_zero": arith_case("sdiv", 0xABC, 0),
            "sdiv_zero_any": arith_case("sdiv", 0xABC, 0, res=77), "sdiv_rand": arith_case("sdiv", big1, big3),
            "smod_pos": arith_case("smod", 0xFFFFFF, 0xABC), "smod_neg": arith_case("smod", NEG + (7 << 128), 0x1234), "smod_by_m1": arith_case("smod", 0xABCDEF, MX),
            "smod_overflow": arith_case("smod", NEG, MX), "smod_zero": arith_case("smod", 0xABC, 0), "smod_rand": arith_case("smod", big2, big3),
            "smod_negneg": arith_case("smod", MX - 1000, MX - 6),
            "sar_8": arith_case("sar", 8, 0x1234), "sar_neg17": arith_case("sar", 17, NEG + 0x5678), "sar_0": arith_case("sar", 0, NEG + 0xABCD),
            "sar_64": arith_case("sar", 64, big1 | NEG), "sar_129": arith_case("sar", 129, NEG), "sar_255": arith_case("sar", 255, MX),
            "sar_256": arith_case("sar", 256, NEG + 0xFFFF), "sar_265": arith_case("sar", 265, 0x12345), "sar_bigshift": arith_case("sar", NEG + 8, NEG + 0x1234),
            "sar_rand": arith_case("sar", 77, big2), "sar_192": arith_case("sar", 192 + 5, big1 | NEG),
        }
    elif part == "evm15":
        ext_code = bytes([0x60, 0x05, 0x7F]) + bytes(range(32)) + bytes([0x00, 0x5B, 0x01])
        scenarios = {
            "codecopy_single": codecopy_case(0, 0, 54), "codecopy_multi": codecopy_case(0, 0x40, 123), "codecopy_oob": codecopy_case(0x10, 0x20, 200, cur_mem=2),
            "codecopy_zero": codecopy_case(3, 0x40, 0),
            "rdc_basic": returndatacopy_case(64, 0, 0, 0x20, 64), "rdc_offset": returndatacopy_case(96, 0x40, 32, 0x100, 48),
            "rdc_one": returndatacopy_case(32, 8, 0, 0x40, 1),  # (a zero-length RETURNDATACOPY cannot verify in the reference:
                                                                 # its copy_lookup is unconditional, returndatacopy.py:36-46)
            "ext_warm": extcodecopy_case(ext_code, True, True, True, 0, 0x20, 30), "ext_cold_oob": extcodecopy_case(ext_code, True, False, True, 10, 0, 64),
            "ext_missing": extcodecopy_case(ext_code, False, False, True, 0, 0x40, 16), "ext_reverted": extcodecopy_case(ext_code, True, True, False, 2, 0x60, 20, rev0=1),
            "ext_zero": extcodecopy_case(ext_code, True, False, True, 0, 0, 0),
            "oog_cdc_root": oog_copy_case(Opcode.CALLDATACOPY, True, 0x40, 64), "oog_codecopy_internal": oog_copy_case(Opcode.CODECOPY, False, 0x100, 33),
            "oog_rdc_root": oog_copy_case(Opcode.RETURNDATACOPY, True, 0, 0), "oog_ext_cold_root": oog_copy_case(Opcode.EXTCODECOPY, True, 0x20, 40, is_warm=False),
            "oog_ext_warm_internal": oog_copy_case(Opcode.EXTCODECOPY, False, 0x20, 40, is_warm=True),
        }
    elif part == "evm14":
        A = 0xCAFE0000000000000000000000000000BEEF1234
        scenarios = {
            "bal_warm_missing": account_case("balance", 0x30000, False, True, True), "bal_cold_exists": account_case("balance", 0x30000, True, False, True, balance=200),
            "bal_reverted": account_case("balance", A, True, False, False, balance=(1 << 255) + 9, rev0=3),
            "bal_reverted_missing": account_case("balance", A, False, True, False),
            "hash_warm": account_case("extcodehash", 0x30000, True, True, True, code=bytes([10, 40])), "hash_cold_missing": account_case("extcodehash", A, False, False, True),
            "hash_reverted": account_case("extcodehash", A, True, False, False, code=bytes(range(50)), rev0=1),
            "size_warm": account_case("extcodesize", 0x30000, True, True, True, code=bytes([10, 40])), "size_cold_missing": account_case("extcodesize", A, False, False, True, code=bytes([1])),
            "size_empty_code": account_case("extcodesize", 0x30000, True, False, True, code=b""),
            "size_reverted": account_case("extcodesize", A, True, True, False, code=bytes(range(100)), rev0=2),
            "oog_bal_warm_root": oog_account_case(Opcode.BALANCE, True, True), "oog_size_cold_internal": oog_account_case(Opcode.EXTCODESIZE, False, False),
            "oog_hash_cold_root": oog_account_case(Opcode.EXTCODEHASH, False, True),
        }
    elif part == "evm13":
        M64 = (1 << 64) - 1
        scenarios = {
            "sha3_root": oog_case("sha3", True, 0x20, 0x40, 40), "sha3_internal_zero": oog_case("sha3", False, 0x20, 0, 29),
            "sha3_mem": oog_case("sha3", True, 0x100, 0x21, 50, cur_mem=2),
            "static_mload_root": oog_case("static", True, 0x40, gas_left=5, op=Opcode.MLOAD),
            "static_mstore_internal": oog_case("static", False, 0x1000, gas_left=300, op=Opcode.MSTORE),
            "static_mstore8": oog_case("static", True, 0x20, gas_left=2, cur_mem=9, op=Opcode.MSTORE8),
            "dynamic_return_root": oog_case("dynamic", True, 0x40, 0x40, 11, op=Opcode.RETURN),
            "dynamic_revert_internal": oog_case("dynamic", False, 0x100, 0x101, 20, cur_mem=1, op=Opcode.REVERT),
            "log0_internal": oog_case("log", False, 32, 32, 636, op=Opcode.LOG0), "log2_root": oog_case("log", True, 32, 32, 1386, op=Opcode.LOG2),
            "log4_zero": oog_case("log", True, 0, 0, 1874, op=Opcode.LOG4),
            "exp_0_internal": oog_case("exp", False, 0, gas_left=9), "exp_10_root": oog_case("exp", True, 10, gas_left=59),
            "exp_max": oog_case("exp", False, (1 << 256) - 1, gas_left=1609),
            "rdo_offset_over": oog_case("rdo", True, M64 + 1, 0, 5, cur_mem=320), "rdo_end_over": oog_case("rdo", False, M64, 1, 5, cur_mem=320),
            "rdo_len": oog_case("rdo", True, 320, 1, 5, cur_mem=320), "rdo_big": oog_case("rdo", False, 0, M64 + 1, 5, cur_mem=320),
        }
    elif part == "evm12":
        scenarios = {
            "estk_under_root": error_case("stack_underflow", True), "estk_over_internal": error_case("stack_overflow", False),
            "einv_0e_root": error_case("invalid_opcode", True, [0x0E]), "einv_fe_internal": error_case("invalid_opcode", False, [0xFE]),
            "einv_many_root": error_case("invalid_opcode", True, [0x5C, 0x5D, 0x5E]),
            "eogc_root": error_case("oog_constant", True), "eogc_internal": error_case("oog_constant", False),
            "ejmp_jump_root": error_case("invalid_jump", True, ("jump", 5, 0x40)),
            "ejmp_jump_oob_root": error_case("invalid_jump", True, ("jump", 20, 0x40)),
            "ejmp_jumpi_internal": error_case("invalid_jump", False, ("jumpi", 5, 0x40)),
            "ejmp_jump_internal_oob": error_case("invalid_jump", False, ("jump", 20, 0x40)),
            "selfbalance_0": selfbalance_case(0, 10), "selfbalance_big": selfbalance_case(0xCAFE0000000000000000000000000000BEEF1234, (1 << 255) + 987654321),
        }
    elif part == "evm10":
        v = 0xFEDCBA9876543210F0E1D2C3B4A5968778695A4B3C2D1E0F0123456789ABCDEF
        scenarios = {
            "shl_0": shift_case("shl", 0, v), "shl_1": shift_case("shl", 1, v), "shl_64": shift_case("shl", 64, v),
            "shl_129": shift_case("shl", 129, v), "shl_255": shift_case("shl", 255, v), "shl_256": shift_case("shl", 256, v),
            "shl_big": shift_case("shl", (1 << 200) + 3, v),
            "shr_0": shift_case("shr", 0, v), "shr_7": shift_case("shr", 7, v), "shr_128": shift_case("shr", 128, v),
            "shr_200": shift_case("shr", 200, v), "shr_255": shift_case("shr", 255, v), "shr_300": shift_case("shr", 300, v),
        }
    elif part == "evm9":
        scenarios = {
            "coinbase": ctx_case("coinbase", 0xC014BA5E0000000000000000000000000000BA5E), "timestamp": ctx_case("timestamp", 1700000000),
            "number": ctx_case("number", 1234567), "gaslimit": ctx_case("gaslimit", 30_000_000),
            "prevrandao": ctx_case("prevrandao", (1 << 255) + 42), "basefee": ctx_case("basefee", 12_000_000_000),
            "chainid": ctx_case("chainid", 1337), "origin": ctx_case("origin", 0x0123456789ABCDEF0123456789ABCDEF01234567),
            "gasprice": ctx_case("gasprice", (1 << 130) + 77),
        }
    elif part == "evm8":
        neg5, neg9, big = (1 << 256) - 5, (1 << 256) - 9, (1 << 254) + 99
        scenarios = {
            "slt_nn": signed_case("slt", neg9, neg5), "slt_np": signed_case("slt", neg5, 7), "slt_pn": signed_case("slt", 7, neg5),
            "slt_pp": signed_case("slt", 7, big), "slt_eq": signed_case("slt", big, big),
            "sgt_nn": signed_case("sgt", neg5, neg9), "sgt_np": signed_case("sgt", neg5, 7), "sgt_pn": signed_case("sgt", 7, neg5),
            "sext_0_neg": signed_case("signextend", 0, 0x1234FF), "sext_0_pos": signed_case("signextend", 0, 0x12347F),
            "sext_5": signed_case("signextend", 5, 0xAB80FFEEDDCC), "sext_30": signed_case("signextend", 30, big),
            "sext_31": signed_case("signextend", 31, neg9), "sext_big": signed_case("signextend", (1 << 100) + 40, 0x80),
        }
    elif part == "evm7":
        x, y = 0x0123456789ABCDEFFEDCBA98765432100F1E2D3C4B5A69788796A5B4C3D2E1F0, (1 << 255) | 0xFF00FF00FF00FF00FF00FF00FF00FF00
        scenarios = {
            "and": bit_case("and", x, y), "or": bit_case("or", x, y), "xor": bit_case("xor", x, y), "not": bit_case("not", x),
            "byte_0": bit_case("byte", 0, x), "byte_31": bit_case("byte", 31, x), "byte_7": bit_case("byte", 7, y),
            "byte_32": bit_case("byte", 32, x), "byte_big": bit_case("byte", 1 << 200, x),
        }
    elif part == "evm6":
        scenarios = {
            "caller": cc_push_case("caller", 0xCAFE0000000000000000000000000000BEEF1234), "callvalue": cc_push_case("callvalue", (1 << 200) + 5),
            "calldatasize": cc_push_case("calldatasize", 1234), "address": cc_push_case("address", 0xABCDEF0123456789ABCDEF0123456789ABCDEF01),
            "returndatasize": cc_push_case("returndatasize", 77), "codesize": cc_push_case("codesize", 0x1234),
        }
    elif part == "evm5":
        big = (1 << 255) + 12345
        scenarios = {
            "msize_0": simple_case("msize", 0), "msize_7": simple_case("msize", 7), "gas": simple_case("gas", 1000),
            "iszero_0": simple_case("iszero", 0), "iszero_big": simple_case("iszero", big),
            "lt_true": simple_case("lt", 5, big), "lt_false": simple_case("lt", big, 5), "lt_hi_eq": simple_case("lt", (7 << 128) + 1, (7 << 128) + 2),
            "gt_true": simple_case("gt", big, 5), "gt_false": simple_case("gt", 5, 5),
            "eq_true": simple_case("eq", big, big), "eq_false": simple_case("eq", big, big + 1),
            "jump": simple_case("jump", 40), "jumpi_zero": simple_case("jumpi", 90, 0), "jumpi_nonzero": simple_case("jumpi", 90, 40),
        }
    elif part == "evm4":
        scenarios = {
            "mload_0": memory_case(Opcode.MLOAD, 0, 0xFF), "mload_1": memory_case(Opcode.MLOAD, 1, 0xFF00, 3),
            "mstore_0": memory_case(Opcode.MSTORE, 0, 0xFF), "mstore_big": memory_case(Opcode.MSTORE, 0x1234, (1 << 255) + 77, 5),
            "mstore8_0": memory_case(Opcode.MSTORE8, 0, 0xFFFF), "mstore8_1": memory_case(Opcode.MSTORE8, 0x21, 0xAB, 1),
        }
    elif part == "evm3":
        scenarios = {
            "stop_root_oob": stop_case(True, False), "stop_root": stop_case(True, True),
            "stop_internal_oob": stop_case(False, False), "stop_internal": stop_case(False, True),
            "stop_internal_create": stop_case(False, True, (True, True, 7, 1000, 12345, 0, 0)),
        }
    else:
      scenarios = {
        "sha3_a": sha3_case(0x20, 0x40), "sha3_b": sha3_case(0x11, 0x23), "sha3_zero": sha3_case(0x202, 0),
        "cdc_root": cdc_case(32, 5, 0xA0, 8, True, 0), "cdc_internal": cdc_case(32, 5, 0xA0, 8, False, 0x20),
        "cdc_oob": cdc_case(32, 5, 0xA0, 45, True, 0), "cdc_zero": cdc_case(32, 5, 0xA0, 0, False, 0x20),
    }
    out = {"names": np.array(list(scenarios.keys()))}
    tot = nfail = 0
    for name, sc_ in scenarios.items():
        steps, bcs, rws, cps, kcs = sc_[:5]
        T = [tx_ints(x) for x in sc_[5]] if len(sc_) > 5 else []
        BL = [blk_ints(x) for x in sc_[6]] if len(sc_) > 6 else []
        S, B, R = [step_ints(x) for x in steps], [bc_ints(x) for x in bcs], [rw_ints(x) for x in rws]
        RF = [int(x.value.is_word) | (int(x.value_prev.is_word) << 1) for x in rws]
        C, K = [copy_ints(x) for x in cps], [kec_ints(x) for x in kcs]
        TF = [int(x.value.is_word) for x in sc_[5]] if part in ("evm17", "evm26", "evm28") and len(sc_) > 5 else None
        BF = [int(x.value.is_word) for x in sc_[6]] if part == "evm18" and len(sc_) > 6 else None
        EX = [exp_ints(x) for x in sc_[7]] if len(sc_) > 7 else []
        AUX = [list(x) for x in sc_[8]] if len(sc_) > 8 else []
        assert run(S, B, R, RF, C, K, T, BL, TF, BF, EX, AUX) == (-1, ""), (name, run(S, B, R, RF, C, K, T, BL, TF, BF, EX, AUX))
        muts = [(-1, 0, 0, 0, -1, "")]
        for k in range({"evm2": 70, "evm3": 160, "evm4": 110, "evm5": 60, "evm6": 90, "evm7": 70, "evm8": 60, "evm9": 70, "evm10": 70, "evm12": 75, "evm13": 75, "evm14": 90, "evm15": 100, "evm16": 45, "evm17": 80, "evm18": 80, "evm19": 75, "evm20": 90, "evm21": 110, "evm22": 100, "evm23": 70, "evm24": 60, "evm25": 50, "evm26": 90, "evm27": 70, "evm28": 30}[part]):
            which = rng.choice([0, 0, 0, 1, 1, 2, 3, 4] if part == "evm2" else [0, 0, 0, 1, 1, 1, 2, 3, 3, 5] if part in ("evm15", "evm21") else [0, 0, 1, 1, 8, 8, 8, 8, 8, 2, 5] if part == "evm16" else [0, 0, 0, 1, 1, 1, 1, 8, 2, 2, 9, 5, 3, 15] if part == "evm24" else [0, 0, 0, 1, 1, 1, 1, 8, 2, 9, 5, 15, 15] if part == "evm25" else [0, 0, 0, 1, 1, 1, 8, 2, 5, 6, 6, 6] if part == "evm26" else [0, 0, 0, 1, 1, 1, 2, 5, 16, 16, 16, 16] if part == "evm27" else [0, 0, 1, 1, 1, 8, 8, 8, 8, 2, 5, 6] if part == "evm28" else [0, 0, 0, 1, 1, 1, 1, 8, 2, 2, 9, 5, 6] if part in ("evm17", "evm23") else [0, 0, 0, 1, 1, 1, 1, 8, 2, 3, 3, 5, 7, 7] if part == "evm18" else [0, 0, 1, 1, 8, 8, 8, 2, 5, 14, 14, 14, 14] if part == "evm19" else
                               [0, 0, 0, 1, 1, 2, 5, 6, 6, 7, 7] if part == "evm9" else [0, 0, 0, 1, 1, 1, 2, 5])
            T2, BL2 = [list(x) for x in T], [list(x) for x in BL]
            TF2 = list(TF) if TF is not None else None
            BF2 = list(BF) if BF is not None else None
            EX2 = [list(x) for x in EX]
            AUX2 = [list(x) for x in AUX]
            S2, R2, RF2, C2, K2 = [list(x) for x in S], [list(x) for x in R], list(RF), [list(x) for x in C], [list(x) for x in K]
            if which == 0:
                cols = [1, 2, 3, 7, 8, 9, 10, 10, 9, 5] if part == "evm2" else [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 7, 7]
                i, c = rng.randrange(len(S)), rng.choice(cols)
                if c == 0:
                    v = rng.choice([int(ExecutionState.EndTx), int(ExecutionState.STOP), int(ExecutionState.ADD),
                                    int(ExecutionState.EndBlock)])
                    if v == S[i][c]:
                        continue
                else:
                    v = (1 - S[i][c]) if c in (3, 4) else corrupt_value(rng, S[i][c])
                S2[i][c] = v
            elif which == 1:
                i, c = rng.randrange(len(R)), rng.randrange(10)
                if c == 9 and not (RF[i] & 1):
                    continue
                v = corrupt_value(rng, R[i][c]); R2[i][c] = v
            elif which == 16:  # ErrorOutOfGasPrecompile: the callee address / the call-data length of the current call
                from zkevm_specs.evm_circuit.table import Target as Target_
                is_addr = rng.random() < 0.5
                tag_ = int(CallContextFieldTag.CalleeAddress if is_addr else CallContextFieldTag.CallDataLength)
                rows_ = [q for q in range(len(R)) if R[q][2] == int(Target_.CallContext) and R[q][3] == 2 and R[q][4] == tag_]
                i, c = rows_[0], 8
                v = rng.choice([1, 2, 3, 5, 6, 7, 9, 0, 10, 4, 8, 1 << 160] if is_addr else
                               [191, 193, 576, 1 << 64, 192 << 50, 32 << 32, (32 << 32) - 31, 100, 7, 0])
                if v == R[i][c]:
                    continue
                R2[i][c] = v; which = 1
            elif which == 9:  # storage key / previous value / committed value cells of an rw row
                i, c = rng.randrange(len(R)), rng.choice([6, 7, 10, 11, 12, 13])
                if c == 11 and not (RF[i] & 2):
                    continue  # the high cell of a non-Word value does not exist in the reference's row
                v = corrupt_value(rng, R[i][c]); R2[i][c] = v; which = 1
            elif which == 6 and T and TF is not None and rng.random() < 0.25:  # the value type of a tx-table row
                i, c, v = rng.randrange(len(T)), 100, 0
                TF2[i] ^= 1; which = 12
            elif which == 7 and BL and BF is not None and rng.random() < 0.2:  # the value type of a block-table row
                i, c, v = rng.randrange(len(BL)), 100, 0
                BF2[i] ^= 1; which = 13
            elif which == 15 and AUX:  # the step's aux_data (the init code's hash)
                i, c = rng.randrange(len(AUX)), rng.choice([1, 2])
                v = corrupt_value(rng, AUX[i][c]); AUX2[i][c] = v
            elif which == 14 and EX:  # a cell of an exp-table row
                i, c = rng.randrange(len(EX)), rng.randrange(11)
                v = corrupt_value(rng, EX[i][c]); EX2[i][c] = v
            elif which == 8:  # a stack word half: the operands and results of the arithmetic gadgets
                i, c = rng.randrange(len(R)), rng.choice([8, 8, 9])
                if c == 9 and not (RF[i] & 1):
                    continue
                v = corrupt_value(rng, R[i][c]); R2[i][c] = v; which = 1
            elif which == 2:
                i, c, v = rng.randrange(len(R)), 100, 0
                RF2[i] ^= 1
                if not RF2[i] & 1:
                    R2[i][9] = 0
            elif which == 5:  # a second rw row with the same key and another value: ambiguous lookup
                i, c = rng.randrange(len(R)), 8
                v = corrupt_value(rng, R[i][c])
                R2.append(list(R[i])); R2[-1][c] = v; RF2.append(RF[i])
            elif which == 6 and T:
                i, c = rng.randrange(len(T)), rng.randrange(5)
                v = corrupt_value(rng, T[i][c]); T2[i][c] = v
            elif which == 7 and BL:
                i, c = rng.randrange(len(BL)), rng.randrange(4)
                v = corrupt_value(rng, BL[i][c]); BL2[i][c] = v
            elif which == 3 and C:
                i, c = rng.randrange(len(C)), rng.randrange(14)
                if c in (2, 5):
                    continue
                v = corrupt_value(rng, C[i][c]); C2[i][c] = v
            elif which == 4 and K:
                i, c = rng.randrange(len(K)), rng.randrange(5)
                v = corrupt_value(rng, K[i][c]); K2[i][c] = v
            else:
                continue
            fr_, ex_ = run(S2, B, R2, RF2, C2, K2, T2, BL2, TF2, BF2, EX2, AUX2)
            muts.append((which, i, c, v, fr_, ex_))
            tot += 1
            nfail += fr_ >= 0
        for key, rows_, ncol in (("steps", S, 13), ("bytecode", B, 6), ("rw", R, 14), ("copy", C, 14), ("keccak", K, 5)):
            out[f"{name}/{key}"] = to_matrix(rows_) if rows_ else np.zeros((ncol, 0, 4), dtype=np.uint64)
        out[f"{name}/rw_flags"] = np.array(RF, dtype=np.uint8)
        if TF is not None:
            out[f"{name}/tx"] = to_matrix(T) if T else np.zeros((5, 0, 4), dtype=np.uint64)
            out[f"{name}/tx_flags"] = np.array(TF, dtype=np.uint8)
        if AUX:
            out[f"{name}/aux"] = to_matrix(AUX)
        if EX:
            out[f"{name}/exp"] = to_matrix(EX)
        if BF is not None:
            out[f"{name}/block_flags"] = np.array(BF, dtype=np.uint8)
        if part in ("evm9", "evm18"):
            out[f"{name}/tx"] = to_matrix(T) if T else np.zeros((5, 0, 4), dtype=np.uint64)
            out[f"{name}/block"] = to_matrix(BL) if BL else np.zeros((4, 0, 4), dtype=np.uint64)
        out[f"{name}/mut_kind"] = np.array([m[0] for m in muts], dtype=np.int64)
        out[f"{name}/mut_row"] = np.array([m[1] for m in muts], dtype=np.int64)
        out[f"{name}/mut_col"] = np.array([m[2] for m in muts], dtype=np.int64)
        out[f"{name}/mut_val"] = np.array([limbs(m[3]) for m in muts], dtype=np.uint64)
        out[f"{name}/exp_row"] = np.array([m[4] for m in muts], dtype=np.int64)
        out[f"{name}/exp_exc"] = np.array([m[5] for m in muts])
        print(name, len(R), "rw", len(C), "copy-table rows", len(K), "keccak rows", len(muts), "vectors")
    np.savez_compressed(os.path.join(HERE, part + ".npz"), **out)
    print(f"{part}: {tot} corruptions, {nfail} failing")


def evm3_cases():
    evm2_cases("evm3")


def evm4_cases():
    evm2_cases("evm4")


def evm5_cases():
    evm2_cases("evm5")


def evm6_cases():
    evm2_cases("evm6")


def evm7_cases():
    evm2_cases("evm7")


def evm8_cases():
    evm2_cases("evm8")


def evm9_cases():
    evm2_cases("evm9")


def evm10_cases():
    evm2_cases("evm10")


def evm28_cases():
    """ErrorGasUintOverflow (error_gas_uint_overflow.py with instruction.memory_size / calc_mem_size64 / safe_mul / to_word_size)"""
    evm2_cases("evm28")


def evm27_cases():
    """ErrorOutOfGasPrecompile (execution/precompiles/error_oog_precompile.py)"""
    evm2_cases("evm27")


def evm26_cases():
    """ErrorOutOfGasCREATE (error_oog_create.py: the root-call branch prices the tx call data byte by byte)"""
    evm2_cases("evm26")


def evm25_cases():
    """ErrorOutOfGasSloadSstore (error_oog_sload_sstore.py; StepState.aux_data = the slot's committed value, an int)"""
    evm2_cases("evm25")


def evm24_cases():
    """CREATE / CREATE2 (create.py): pre-check failures, address collisions, creations without and with init code (new call
    context; StepState.aux_data = the init code's hash)"""
    evm2_cases("evm24")


def evm23_cases():
    """CALL / CALLCODE / DELEGATECALL / STATICCALL (callop.py): callee without code or failed pre-check (stays in the caller)
    and callee with code (new call context)"""
    evm2_cases("evm23")


def evm22_cases():
    """ErrorOutOfGasCall (error_oog_call.py + util/call_gadget.py)"""
    evm2_cases("evm22")


def evm21_cases():
    """RETURN / REVERT (return_revert.py): root, internal (return data copy + restored caller context) and CREATE endings"""
    evm2_cases("evm21")


def evm20_cases():
    """ErrorMaxCodeSizeExceeded / ErrorOutOfGasCodeStore (error_code_store.py) and ErrorInvalidCreationCode"""
    evm2_cases("evm20")


def evm19_cases():
    """EXP (exp-table lookups of the first and last step rows, base^2 through mul_add_words)"""
    evm2_cases("evm19")


def evm18_cases():
    """LOG0..LOG4 (tx-log rows, the data through a copy-table lookup whose destination address carries the log id),
    ErrorWriteProtection and BLOCKHASH (block-table lookups keyed on the block number)"""
    evm2_cases("evm18")


def evm17_cases():
    """SLOAD / SSTORE (storage reads and reversible writes keyed on the storage key, the refund rule) and CALLDATALOAD
    (32 tx-table or memory lookups behind the buffer reader)"""
    evm2_cases("evm17")


def evm16_cases():
    """ADDMOD / MULMOD / SDIV_SMOD / SAR (witnesses the gadgets derive from the stack words by 256- and 512-bit division)"""
    evm2_cases("evm16")


def evm15_cases():
    """CODECOPY / RETURNDATACOPY / EXTCODECOPY (copy-table lookups with Word and value ids) and ErrorOutOfGasMemoryCopy"""
    evm2_cases("evm15")


def evm14_cases():
    """BALANCE / EXTCODEHASH / EXTCODESIZE (access-list write with its reversion row, account reads) and
    ErrorOutOfGasAccountAccess"""
    evm2_cases("evm14")


def evm13_cases():
    """out-of-gas / out-of-bound error states: ErrorOutOfGasSHA3, ...StaticMemoryExpansion, ...DynamicMemoryExpansion, ...LOG,
    ...EXP and ErrorReturnDataOutOfBound"""
    evm2_cases("evm13")


def evm12_cases():
    """error states (ErrorStack, ErrorInvalidOpcode, ErrorOutOfGasConstant, ErrorInvalidJump: constrain_error_state in the
    root call and with the restore-to-caller branch) and SELFBALANCE"""
    evm2_cases("evm12")


# --------------------------------------------------------------------------- exp
def exp_cases():
    """Exp-circuit rows built by the reference's ExpCircuit.add_event / fill_dummy_events
    (evm_circuit/typing.py:868-994) and checked by the reference's verify_step under the loop of
    verify_exp_circuit (exp_circuit.py:88-97)."""
    from zkevm_specs import exp_circuit as xc
    from zkevm_specs.evm_circuit import ExpCircuit, ExpCircuitRow
    from zkevm_specs.util import ConstraintSystem, FQ, Word

    rng = random.Random(6)

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def ints(x):
        out = [n_of(x.q_usable), n_of(x.is_step), n_of(x.identifier), n_of(x.is_last)]
        for wd in (x.base, x.exponent, x.exponentiation, x.a, x.b, x.c, x.d, x.q):
            out += [n_of(wd.lo), n_of(wd.hi)]
        return out + [n_of(x.r)]

    def from_ints(v):
        f = [FQ(x) for x in v]
        ws = [W(v[4 + 2 * k], v[5 + 2 * k]) for k in range(8)]
        return ExpCircuitRow(f[0], f[1], f[2], f[3], *ws, f[20])

    def run(R):
        rows = [from_ints(v) for v in R]
        cs = ConstraintSystem()
        for i in range(len(rows)):
            try:
                cs.cond = None
                xc.verify_step(cs, [rows[i], rows[(i + 1) % len(rows)]])
            except Exception as e:  # noqa: BLE001
                return i, type(e).__name__
        return -1, ""

    scen = {
        "small": [(3, 13, 7), (2, 10, 14)],
        "big": [(rng.randrange(1 << 256), rng.randrange(2, 1 << 40), 21), ((1 << 256) - 1, 5, 28)],
        "pow2": [(2, 255, 35), (7, 2, 42), (0, 9, 49)],
    }
    out = {"names": np.array(list(scen.keys()))}
    tot = nfail = 0
    for name, events in scen.items():
        c = ExpCircuit(max_exp_steps=2)
        for b, e, ident in events:
            c.add_event(b, e, ident)
        c.max_exp_steps = (len(c.rows) + 6) // 7 + 1
        c.fill_dummy_events()
        R = [ints(x) for x in c.table()]
        assert run(R) == (-1, ""), (name, run(R))
        muts = [(-1, 0, 0, -1, "")]
        for k in range(120):
            i, col = rng.randrange(len(R)), rng.randrange(1, 21)
            old = R[i][col]
            v = (1 - old) if (old in (0, 1) and rng.random() < 0.5) else corrupt_value(rng, old)
            R2 = [list(x) for x in R]
            R2[i][col] = v
            fr_, ex_ = run(R2)
            muts.append((i, col, v, fr_, ex_))
            tot += 1
            nfail += fr_ >= 0
        out[f"{name}/rows"] = to_matrix(R)
        out[f"{name}/mut_row"] = np.array([m[0] for m in muts], dtype=np.int64)
        out[f"{name}/mut_col"] = np.array([m[1] for m in muts], dtype=np.int64)
        out[f"{name}/mut_val"] = np.array([limbs(m[2]) for m in muts], dtype=np.uint64)
        out[f"{name}/exp_row"] = np.array([m[3] for m in muts], dtype=np.int64)
        out[f"{name}/exp_exc"] = np.array([m[4] for m in muts])
        print(name, len(R), "rows", len(muts), "vectors")
    np.savez_compressed(os.path.join(HERE, "exp.npz"), **out)
    print(f"exp: {tot} corruptions, {nfail} failing")


# --------------------------------------------------------------------------- public-inputs circuit
PI_COLS = 28


def pi_row_ints(x):
    """pi_circuit.Row -> the 28 cells of include/zkcheck.h ZK_CIRCUIT_PI"""
    t, wd = x.tx_table, x.withdrawal_table
    addr = wd.address
    a_lo, a_hi = (n_of(addr.lo), n_of(addr.hi)) if hasattr(addr, "lo") else (n_of(addr), 0)
    return [n_of(x.q_bytes_last), n_of(x.q_tx_table), n_of(x.q_tx_calldata), n_of(x.q_tx_calldata_start),
            n_of(x.q_rpi_keccak_lookup), n_of(x.q_rpi_value_start), n_of(x.tx_id_inv), n_of(x.tx_value_lo_inv),
            n_of(x.tx_id_diff_inv), n_of(x.calldata_gas_cost), n_of(x.is_final), n_of(x.q_withdrawal_table),
            n_of(x.rpi_bytes), n_of(x.rpi_bytes_keccakrlc), n_of(x.rpi_value_lc), n_of(x.rpi_digest_word.lo),
            n_of(x.rpi_digest_word.hi), n_of(x.q_rpi_byte_enable), n_of(t.tx_id), n_of(t.tag), n_of(t.index),
            n_of(t.value.lo), n_of(t.value.hi), n_of(wd.id), n_of(wd.validator_id), a_lo, a_hi, n_of(wd.amount)]


def pi_reference_runner():
    """(run_rows, row_from, tables_from): evaluate the reference's check_row on cell vectors"""
    from zkevm_specs import pi_circuit as pc
    from zkevm_specs.util import FQ, Word, WordOrValue

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def row_from(v, kt):
        val = WordOrValue(FQ(v[21]))
        val.hi = FQ(v[22])
        f = [FQ(x) for x in v]
        return pc.Row(f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7], f[8], f[9], f[10], f[11], f[12], f[13], f[14],
                      W(v[15], v[16]), f[17], kt, pc.TxTableRow(f[18], f[19], f[20], val),
                      pc.WithdrawalTableRow(f[23], f[24], W(v[25], v[26]), f[27]))

    def tables_from(K, G):
        kt = pc.KeccakTable()
        kt.table = set((FQ(k[0]), FQ(k[1]), FQ(k[2]), W(k[3], k[4])) for k in K)
        gas = set(pc.TxCallDataGasCostAccRow(FQ(g[0]), FQ(g[1]), FQ(g[2])) for g in G)
        return kt, gas

    u16 = set(pc.FixedU16Row(FQ(i)) for i in range(1 << 16))

    def run_rows(R, K, G, circuit_len, which):
        """first failing row among `which` (ascending), as the loop of verify_circuit (pi_circuit.py:447-459)"""
        kt, gas = tables_from(K, G)
        n = len(R)
        for i in sorted(which):
            try:
                pc.check_row(row_from(R[i], kt), row_from(R[(i + 1) % n], kt), gas, u16, kt, circuit_len)
            except Exception as e:  # noqa: BLE001
                return i, type(e).__name__
        return -1, ""

    return run_rows


def pi_cases():
    """Public-inputs circuit: witnesses built by the reference's public_data2witness (pi_circuit.py:839-1073) from
    seeded random PublicData (the recipe of tests/test_public_inputs.py:66-128), checked by the reference's check_row
    under the loop of verify_circuit; negatives are single-cell corruptions of the witness, the keccak table and the
    calldata gas-cost table."""
    from zkevm_specs import pi_circuit as pc
    from zkevm_specs.util import U64, U160, U256

    rng = random.Random(12)
    run_rows = pi_reference_runner()

    def rand_block():
        r256 = lambda: U256(rng.randrange(1 << 256))  # noqa: E731
        r64 = lambda: U64(rng.randrange(1 << 64))  # noqa: E731
        return pc.Block(hash=r256(), parent_hash=r256(), uncle_hash=r256(), coinbase=U160(rng.randrange(1 << 160)),
                        state_root=r256(), tx_hash=r256(), receipt_hash=r256(), bloom=rng.randbytes(256), prev_randao=r256(),
                        number=r64(), gas_limit=r64(), gas_used=r64(), time=r64(), extra=bytes([]), mix_digest=r256(),
                        nonce=r64(), base_fee=U256(0), withdrawals_root=r256())

    def rand_tx(data):
        return pc.Transaction(nonce=U64(rng.randrange(1 << 64)), gas_price=U256(rng.randrange(1 << 256)),
                              gas=U64(rng.randrange(1 << 64)), from_addr=U160(rng.randrange(1 << 160)),
                              to_addr=U160(rng.randrange(1 << 160)), value=U256(rng.randrange(1 << 256)), data=data,
                              tx_sign_hash=U256(rng.randrange(1 << 256)))

    def calldata(n):
        return bytes(0 if rng.random() < 0.3 else rng.randrange(1, 256) for _ in range(n))

    scen = {
        # name: (MAX_TXS, MAX_CALLDATA_BYTES, MAX_WITHDRAWALS, calldata lengths of the txs, withdrawals)
        "basic": (2, 8, 2, [5], 2),
        "full": (3, 40, 3, [17, 0, 23], 3),
        "one_empty": (2, 16, 2, [0], 2),
    }
    out = {"names": np.array(list(scen.keys()))}
    tot = nfail = 0
    for name, (max_txs, max_cd, max_wd, lens, n_wd) in scen.items():
        pd = pc.PublicData(U64(rng.randrange(1, 128)), rand_block(), U256(rng.randrange(1 << 256)),
                           [U256(rng.randrange(1 << 256)) for _ in range(256)], [rand_tx(calldata(n)) for n in lens],
                           [pc.Withdrawal(id=k, validator_id=U64(rng.randrange(1 << 64)), address=U160(rng.randrange(1 << 160)),
                                          amount=U64(rng.randrange(1, 1 << 64))) for k in range(n_wd)])
        w = pc.public_data2witness(pd, max_txs, max_cd, max_wd)
        pc.verify_circuit(w, max_txs, max_cd, max_wd)  # the reference accepts its own witness (incl. copy constraints)
        w = pc.public_data2witness(pd, max_txs, max_cd, max_wd)  # verify_circuit consumed copy_constrains
        R = [pi_row_ints(x) for x in w.rows]
        K = sorted([n_of(k[0]), n_of(k[1]), n_of(k[2]), n_of(k[3].lo), n_of(k[3].hi)] for k in w.keccak_table.table)
        G = sorted([n_of(g.tx_id), n_of(g.is_final), n_of(g.gas_cost_acc)] for g in w.calldata_gas_cost_table)
        n = len(R)
        assert n == w.circuit_len
        assert run_rows(R, K, G, w.circuit_len, range(n)) == (-1, "")
        lookups = [i for i in range(n) if R[i][4] or R[i][1]]
        hot = 10 * max_txs + 1 + max_cd + max_wd + 2  # tx-table, calldata and withdrawal rows sit at the top
        muts = [(0, -1, 0, 0, -1, "")]
        for k in range(260):
            kind = 0 if k < 200 else (1 if k < 230 else 2)
            if kind == 0:
                i = rng.randrange(hot) if rng.random() < 0.75 else rng.randrange(n)
                if rng.random() < 0.05:
                    i = n - 1 - rng.randrange(3)
                col = rng.randrange(PI_COLS)
                old = R[i][col]
                v = (1 - old) if (old in (0, 1) and rng.random() < 0.5) else corrupt_value(rng, old)
                R2 = [list(x) for x in (R[(i - 1) % n], R[i])]
                R2[1][col] = v
                Rm = list(R)
                Rm[i] = R2[1]
                fr_, ex_ = run_rows(Rm, K, G, w.circuit_len, {(i - 1) % n, i})
            elif kind == 1:
                i, col = rng.randrange(len(K)), rng.randrange(5)
                v = corrupt_value(rng, K[i][col])
                K2 = [list(x) for x in K]
                K2[i][col] = v
                fr_, ex_ = run_rows(R, K2, G, w.circuit_len, lookups)
            else:
                i, col = rng.randrange(len(G)), rng.randrange(3)
                v = corrupt_value(rng, G[i][col])
                G2 = [list(x) for x in G]
                G2[i][col] = v
                fr_, ex_ = run_rows(R, K, G2, w.circuit_len, lookups)
            muts.append((kind, i, col, v, fr_, ex_))
            tot += 1
            nfail += fr_ >= 0
        out[f"{name}/rows"] = to_matrix(R)
        out[f"{name}/keccak"] = to_matrix(K)
        out[f"{name}/gas"] = to_matrix(G)
        import json
        b = pd.block
        out[f"{name}/public_data"] = np.array(json.dumps({
            "chain_id": int(pd.chain_id), "state_root_prev": int(pd.state_root_prev), "block_hashes": [int(h) for h in pd.block_hashes],
            "block": {k: (getattr(b, k).hex() if isinstance(getattr(b, k), bytes) else int(getattr(b, k)))
                      for k in ("hash", "parent_hash", "uncle_hash", "coinbase", "state_root", "tx_hash", "receipt_hash", "bloom",
                                "prev_randao", "number", "gas_limit", "gas_used", "time", "extra", "mix_digest", "nonce", "base_fee",
                                "withdrawals_root")},
            "txs": [{"nonce": int(t.nonce), "gas_price": int(t.gas_price), "gas": int(t.gas), "from_addr": int(t.from_addr),
                     "to_addr": int(t.to_addr), "value": int(t.value), "data": bytes(t.data).hex(), "tx_sign_hash": int(t.tx_sign_hash)}
                    for t in pd.txs],
            "withdrawals": [{"id": int(x.id), "validator_id": int(x.validator_id), "address": int(x.address), "amount": int(x.amount)}
                            for x in pd.withdrawals]}))
        out[f"{name}/circuit_len"] = np.array([w.circuit_len], dtype=np.int64)
        out[f"{name}/params"] = np.array([max_txs, max_cd, max_wd], dtype=np.int64)
        out[f"{name}/mut_kind"] = np.array([m[0] for m in muts], dtype=np.int64)
        out[f"{name}/mut_row"] = np.array([m[1] for m in muts], dtype=np.int64)
        out[f"{name}/mut_col"] = np.array([m[2] for m in muts], dtype=np.int64)
        out[f"{name}/mut_val"] = np.array([limbs(m[3]) for m in muts], dtype=np.uint64)
        out[f"{name}/exp_row"] = np.array([m[4] for m in muts], dtype=np.int64)
        out[f"{name}/exp_exc"] = np.array([m[5] for m in muts])
        print(name, n, "rows", len(muts), "vectors", "failing", sum(1 for m in muts if m[4] >= 0))
    for name in scen:  # one file per case: each stays under 1 MB (golden_util.load_pi merges them)
        np.savez_compressed(os.path.join(HERE, f"pi_{name}.npz"),
                            **{k[len(name) + 1:]: v for k, v in out.items() if k.startswith(name + "/")})
    print(f"pi: {tot} corruptions, {nfail} failing")


# --------------------------------------------------------------------------- tx circuit (Fr parts)
def tx_cases():
    """The reference's tx_circuit.verify_circuit (tx_circuit.py:253-289) run UNMODIFIED on witnesses
    whose ECDSA chip is a stand-in: eth_keys (secp256k1) is a third-party dependency that is absent
    here, so the chips are built directly from random public-key bytes and `ECDSAVerifyChip.verify`
    is replaced by a per-chip flag.  Everything the path covers — the public-key RLC, the
    keccak-table membership, address / msg-hash equalities, the copy constraints — is the
    reference's own code.  Corruptions: any of the 14 cells of a tx (as the reference objects they
    come from), the Word/value type of the CallerAddress row, the ECDSA flag, keccak-table cells."""
    from zkevm_specs import tx_circuit as tc
    from zkevm_specs.util import FQ, Word, WordOrValue
    from eth_utils import keccak

    r = FQ(0x0123456789ABCDEF0123456789ABCDEF0123456789ABCDEF0123456789ABCDEF % P)
    rng = random.Random(19)
    MAX_TXS = 6

    class StubECDSA:
        def __init__(self, x_le, y_le, msg_le, ok=True):
            self.pub_key_x_bytes, self.pub_key_y_bytes, self.msg_hash_bytes, self.ok = x_le, y_le, msg_le, ok

        def verify(self, assert_msg):
            assert self.ok, f"{assert_msg}: ecdsa_verify failed"

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def wbytes(lo, hi):  # the 32 bytes whose Word is (lo, hi); None if not representable as bytes
        if lo >= 1 << 128 or hi >= 1 << 128:
            return None
        return lo.to_bytes(16, "little") + hi.to_bytes(16, "little")

    def base_cells():
        cells, flags, pks = [], [], []
        for i in range(MAX_TXS):
            if i >= 4:  # padding txs: all zero (tx_circuit.py:273-275)
                cells.append([0] * 14); flags.append(0); pks.append(None)
                continue
            pk = bytes(rng.randrange(256) for _ in range(64))  # x_be + y_be
            x_le, y_le = bytes(reversed(pk[:32])), bytes(reversed(pk[32:]))
            h = keccak(pk)
            addr = int.from_bytes(h[-20:], "big")
            msg = bytes(rng.randrange(256) for _ in range(32))  # tx sign hash, big-endian
            msg_le = bytes(reversed(msg))
            mw = Word(int.from_bytes(msg, "big"))
            c = [addr, int.from_bytes(x_le[:16], "little"), int.from_bytes(x_le[16:], "little"),
                 int.from_bytes(y_le[:16], "little"), int.from_bytes(y_le[16:], "little"),
                 int.from_bytes(h[:16], "little"), int.from_bytes(h[16:], "little"), n_of(mw.lo), n_of(mw.hi),
                 int.from_bytes(msg_le[:16], "little"), int.from_bytes(msg_le[16:], "little"), addr, n_of(mw.lo), n_of(mw.hi)]
            assert (c[9], c[10]) == (c[7], c[8])
            cells.append(c); flags.append(0); pks.append(pk)
        return cells, flags, pks

    def keccak_rows(pks):
        kt = tc.KeccakTable()
        for pk in pks:
            if pk is not None:
                kt.add(pk, r)
        return sorted([[n_of(a), n_of(b), n_of(l), n_of(o.lo), n_of(o.hi)] for a, b, l, o in kt.table])

    def run(cells, flags, K):
        kt = tc.KeccakTable()
        kt.table = set((FQ(v[0]), FQ(v[1]), FQ(v[2]), W(v[3], v[4])) for v in K)
        rows, chips = [], []
        for c, f in zip(cells, flags):
            xb, yb, hb, mb = wbytes(c[1], c[2]), wbytes(c[3], c[4]), wbytes(c[5], c[6]), wbytes(c[9], c[10])
            if None in (xb, yb, hb, mb):
                return None  # not representable as `bytes` objects: no reference verdict
            chips.append(tc.SignVerifyChip(hb, FQ(c[0]), W(c[7], c[8]), StubECDSA(xb, yb, mb, ok=not (f & 2))))
            for tag in range(1, 13):  # TxContextFieldTag Nonce=1 .. TxSignHash=12 (CallerAddress=4)
                if tag == 4:
                    v = W(c[11], 0) if f & 1 else FQ(c[11])
                elif tag == 12:
                    v = W(c[12], c[13])
                else:
                    v = FQ(0)
                rows.append(tc.Row(FQ(len(chips)), FQ(tag), FQ(0), v))
        # verify_circuit(witness, m, ..) checks tx 0..m-1 and stops at the first failing assert (not
        # every assert carries the tx_index in its message): grow m to find the failing tx
        for m in range(1, MAX_TXS + 1):
            try:
                tc.verify_circuit(tc.Witness(rows, kt, chips), m, 0, r)
            except Exception as e:  # noqa: BLE001
                return m - 1, type(e).__name__
        return -1, ""

    import re
    cells, flags, pks = base_cells()
    K = keccak_rows(pks)
    assert run(cells, flags, K) == (-1, "")
    muts = [(-1, 0, 0, 0, -1, "")]
    tot = nfail = 0
    for k in range(420):
        which = rng.choice([0, 0, 0, 0, 1, 2, 3, 3])
        c2, f2, K2 = [list(x) for x in cells], list(flags), [list(x) for x in K]
        if which == 0:
            i, col = rng.randrange(MAX_TXS), rng.randrange(14)
            v = corrupt_value(rng, cells[i][col]); c2[i][col] = v
        elif which == 1:
            i, col, v = rng.randrange(MAX_TXS), 100, 0
            f2[i] ^= 1
        elif which == 2:
            i, col, v = rng.randrange(MAX_TXS), 101, 0
            f2[i] ^= 2
        else:
            i, col = rng.randrange(len(K)), rng.randrange(5)
            v = corrupt_value(rng, K[i][col]); K2[i][col] = v
        out = run(c2, f2, K2)
        if out is None:
            continue
        muts.append((which, i, col, v, out[0], out[1]))
        tot += 1
        nfail += out[0] >= 0
    out = {"rows": to_matrix(cells), "flags": np.array(flags, dtype=np.uint8), "keccak": to_matrix(K),
           "r": np.array(limbs(r.n), dtype=np.uint64),
           "mut_kind": np.array([m[0] for m in muts], dtype=np.int64), "mut_row": np.array([m[1] for m in muts], dtype=np.int64),
           "mut_col": np.array([m[2] for m in muts], dtype=np.int64), "mut_val": np.array([limbs(m[3]) for m in muts], dtype=np.uint64),
           "exp_row": np.array([m[4] for m in muts], dtype=np.int64), "exp_exc": np.array([m[5] for m in muts])}
    np.savez_compressed(os.path.join(HERE, "tx.npz"), **out)
    print(f"tx: {tot} corruptions, {nfail} failing")


# --------------------------------------------------------------------------- sig circuit (Fr parts)
def sig_cases():
    """sig_circuit.verify_circuit (sig_circuit.py:113-123) run UNMODIFIED on rows whose ECDSA chip
    is a stand-in (eth_keys absent): chips carry random public-key / signature bytes and a verdict
    flag returned by verify().  Corruptions: any of the 21 cells (as the reference attributes they
    come from), the verdict flag, keccak-table cells."""
    from zkevm_specs import sig_circuit as sc
    from zkevm_specs.util import FQ, Word, KeccakTable
    from eth_utils import keccak

    r = FQ(0x0FEDCBA9876543210FEDCBA9876543210FEDCBA9876543210FEDCBA987654321 % P)
    rng = random.Random(23)
    N = 5

    class LE:
        def __init__(self, v):
            self.le_bytes = v.to_bytes(32, "little")

    class StubECDSA:
        def __init__(self, x_le, y_le, msg_b, v, rr, ss, ok):
            self.pub_key_x_bytes, self.pub_key_y_bytes, self.msg_hash_bytes = x_le, y_le, msg_b
            self.sig_v, self.sig_r, self.sig_s, self.ok = LE(v), LE(rr), LE(ss), ok

        def verify(self):
            return self.ok

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def wbytes(lo, hi):
        if lo >= 1 << 128 or hi >= 1 << 128:
            return None
        return lo.to_bytes(16, "little") + hi.to_bytes(16, "little")

    def halves(b):
        return [int.from_bytes(b[:16], "little"), int.from_bytes(b[16:], "little")]

    cells, flags, pks = [], [], []
    for i in range(N):
        pk = bytes(rng.randrange(256) for _ in range(64))
        x_le, y_le = bytes(reversed(pk[:32])), bytes(reversed(pk[32:]))
        h = keccak(pk)
        addr = int.from_bytes(h[-20:], "big")
        msg_b = bytes(rng.randrange(256) for _ in range(32))  # ECDSAVerifyChip.msg_hash_bytes (util/ec.py:88)
        mw = Word(msg_b)
        rr, ss = rng.getrandbits(256), rng.getrandbits(256)
        ok = i != 3  # one row of an invalid signature with is_valid = False
        cells.append([i & 1, addr, *halves(x_le), *halves(y_le), *halves(h), n_of(mw.lo), n_of(mw.hi), *halves(msg_b),
                      int(ok), rr & ((1 << 128) - 1), rr >> 128, ss & ((1 << 128) - 1), ss >> 128,
                      rr & ((1 << 128) - 1), rr >> 128, ss & ((1 << 128) - 1), ss >> 128])
        flags.append(int(ok) << 1)
        pks.append(pk)
    kt0 = KeccakTable()
    for pk in pks:
        kt0.add(pk, r)
    K = sorted([[n_of(a), n_of(b), n_of(l), n_of(o.lo), n_of(o.hi)] for a, b, l, o in kt0.table])

    def run(cells, flags, K):
        kt = KeccakTable()
        kt.table = set((FQ(v[0]), FQ(v[1]), FQ(v[2]), W(v[3], v[4])) for v in K)
        rows = []
        for c, f in zip(cells, flags):
            xb, yb, hb, mb = wbytes(c[2], c[3]), wbytes(c[4], c[5]), wbytes(c[6], c[7]), wbytes(c[10], c[11])
            if None in (xb, yb, hb, mb) or max(c[17:21]) >= 1 << 128:
                return None
            chip = StubECDSA(xb, yb, mb, 0, c[17] + (c[18] << 128), c[19] + (c[20] << 128), bool(f & 2))
            row = sc.Row(hb, FQ(c[1]), W(c[8], c[9]), chip, c[12])
            row.sig_v, row.sig_r, row.sig_s = FQ(c[0]), W(c[13], c[14]), W(c[15], c[16])
            rows.append(row)
        for m in range(1, len(rows) + 1):
            try:
                sc.verify_circuit(sc.Witness(rows[:m], kt), r)
            except Exception as e:  # noqa: BLE001
                return m - 1, type(e).__name__
        return -1, ""

    assert run(cells, flags, K) == (-1, ""), run(cells, flags, K)
    muts = [(-1, 0, 0, 0, -1, "")]
    tot = nfail = 0
    for k in range(420):
        which = rng.choice([0, 0, 0, 0, 0, 2, 3, 3])
        c2, f2, K2 = [list(x) for x in cells], list(flags), [list(x) for x in K]
        if which == 0:
            i, col = rng.randrange(N), rng.randrange(21)
            v = corrupt_value(rng, cells[i][col]); c2[i][col] = v
        elif which == 2:
            i, col, v = rng.randrange(N), 101, 0
            f2[i] ^= 2
        else:
            i, col = rng.randrange(len(K)), rng.randrange(5)
            v = corrupt_value(rng, K[i][col]); K2[i][col] = v
        out = run(c2, f2, K2)
        if out is None:
            continue
        muts.append((which, i, col, v, out[0], out[1]))
        tot += 1
        nfail += out[0] >= 0
    out = {"rows": to_matrix(cells), "flags": np.array(flags, dtype=np.uint8), "keccak": to_matrix(K),
           "r": np.array(limbs(r.n), dtype=np.uint64),
           "mut_kind": np.array([m[0] for m in muts], dtype=np.int64), "mut_row": np.array([m[1] for m in muts], dtype=np.int64),
           "mut_col": np.array([m[2] for m in muts], dtype=np.int64), "mut_val": np.array([limbs(m[3]) for m in muts], dtype=np.uint64),
           "exp_row": np.array([m[4] for m in muts], dtype=np.int64), "exp_exc": np.array([m[5] for m in muts])}
    np.savez_compressed(os.path.join(HERE, "sig.npz"), **out)
    print(f"sig: {tot} corruptions, {nfail} failing")



# --------------------------------------------------------------------------- evm11: BeginTx / EndTx / EndBlock
def evm11_cases():
    """BeginTx, EndTx and EndBlock steps built like the reference's tests (tests/evm/test_begin_tx.py:278-391,
    test_end_tx.py:93-170, test_end_block.py:38-155), verified by the reference's verify_step with the first / last
    step flags of verify_steps (main.py:14-44); corruptions of step cells, rw rows (all 14 cells + both type flags),
    tx / block / withdrawal table cells (+ value type flags), copy- and keccak-table cells, duplicated rw rows."""
    import rlp
    from zkevm_specs.evm_circuit import (AccessTuple, Account, AccountFieldTag, Block, BlockTableRow, Bytecode,
                                         BytecodeTableRow, CallContextFieldTag, CopyCircuit, CopyDataTypeTag, CopyTableRow,
                                         ExecutionState, KeccakTableRow, RW, RWDictionary, RWTableRow, StepState, Tables,
                                         Target, Transaction, TxReceiptFieldTag, TxTableRow, Withdrawal, WithdrawalTableRow)
    from zkevm_specs.evm_circuit.instruction import Instruction
    from zkevm_specs.evm_circuit.main import DUMMY_STEP_STATE, verify_step
    from zkevm_specs.evm_circuit.typing import KeccakCircuit
    from zkevm_specs.util import EMPTY_CODE_HASH, FQ, MAX_REFUND_QUOTIENT_OF_GAS_USED, U64, Word, WordOrValue
    from zkevm_specs.util.hash import keccak256

    rng = random.Random(23)
    r_keccak = FQ(0x0BADC0FFEE0DDF00D0BADC0FFEE0DDF00D0BADC0FFEE0DDF00D0BADC0FFEE % P)

    def W(lo, hi):
        return Word((FQ(lo), FQ(hi)), check=False)

    def wov(lo, hi, is_word):
        return WordOrValue(W(lo, hi)) if is_word else WordOrValue(FQ(lo))

    # ---- scenario builders: (steps, bytecode rows, rw rows, copy-table rows, keccak rows, tx rows, block rows,
    #      withdrawal rows, begin_with_first_step, end_with_last_step)
    def end_tx_case(tx, gas_left, refund, is_last_tx, cum_gas):
        block = Block()
        eff = min(refund, (tx.gas - gas_left) // MAX_REFUND_QUOTIENT_OF_GAS_USED)
        caller_prev = int(1e18) - (tx.value + tx.gas * tx.gas_price)
        caller = caller_prev + (gas_left + eff) * tx.gas_price
        coinbase = (tx.gas - gas_left) * (tx.gas_price - block.base_fee)
        d = (RWDictionary(17)
             .call_context_read(1, CallContextFieldTag.TxId, tx.id)
             .call_context_read(1, CallContextFieldTag.IsPersistent, 1)
             .tx_refund_read(tx.id, refund)
             .account_write(tx.caller_address, AccountFieldTag.Balance, Word(caller), Word(caller_prev))
             .account_write(block.coinbase, AccountFieldTag.Balance, Word(coinbase), Word(0))
             .tx_receipt_write(tx.id, TxReceiptFieldTag.PostStateOrStatus, 1 - tx.invalid_tx)
             .tx_receipt_write(tx.id, TxReceiptFieldTag.LogLength, 0))
        first = tx.id == 1
        if first:
            d.tx_receipt_write(tx.id, TxReceiptFieldTag.CumulativeGasUsed, tx.gas - gas_left)
        else:
            d.tx_receipt_read(tx.id - 1, TxReceiptFieldTag.CumulativeGasUsed, cum_gas)
            d.tx_receipt_write(tx.id, TxReceiptFieldTag.CumulativeGasUsed, tx.gas - gas_left + cum_gas)
        if not is_last_tx:
            d.call_context_read(27 - first, CallContextFieldTag.TxId, tx.id + 1)
        steps = [StepState(ExecutionState.EndTx, rw_counter=17, call_id=1, is_root=True, is_create=False,
                           code_hash=Word(EMPTY_CODE_HASH), program_counter=0, stack_pointer=1024, gas_left=gas_left,
                           reversible_write_counter=2),
                 StepState(ExecutionState.EndBlock if is_last_tx else ExecutionState.BeginTx,
                           rw_counter=27 - first - is_last_tx, call_id=1 if is_last_tx else 0)]
        return steps, [], list(d.rws), [], [], list(tx.table_assignments()), block.table_assignments(), [], False, False

    def end_block_case(is_last_step, empty_block, max_txs, max_wds, cum_gas):
        MAX_RWS = 32
        tx = Transaction()
        wd1, wd2 = Withdrawal(0, 99, 3, int(1e9)), Withdrawal(1, 999, 4, int(1.4e9))
        rws, rwc = [], 1
        if not empty_block:
            rws += [RWTableRow(FQ(i + 1), *2 * [FQ(0)]) for i in range(21)]
            rwc += 21
            if is_last_step:
                rws.append(RWTableRow(FQ(22), FQ(RW.Read), key0=FQ(Target.CallContext), id=FQ(1), address=FQ(3),
                                      field_tag=FQ(CallContextFieldTag.TxId), value=WordOrValue(FQ(tx.id))))
                rws.append(RWTableRow(FQ(23), FQ(RW.Read), key0=FQ(Target.TxReceipt), id=FQ(tx.id), address=FQ(0),
                                      field_tag=FQ(TxReceiptFieldTag.CumulativeGasUsed), storage_key=Word(0),
                                      value=WordOrValue(FQ(cum_gas))))
            rws.append(RWTableRow(FQ(22 + is_last_step * 2), FQ(RW.Write), key0=FQ(Target.Account), address=FQ(wd1.address),
                                  field_tag=FQ(AccountFieldTag.Balance), value=Word(int(5e18)), value_prev=Word(int(4e18))))
            rws.append(RWTableRow(FQ(23 + is_last_step * 2), FQ(RW.Write), key0=FQ(Target.Account), address=FQ(wd2.address),
                                  field_tag=FQ(AccountFieldTag.Balance), value=Word(int(5.5e18)), value_prev=Word(int(4.1e18))))
        pad = [RWTableRow(FQ(i + 1), FQ(0), FQ(Target.Start)) for i in range(MAX_RWS - len(rws))]
        n_tx = 0 if empty_block else 1
        txs = []
        for i in range(n_tx, max_txs):
            txs += Transaction.padding(id=i + 1).table_fixed()
        if not empty_block:
            txs = list(tx.table_assignments())
        n_wd = 0 if empty_block else 2
        wds = []
        for i in range(n_wd, max_wds):
            wds += Withdrawal.padding(id=i).table_assignments()
        if not empty_block:
            wds += list(wd1.table_assignments()) + list(wd2.table_assignments())
        steps = [StepState(ExecutionState.EndBlock, rw_counter=rwc, call_id=1),
                 StepState(ExecutionState.EndBlock, rw_counter=rwc, call_id=1)]
        return steps, [], pad + rws, [], [], txs, Block().table_assignments(), wds, False, is_last_step

    RETURN_CODE, REVERT_CODE = Bytecode().return_(0, 0), Bytecode().revert(0, 0)

    def initcode(is_return):
        b = Bytecode().push(0x2222222222222222222222222222222222222222222222222222222222222222, n_bytes=32).push(0, n_bytes=1).mstore()
        return b.return_() if is_return else b.revert()

    def begin_tx_case(tx, callee, is_success):
        block = Block()
        valid = 1 - tx.invalid_tx
        create = tx.callee_address is None
        rev_end = 24
        caller_prev = int(1e20)
        caller = caller_prev - (tx.value + tx.gas * tx.gas_price) if valid else caller_prev
        callee_bal = callee.balance + tx.value if valid else callee.balance
        calldata_hash = Word(int.from_bytes(keccak256(tx.call_data), "big"))
        code_hash = calldata_hash if create else Word(callee.code_hash())
        caddr = int.from_bytes(keccak256(rlp.encode([tx.caller_address.to_bytes(20, "big"), tx.nonce]))[-20:], "big")
        callee_address = caddr if create else tx.callee_address
        d = (RWDictionary(1)
             .call_context_read(1, CallContextFieldTag.TxId, tx.id)
             .call_context_read(1, CallContextFieldTag.RwCounterEndOfReversion, 0 if is_success else rev_end)
             .call_context_read(1, CallContextFieldTag.IsPersistent, is_success)
             .call_context_read(1, CallContextFieldTag.IsSuccess, is_success)
             .account_write(tx.caller_address, AccountFieldTag.Nonce, valid, 0)
             .tx_access_list_account_write(tx.id, block.coinbase, True, False)
             .tx_access_list_account_write(tx.id, tx.caller_address, True, False)
             .tx_access_list_account_write(tx.id, callee_address, True, False)
             .account_write(tx.caller_address, AccountFieldTag.Balance, Word(caller), Word(caller_prev),
                            rw_counter_of_reversion=None if is_success else rev_end)
             .account_write(callee_address, AccountFieldTag.Balance, Word(callee_bal), Word(callee.balance),
                            rw_counter_of_reversion=None if is_success else rev_end - 1))
        with_calldata = create and len(tx.call_data) > 0
        is_contract = not create and callee.code_hash() != EMPTY_CODE_HASH
        copy_rows, kec_rows = CopyCircuit().rows, KeccakCircuit().rows
        if not create:
            d.account_read(tx.callee_address, AccountFieldTag.CodeHash, code_hash)
        elif len(tx.call_data) > 0:
            src = dict((i, tx.call_data[i]) for i in range(len(tx.call_data)))
            c1 = CopyCircuit().copy(r_keccak, d, 1, CopyDataTypeTag.TxCalldata, 1, CopyDataTypeTag.RlcAcc, FQ.zero(),
                                    len(tx.call_data), FQ.zero(), len(tx.call_data), src)
            bc = Bytecode(tx.call_data)
            src2 = dict((i, (bc.code[i], bc.is_code[i])) for i in range(len(bc.code)))
            c2 = CopyCircuit().copy(r_keccak, d, 1, CopyDataTypeTag.TxCalldata, calldata_hash, CopyDataTypeTag.Bytecode,
                                    FQ.zero(), len(tx.call_data), FQ.zero(), len(tx.call_data), src2)
            copy_rows = c1.rows + c2.rows
            kec_rows = KeccakCircuit().add(tx.call_data, r_keccak).rows
        if (with_calldata or is_contract) and valid == 1:
            (d.call_context_read(1, CallContextFieldTag.Depth, 1)
              .call_context_read(1, CallContextFieldTag.CallerAddress, Word(tx.caller_address))
              .call_context_read(1, CallContextFieldTag.CalleeAddress, Word(callee_address))
              .call_context_read(1, CallContextFieldTag.CallDataOffset, 0)
              .call_context_read(1, CallContextFieldTag.CallDataLength, len(tx.call_data))
              .call_context_read(1, CallContextFieldTag.Value, Word(tx.value))
              .call_context_read(1, CallContextFieldTag.IsStatic, False)
              .call_context_read(1, CallContextFieldTag.LastCalleeId, 0)
              .call_context_read(1, CallContextFieldTag.LastCalleeReturnDataOffset, 0)
              .call_context_read(1, CallContextFieldTag.LastCalleeReturnDataLength, 0)
              .call_context_read(1, CallContextFieldTag.IsRoot, True)
              .call_context_read(1, CallContextFieldTag.IsCreate, create)
              .call_context_read(1, CallContextFieldTag.CodeHash, code_hash))
        t = Tables(block_table=set(), tx_table=set(), withdrawal_table=set(), bytecode_table=set(), rw_table=set(),
                   copy_circuit=copy_rows, keccak_table=kec_rows)
        steps = [StepState(ExecutionState.BeginTx, rw_counter=1),
                 StepState(ExecutionState.EndTx if callee.code_hash() == EMPTY_CODE_HASH or valid == 0 else ExecutionState.PUSH,
                           rw_counter=d.rw_counter, call_id=1, is_root=True, is_create=create, code_hash=code_hash,
                           program_counter=0, stack_pointer=1024, gas_left=0, reversible_write_counter=2)]
        return (steps, list(callee.code.table_assignments()), list(d.rws), list(t.copy_table), list(t.keccak_table),
                list(tx.table_assignments()), block.table_assignments(), [], True, False)

    CALLEE = 0xFF
    EOA, RET, REV = Account(address=CALLEE), Account(address=CALLEE, code=RETURN_CODE), Account(address=CALLEE, code=REVERT_CODE)
    scenarios = {
        "endtx_refund": end_tx_case(Transaction(id=1, caller_address=0xFE, callee_address=CALLEE, gas=27000, gas_price=int(2e9)), 994, 4800, False, 0),
        "endtx_capped": end_tx_case(Transaction(id=2, caller_address=0xFE, callee_address=CALLEE, gas=65000, gas_price=int(2e9)), 3952, 38400, False, 100),
        "endtx_last": end_tx_case(Transaction(id=3, caller_address=0xFE, callee_address=CALLEE, gas=21000, gas_price=int(2e9)), 0, 0, True, 20000),
        "endtx_invalid": end_tx_case(Transaction(id=1, caller_address=0xFE, callee_address=CALLEE, gas=60000, gas_price=int(2e9), invalid_tx=1), 60000, 0, False, 0),
        "endtx_last_invalid": end_tx_case(Transaction(id=2, caller_address=0xFE, callee_address=CALLEE, gas=65000, gas_price=int(2e9), invalid_tx=1), 65000, 0, True, 21000),
        "endblock_mid": end_block_case(False, False, 2, 5, 0),
        "endblock_last": end_block_case(True, False, 2, 5, 0),
        "endblock_last_full": end_block_case(True, False, 1, 2, 0),
        "endblock_empty": end_block_case(True, True, 1, 5, 0),
        "endblock_gas_ok": end_block_case(True, False, 1, 5, int(15e6)),
        "endblock_gas_over": end_block_case(True, False, 1, 2, int(15e6) + 1),
        "begintx_eoa": begin_tx_case(Transaction(caller_address=0xFE, callee_address=CALLEE, value=int(1e18)), EOA, True),
        "begintx_contract": begin_tx_case(Transaction(caller_address=0xFE, callee_address=CALLEE, value=int(1e18)), RET, True),
        "begintx_revert": begin_tx_case(Transaction(caller_address=0xFE, callee_address=CALLEE, value=int(1e18)), REV, False),
        "begintx_calldata": begin_tx_case(Transaction(caller_address=0xFE, callee_address=CALLEE, gas=21080, call_data=bytes([1, 2, 3, 4, 0, 0, 0, 0])), RET, True),
        "begintx_bad_nonce": begin_tx_case(Transaction(caller_address=0xFE, callee_address=CALLEE, value=int(1e18), nonce=U64(100), invalid_tx=1), EOA, True),
        "begintx_poor": begin_tx_case(Transaction(caller_address=0xFE, callee_address=CALLEE, gas=21080, value=int(1e21), invalid_tx=1), REV, True),
        "begintx_accesslist": begin_tx_case(Transaction(caller_address=0xFE, callee_address=CALLEE, gas=21080 + 2400 + 1900 * 2, value=int(1e17),
                                                        access_list=[AccessTuple(address=0xFE, storage_keys=[5, 6])]), EOA, True),
        "begintx_low_gas": begin_tx_case(Transaction(caller_address=0xFE, callee_address=CALLEE, gas=21080, value=int(1e17), invalid_tx=1,
                                                     access_list=[AccessTuple(address=0xFE, storage_keys=[5, 6])]), EOA, True),
        "begintx_create_empty": begin_tx_case(Transaction(caller_address=0xFE, callee_address=None, gas=53000, value=1), EOA, True),
        "begintx_create_code": begin_tx_case(Transaction(caller_address=0xFE, callee_address=None, gas=53584, value=1, call_data=bytes(initcode(True).code)), EOA, True),
        "begintx_create_revert": begin_tx_case(Transaction(caller_address=0xFE, callee_address=None, gas=53584, value=1, call_data=bytes(initcode(False).code)), EOA, True),
    }

    def step_ints(s):
        return [int(s.execution_state), n_of(s.rw_counter), n_of(s.call_id), int(s.is_root), int(s.is_create),
                n_of(s.code_hash.lo), n_of(s.code_hash.hi), n_of(s.program_counter), n_of(s.stack_pointer),
                n_of(s.gas_left), n_of(s.memory_word_size), n_of(s.reversible_write_counter), n_of(s.log_id)]

    def step_from(v):
        s = StepState(ExecutionState(v[0]), rw_counter=0)
        s.rw_counter, s.call_id, s.is_root, s.is_create = FQ(v[1]), FQ(v[2]), v[3], v[4]
        s.code_hash = W(v[5], v[6])
        s.program_counter, s.stack_pointer, s.gas_left = FQ(v[7]), FQ(v[8]), FQ(v[9])
        s.memory_word_size, s.reversible_write_counter, s.log_id = FQ(v[10]), FQ(v[11]), FQ(v[12])
        return s

    bc_ints = lambda x: [n_of(x.bytecode_hash.lo), n_of(x.bytecode_hash.hi), n_of(x.field_tag), n_of(x.index), n_of(x.is_code), n_of(x.value)]  # noqa: E731
    rw_ints = lambda x: [n_of(x.rw_counter), n_of(x.rw), n_of(x.key0), n_of(x.id), n_of(x.address), n_of(x.field_tag),  # noqa: E731
                         n_of(x.storage_key.lo), n_of(x.storage_key.hi), n_of(x.value.lo), n_of(x.value.hi),
                         n_of(x.value_prev.lo), n_of(x.value_prev.hi), n_of(x.aux0.lo), n_of(x.aux0.hi)]
    copy_ints = lambda x: [n_of(x.is_first), n_of(x.src_id.lo), n_of(x.src_id.hi), n_of(x.src_tag), n_of(x.dst_id.lo), n_of(x.dst_id.hi),  # noqa: E731
                           n_of(x.dst_tag), n_of(x.src_addr), n_of(x.src_addr_end), n_of(x.dst_addr), n_of(x.length), n_of(x.rlc_acc),
                           n_of(x.rw_counter), n_of(x.rwc_inc)]
    kec_ints = lambda x: [n_of(x.state_tag), n_of(x.input_rlc), n_of(x.input_len), n_of(x.output.lo), n_of(x.output.hi)]  # noqa: E731
    tx_ints = lambda x: [n_of(x.tx_id), n_of(x.field_tag), n_of(x.call_data_index_or_zero), n_of(x.value.lo), n_of(x.value.hi)]  # noqa: E731
    blk_ints = lambda x: [n_of(x.field_tag), n_of(x.block_number_or_zero), n_of(x.value.lo), n_of(x.value.hi)]  # noqa: E731
    wd_ints = lambda x: [n_of(x.id), n_of(x.validator_id), n_of(x.address), n_of(x.amount)]  # noqa: E731

    def run(S, B, R, RF, C, CF, K, T, TF, BL, BF, WD, first, last):
        steps = [step_from(v) for v in S]
        t = Tables(block_table=set(BlockTableRow(FQ(v[0]), FQ(v[1]), wov(v[2], v[3], f)) for v, f in zip(BL, BF)),
                   tx_table=set(TxTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), wov(v[3], v[4], f)) for v, f in zip(T, TF)),
                   withdrawal_table=set(WithdrawalTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), FQ(v[3])) for v in WD),
                   bytecode_table=set(BytecodeTableRow(W(v[0], v[1]), FQ(v[2]), FQ(v[3]), FQ(v[4]), FQ(v[5])) for v in B),
                   rw_table=set(RWTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), FQ(v[3]), FQ(v[4]), FQ(v[5]), W(v[6], v[7]),
                                           wov(v[8], v[9], f & 1), wov(v[10], v[11], (f >> 1) & 1), W(v[12], v[13]))
                                for v, f in zip(R, RF)))
        t.copy_table = set(CopyTableRow(FQ(v[0]), wov(v[1], v[2], f & 1), FQ(v[3]), wov(v[4], v[5], (f >> 1) & 1), FQ(v[6]),
                                        FQ(v[7]), FQ(v[8]), FQ(v[9]), FQ(v[10]), FQ(v[11]), FQ(v[12]), FQ(v[13])) for v, f in zip(C, CF))
        t.keccak_table = set(KeccakTableRow(FQ(v[0]), FQ(v[1]), FQ(v[2]), W(v[3], v[4])) for v in K)
        if last:
            steps = steps + [DUMMY_STEP_STATE]
        for idx, (cur, nxt) in enumerate(zip(steps, steps[1:])):
            try:
                verify_step(Instruction(tables=t, curr=cur, next=nxt, is_first_step=first and idx == 0,
                                        is_last_step=last and idx == len(steps) - 2))
            except Exception as e:  # noqa: BLE001
                return idx, type(e).__name__
        return -1, ""

    out = {"names": np.array(list(scenarios.keys()))}
    tot = nfail = 0
    for name, (steps, bcs, rws, cps, kcs, txs, blks, wds, first, last) in scenarios.items():
        S, B, R = [step_ints(x) for x in steps], [bc_ints(x) for x in bcs], [rw_ints(x) for x in rws]
        RF = [int(getattr(x.value, 'is_word', True)) | (int(getattr(x.value_prev, 'is_word', True)) << 1) for x in rws]
        C, K = [copy_ints(x) for x in cps], [kec_ints(x) for x in kcs]
        CF = [int(x.src_id.is_word) | (int(x.dst_id.is_word) << 1) for x in cps]
        T, BL, WD = [tx_ints(x) for x in txs], [blk_ints(x) for x in blks], [wd_ints(x) for x in wds]
        TF, BF = [int(x.value.is_word) for x in txs], [int(x.value.is_word) for x in blks]
        base = run(S, B, R, RF, C, CF, K, T, TF, BL, BF, WD, first, last)
        if name == "endblock_gas_over":
            assert base == (1, "AssertionError"), base
        else:
            assert base == (-1, ""), (name, base)
        muts = [(-1, 0, 0, 0) + base]
        for k in range(150):
            which = rng.choice([0, 0, 0, 1, 1, 1, 1, 1, 2, 2, 5, 6, 6, 6, 8, 7, 7, 9, 3, 4, 10])
            S2, R2, RF2 = [list(x) for x in S], [list(x) for x in R], list(RF)
            T2, TF2, BL2, BF2, WD2 = [list(x) for x in T], list(TF), [list(x) for x in BL], list(BF), [list(x) for x in WD]
            C2, K2 = [list(x) for x in C], [list(x) for x in K]
            if which == 0:
                i, c = rng.randrange(len(S)), rng.randrange(13)
                if c == 0:
                    v = rng.choice([int(ExecutionState.EndTx), int(ExecutionState.BeginTx), int(ExecutionState.ADD), int(ExecutionState.EndBlock),
                                    int(ExecutionState.STOP)])
                    if v == S[i][c]:
                        continue
                else:
                    v = (1 - S[i][c]) if c in (3, 4) else corrupt_value(rng, S[i][c])
                S2[i][c] = v
            elif which == 1 and R:
                i, c = rng.randrange(len(R)), rng.randrange(14)
                if (c == 9 and not (RF[i] & 1)) or (c == 11 and not (RF[i] & 2)):
                    continue
                v = corrupt_value(rng, R[i][c]); R2[i][c] = v
            elif which == 2 and R:  # flip a value / value_prev type flag
                i, c, v = rng.randrange(len(R)), 100 + rng.randrange(2), 0
                bit = 1 << (c - 100)
                RF2[i] ^= bit
                if not RF2[i] & bit:
                    R2[i][9 if bit == 1 else 11] = 0
            elif which == 5 and R:  # a second rw row with the same key and another value: ambiguous lookup
                i, c = rng.randrange(len(R)), rng.choice([8, 10])
                v = corrupt_value(rng, R[i][c])
                R2.append(list(R[i])); R2[-1][c] = v; RF2.append(RF[i])
            elif which == 6 and T:
                i, c = rng.randrange(len(T)), rng.randrange(5)
                if c == 4 and not TF[i]:
                    continue
                v = corrupt_value(rng, T[i][c]); T2[i][c] = v
            elif which == 8 and T:  # tx value type flag
                i, c, v = rng.randrange(len(T)), 100, 0
                TF2[i] ^= 1
                if not TF2[i]:
                    T2[i][4] = 0
            elif which == 7 and BL:
                i, c = rng.randrange(len(BL)), rng.randrange(5)
                if c == 4:
                    c, v = 100, 0
                    BF2[i] ^= 1
                    if not BF2[i]:
                        BL2[i][3] = 0
                elif c == 3 and not BF[i]:
                    continue
                else:
                    v = corrupt_value(rng, BL[i][c]); BL2[i][c] = v
            elif which == 9 and WD:
                i, c = rng.randrange(len(WD)), rng.randrange(4)
                v = corrupt_value(rng, WD[i][c])
                if c == 0 and any(v == x[0] for x in WD):
                    continue  # two withdrawals with one id: sorted() over a Python set leaves their order unspecified
                WD2[i][c] = v
            elif which == 3 and C:
                i, c = rng.randrange(len(C)), rng.randrange(14)
                if c in (2, 5):
                    continue
                v = corrupt_value(rng, C[i][c]); C2[i][c] = v
            elif which == 4 and K:
                i, c = rng.randrange(len(K)), rng.randrange(5)
                v = corrupt_value(rng, K[i][c]); K2[i][c] = v
            elif which == 10 and R:  # drop an rw row
                i, c, v = rng.randrange(len(R)), 200, 0
                del R2[i]; del RF2[i]
            else:
                continue
            fr_, ex_ = run(S2, B, R2, RF2, C2, CF, K2, T2, TF2, BL2, BF2, WD2, first, last)
            muts.append((which, i, c, v, fr_, ex_))
            tot += 1
            nfail += fr_ >= 0
        for key, rows_, ncol in (("steps", S, 13), ("bytecode", B, 6), ("rw", R, 14), ("copy", C, 14), ("keccak", K, 5),
                                 ("tx", T, 5), ("block", BL, 4), ("wd", WD, 4)):
            out[f"{name}/{key}"] = to_matrix(rows_) if rows_ else np.zeros((ncol, 0, 4), dtype=np.uint64)
        for key, fl in (("rw_flags", RF), ("copy_flags", CF), ("tx_flags", TF), ("block_flags", BF)):
            out[f"{name}/{key}"] = np.array(fl, dtype=np.uint8)
        out[f"{name}/first_last"] = np.array([int(first), int(last)], dtype=np.int64)
        out[f"{name}/mut_kind"] = np.array([m[0] for m in muts], dtype=np.int64)
        out[f"{name}/mut_row"] = np.array([m[1] for m in muts], dtype=np.int64)
        out[f"{name}/mut_col"] = np.array([m[2] for m in muts], dtype=np.int64)
        out[f"{name}/mut_val"] = np.array([limbs(m[3]) for m in muts], dtype=np.uint64)
        out[f"{name}/exp_row"] = np.array([m[4] for m in muts], dtype=np.int64)
        out[f"{name}/exp_exc"] = np.array([m[5] for m in muts])
        print(name, len(R), "rw", len(T), "tx", len(WD), "wd", len(C), "copy", len(muts), "vectors",
              sorted(set(m[5] for m in muts)))
    np.savez_compressed(os.path.join(HERE, "evm11.npz"), **out)
    print(f"evm11: {tot} corruptions, {nfail} failing")

if __name__ == "__main__":
    which = sys.argv[1] if len(sys.argv) > 1 else "all"
    todo = {"bytecode": bytecode_cases}
    g = globals()
    for nm in ["state", "copy", "evm", "evm2", "evm3", "evm4", "evm5", "evm6", "evm7", "evm8", "evm9", "evm10", "evm11", "evm12", "evm13", "evm14", "evm15", "evm16", "evm17", "evm18", "evm19", "evm20", "evm21", "evm22", "evm23", "evm24", "evm25", "evm26", "evm27", "evm28", "exp", "pi", "tx", "sig", "fr", "synth"]:
        if nm + "_cases" in g:
            todo[nm] = g[nm + "_cases"]
    for nm, fn in todo.items():
        if which in ("all", nm):
            fn()
