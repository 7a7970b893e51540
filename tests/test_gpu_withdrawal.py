"""GPU parity of the CUDA withdrawal-circuit checker (csrc/withdrawal.cu) against the reference's verdicts
(tests/golden/withdrawal.npz), the CPU oracle array for array at 2^16-2^20 rows, row shards and the packed upload; the
device witness assignment against the host mirror; and the reference's tests/test_withdrawal_circuit.py rewritten
against the host API."""
import random

import numpy as np
import pytest

import oracle_lib
import withdrawal_cases as wc
from zkevm_specs_b200 import native, packing, synth
from zkevm_specs_b200 import withdrawal_circuit as wdc
from zkevm_specs_b200.evm_circuit.spec import BlockContextFieldTag, MPTProofType
from zkevm_specs_b200.evm_circuit.table import BlockTableRow, MPTTableRow
from zkevm_specs_b200.util import FQ, Word
from zkevm_specs_b200.util.hash import keccak256

pytestmark = pytest.mark.gpu


def gpu_check(ctx, w, mx, r, row_begin=0, row_end=None, row_base=0):
    return wdc.check_matrices(ctx, w["rows"], w["keccak"], w["mpt"], w["block"], oracle_lib.from_limbs(r), mx, row_begin,
                              row_end, row_base)


def test_withdrawal_golden_and_oracle_parity():
    ctx = native.default_context()
    n = 0
    for name, k, w, mx, r, exp_row, exp_exc in wc.vectors():
        _, end, _ = wc.plan(w["rows"].shape[1], mx)
        if end == 0:
            continue
        u = dict(w, rows=wc.used_rows(w["rows"], mx))
        ff, fc = gpu_check(ctx, u, mx, r, 0, end)
        off, ofc = wc.oracle_check(u["rows"], w["keccak"], w["mpt"], w["block"], r, mx, 0, end)
        assert np.array_equal(ff, off) and np.array_equal(fc, ofc), f"{name}[{k}] differs from oracle"
        assert wc.verdict(ff, mx, w["rows"].shape[1]) == (exp_row, exp_exc), f"{name}[{k}]"
        n += 1
    assert n > 400


@pytest.mark.parametrize("log_n", [16, 20])
def test_large_witness_matches_oracle_sharded_and_packed(log_n):
    n = 1 << log_n
    ctx = native.default_context()
    r = 0x0DDBA11 + log_n
    ctx.set_challenge(native.CHALLENGE_KECCAK, r)
    s = synth.withdrawals(n, n, seed=log_n, ctx=ctx)
    ff, fc = ctx.check(native.CIRCUIT_WITHDRAWAL, 0, n, 0, 0)
    assert (ff == native.PASS).all(), native.first_failure(ff, native.CIRCUIT_WITHDRAWAL)
    rl = oracle_lib.limbs(r)
    w = {"rows": s["rows"].copy(), "keccak": wc.oracle_keccak_rows(s["rows"], rl), "mpt": s["mpt"].copy(), "block": s["block"]}
    rng = np.random.default_rng(log_n)
    for col in range(8):  # corruptions in every cell of some rows, the first and the last row included
        for row in list(rng.integers(0, n, 3)) + [0, n - 1]:
            w["rows"][col, row, int(rng.integers(0, 2))] ^= np.uint64(1 << int(rng.integers(0, 8)))
    for t in ("keccak", "mpt"):
        w[t][int(rng.integers(0, w[t].shape[0])), int(rng.integers(1, w[t].shape[1])), 0] ^= np.uint64(1)
    off, ofc = wc.oracle_check(w["rows"], w["keccak"], w["mpt"], w["block"], rl, n)
    ff, fc = gpu_check(ctx, w, n, rl)
    assert np.array_equal(ff, off) and np.array_equal(fc, ofc)
    assert (ff != native.PASS).sum() >= 3
    # four row shards, each with its halo rows (global row b - 1 and e), no halo past the circuit's ends
    acc_ff, acc_fc = np.full_like(ff, native.PASS), np.zeros_like(fc)
    for q in range(4):
        b, e = n * q // 4, n * (q + 1) // 4
        lo, hi = max(b - 1, 0), min(e + 1, n)
        sub = dict(w, rows=np.ascontiguousarray(w["rows"][:, lo:hi]))
        sff, sfc = gpu_check(ctx, sub, n, rl, b - lo, e - lo, lo)
        acc_ff, acc_fc = np.minimum(acc_ff, sff), acc_fc + sfc
    assert np.array_equal(acc_ff, off) and np.array_equal(acc_fc, ofc)
    # packed narrow columns == canonical
    ctx.upload_columns_packed(native.CIRCUIT_WITHDRAWAL, packing.pack_matrix(w["rows"]))
    pff, pfc = ctx.check(native.CIRCUIT_WITHDRAWAL, 0, n, 0, 0)
    assert np.array_equal(pff, off) and np.array_equal(pfc, ofc)


def test_device_assignment_equals_host_mirror():
    ctx = native.default_context()
    rng = random.Random(5)
    r = FQ(rng.randrange(FQ.field_modulus))
    ctx.set_challenge(native.CHALLENGE_KECCAK, r.n)
    P = FQ.field_modulus
    for n, mx in ((0, 0), (0, 3), (1, 1), (4, 4), (5, 9), (37, 40)):
        recs = []
        for k in range(n):
            f = [rng.choice([0, 1, 0x7F, 0x80, P - 1, rng.randrange(1 << rng.choice([8, 64, 160, 253])) % P]) for _ in range(4)]
            recs.append(f + [rng.randrange(1 << 255)])
        arr = np.zeros((n, 5, 4), dtype=np.uint64)
        for k, f in enumerate(recs):
            for c, v in enumerate(f):
                arr[k, c] = packing.int_to_cell(v)
        ctx.assign_withdrawal_circuit(arr, mx)
        rows, _ = ctx.download_columns(native.CIRCUIT_WITHDRAWAL)
        host, kt, last = [], wdc.KeccakTable(), Word(0)
        for f in recs:
            enc = wdc.rlp_encode_ints(f[:4])
            kt.add(enc, r)
            last = Word(f[4])
            host.append(wdc.Row(FQ(f[0]), FQ(f[1]), FQ(f[2]), FQ(f[3]), Word(keccak256(enc)), last))
        host += [wdc.Row(FQ(0), FQ(0), FQ(0), FQ(0), Word(0), last) for _ in range(mx - n)]
        assert np.array_equal(rows, wdc.pack_rows(host)), (n, mx)
        # the device keccak table is the host one: a check of every row against it equals the check against the host's
        if mx:
            ctx.set_challenge(native.PARAM_WITHDRAWAL_MAX, mx)
            ctx.upload_table(native.TABLE_MPT, np.zeros((12, 0, 4), dtype=np.uint64))
            ctx.upload_table(native.TABLE_BLOCK, np.zeros((4, 0, 4), dtype=np.uint64))
            dev_ff, dev_fc = ctx.check(native.CIRCUIT_WITHDRAWAL, 0, mx, 0, 0)
            ctx.upload_table(native.TABLE_KECCAK, kt.matrix())
            ff, fc = ctx.check(native.CIRCUIT_WITHDRAWAL, 0, mx, 0, 0)
            assert np.array_equal(dev_ff, ff) and np.array_equal(dev_fc, fc)
            assert ff[wc.n_constraints() - 4] == native.PASS or n < mx  # WD_KECCAK_LOOKUP holds on every assigned row
    # an assigned witness of withdrawals with the reference's mock MPT rows verifies
    s = synth.withdrawals(300, 300, seed=1, ctx=ctx)
    ff, _ = ctx.check(native.CIRCUIT_WITHDRAWAL, 0, 300, 0, 0)
    assert (ff == native.PASS).all()


# ---- the reference's tests/test_withdrawal_circuit.py against the host API ---------------------------------------
R = FQ(0x1F2E3D4C5B6A79881F2E3D4C5B6A79881F2E3D4C5B6A79881F2E3D4C5B6A798)


def mock_mpt_update(id, validator_id, address, amount, prev_root):
    h = keccak256(wdc.rlp_encode_ints([id, validator_id, address, amount]))
    return MPTTableRow(FQ(address), FQ(int(MPTProofType.WithdrawalMod)), Word(id), Word(prev_root + 5), Word(prev_root),
                       Word(h), Word(0))


def gen_withdrawals(num, rng):
    wid = rng.randrange(0, 2**64)
    wds, roots, prev = [], [], 0
    for i in range(num):
        v, a, m = rng.randrange(0, 2**64), rng.randrange(1, 2**160), rng.randrange(1, 2**64)
        wds.append((wid + i, v, a, m))
        prev = mock_mpt_update(wid + i, v, a, m, prev).root.int_value()
        roots.append(prev)
    return wds, roots


def withdrawals2witness(wds, MAX, roots, r):
    last, rows, kt, mpt = 0, [], wdc.KeccakTable(), set()
    for (i, v, a, m), root in zip(wds, roots):
        enc = wdc.rlp_encode_ints([i, v, a, m])
        kt.add(enc, r)
        mpt.add(mock_mpt_update(i, v, a, m, last))
        rows.append(wdc.Row(FQ(i), FQ(v), FQ(a), FQ(m), Word(keccak256(enc)), Word(root)))
        last = root
    for _ in range(len(wds), MAX):
        rows.append(wdc.Row(FQ(0), FQ(0), FQ(0), FQ(0), Word(0), Word(last)))
    block = {BlockTableRow(FQ(int(BlockContextFieldTag.WithdrawalRoot)), FQ(0), Word(last))}
    return wdc.Witness(rows, wdc.MPTTable(mpt), kt, wdc.BlockTable(block))


def verify(witness, MAX, r, success=True):
    assert len(witness.rows) == MAX
    if success:
        wdc.verify_circuit(witness, MAX, r)
    else:
        with pytest.raises(Exception):
            wdc.verify_circuit(witness, MAX, r)


def test_withdrawal_withdrawals2witness():
    wds, roots = gen_withdrawals(20, random.Random(11))
    witness = withdrawals2witness(wds, 20, roots, R)
    for wd, row in zip(wds, witness.rows):
        assert wd[0] == row.withdrawal_id.n and wd[2] == row.address.n


@pytest.mark.parametrize("name", ["basic", "id_not_incremental", "inconsistent_id", "inconsistent_validator_id",
                                  "inconsistent_address", "inconsistent_amount"])
def test_withdrawal_reference_cases(name):
    MAX = 2 if name == "inconsistent_amount" else 5
    wds, roots = gen_withdrawals(MAX, random.Random(len(name)))
    witness = withdrawals2witness(wds, MAX, roots, R)
    if name == "basic":
        return verify(witness, MAX, R)
    row0 = witness.rows[0]
    if name == "id_not_incremental":
        witness.rows[1].withdrawal_id -= 1
    elif name == "inconsistent_id":
        row0.withdrawal_id = FQ(999)
    elif name == "inconsistent_validator_id":
        row0.validator_id = FQ(999)
    elif name == "inconsistent_address":
        row0.address = FQ(0xDEADBEEF)
    else:
        row0.amount = FQ(10)
    verify(witness, MAX, R, success=False)
