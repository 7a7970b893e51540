"""GPU parity of the CUDA public-inputs-circuit checker (csrc/pi.cu) against the reference's verdicts
(tests/golden/pi_*.npz: check_row under verify_circuit's loop, pi_circuit.py:150-321, 447-459), the CPU oracle array
for array, and through the host API in the style of the reference's tests/test_public_inputs.py."""
import numpy as np
import pytest

import golden_util
import oracle_lib
from test_pi_host import cases, load_public_data
from zkevm_specs_b200 import native, packing, synth
from zkevm_specs_b200 import pi_circuit as pc
from zkevm_specs_b200.util import FQ, Word, WordOrValue

pytestmark = pytest.mark.gpu


def test_pi_golden_and_oracle_parity():
    ctx = native.default_context()
    n = n_fail = 0
    for name, k, R, K, G, clen, exp_row, exp_exc in golden_util.pi_vectors():
        ff, fc = pc.check_matrices(ctx, R, K, G, clen)
        off, ofc = oracle_lib.check_pi(R, K, G, clen)
        assert np.array_equal(ff, off) and np.array_equal(fc, ofc), f"{name}[{k}] differs from oracle"
        hit = native.first_failure(ff, native.CIRCUIT_PI)
        got = (-1, "") if hit is None else (hit[0], oracle_lib.EXC_OF_CLASS[hit[2]])
        assert got == (exp_row, exp_exc), f"{name}[{k}] cuda {got} reference {(exp_row, exp_exc)}"
        n += 1
        n_fail += exp_row >= 0
    assert n > 700 and n_fail > 300


def test_pi_host_api_like_reference_test_public_inputs():
    """tests/test_public_inputs.py: test_basic + the override_not_success family"""
    MAX_TXS, MAX_CALLDATA_BYTES, MAX_WITHDRAWALS = 2, 8, 2
    pd = synth.pi_public_data(MAX_TXS - 1, MAX_CALLDATA_BYTES, MAX_WITHDRAWALS, seed=0)
    pc.verify_circuit(pc.public_data2witness(pd, MAX_TXS, MAX_CALLDATA_BYTES, MAX_WITHDRAWALS), MAX_TXS, MAX_CALLDATA_BYTES,
                      MAX_WITHDRAWALS)
    overrides = [
        lambda w: w.block_table.table.__setitem__(5, WordOrValue(Word(123))),
        lambda w: setattr(w.tx_table.table[5], "tx_id", FQ(123)),
        lambda w: setattr(w.public_inputs, "pi_keccak", Word(123)),
        # gate-level overrides: these pass the copy constraints and are caught on the device
        lambda w: w.cells.__setitem__((pc.P_KRLC, 77), packing.int_to_cell(5)),
        lambda w: w.cells.__setitem__((pc.P_CD_GAS, 10 * MAX_TXS + 2), packing.int_to_cell(5)),
        lambda w: w.cells.__setitem__((pc.P_WD_AMOUNT, 10 * MAX_TXS + 1 + MAX_CALLDATA_BYTES), packing.int_to_cell(0)),
    ]
    for ov in overrides:
        w = pc.public_data2witness(pd, MAX_TXS, MAX_CALLDATA_BYTES, MAX_WITHDRAWALS)
        ov(w)
        with pytest.raises(AssertionError):
            pc.verify_circuit(w, MAX_TXS, MAX_CALLDATA_BYTES, MAX_WITHDRAWALS)
    w = pc.public_data2witness(pd, MAX_TXS, MAX_CALLDATA_BYTES, MAX_WITHDRAWALS)
    w.calldata_gas_cost_table = {(0, 0, 0)}  # the CallDataLength rows look their gas cost up: unsat
    with pytest.raises(Exception) as ei:
        pc.verify_circuit(w, MAX_TXS, MAX_CALLDATA_BYTES, MAX_WITHDRAWALS)
    assert type(ei.value).__name__ == "LookupUnsatFailure"


def test_pi_full_size_sharded_and_packed_match_oracle():
    """a 64-tx block with 2^17 calldata bytes (~1.5e5 circuit rows): whole circuit == oracle; row shards with a halo row
    == whole; packed narrow columns == canonical; planted corruptions are found at the oracle's rows"""
    MAX_TXS, MAX_CD, MAX_WD = 64, 1 << 17, 16
    pd = synth.pi_public_data(48, MAX_CD, MAX_WD, seed=5)
    w = pc.public_data2witness(pd, MAX_TXS, MAX_CD, MAX_WD)
    n = w.cells.shape[1]
    K, G = w.keccak_table.matrix(), w.gas_matrix()
    ctx = native.default_context()
    ff, fc = pc.check_matrices(ctx, w.cells, K, G, w.circuit_len)
    assert (ff == native.PASS).all(), native.first_failure(ff, native.CIRCUIT_PI)
    cells = w.cells.copy()
    for col, row in ((pc.P_KRLC, n - 3), (pc.P_IS_FINAL, 700), (pc.P_TX_INDEX, 10 * MAX_TXS + 500), (pc.P_VALUE_LC, n // 2),
                     (pc.P_TXID_DIFF_INV, 10 * MAX_TXS + 1 + 3000), (pc.P_WD_ID, 10 * MAX_TXS + 1 + MAX_CD + 3)):
        cells[col, row, 0] ^= np.uint64(1)
    off, ofc = oracle_lib.check_pi(cells, K, G, w.circuit_len)
    ff, fc = pc.check_matrices(ctx, cells, K, G, w.circuit_len)
    assert np.array_equal(ff, off) and np.array_equal(fc, ofc)
    assert (ff != native.PASS).sum() >= 5
    # row shards with a +1 halo, no wrap except through the last shard's halo = row 0
    acc_ff = np.full_like(ff, native.PASS)
    acc_fc = np.zeros_like(fc)
    for s in range(4):
        b, e = n * s // 4, n * (s + 1) // 4
        idx = np.arange(b, e + 1) % n
        sub = np.ascontiguousarray(cells[:, idx])
        sff, sfc = pc.check_matrices(ctx, sub, K, G, w.circuit_len, 0, e - b, b, 0)
        acc_ff = np.minimum(acc_ff, sff)
        acc_fc += sfc
    assert np.array_equal(acc_ff, off) and np.array_equal(acc_fc, ofc)
    ctx.set_challenge(native.CHALLENGE_PI_KECCAK, pc.keccak_rand.n)
    ctx.upload_columns_packed(native.CIRCUIT_PI, packing.pack_matrix(cells))
    pff, pfc = ctx.check(native.CIRCUIT_PI, 0, n, 0, native.FLAG_WRAP)
    assert np.array_equal(pff, off) and np.array_equal(pfc, ofc)
