"""Host mirror of the public-inputs circuit (zkevm-specs_b200/pi_circuit.py) on the CPU: public_data2witness builds,
cell for cell, the witness the reference's public_data2witness built for the same PublicData (tests/golden/pi_*.npz
stores both), and the copy-constraint half of verify_circuit rejects what the reference's own negative tests override
(tests/test_public_inputs.py:163-210).  The gates themselves run on the GPU (tests/test_gpu_pi.py)."""
import json

import numpy as np
import pytest

import golden_util
import oracle_lib
from zkevm_specs_b200 import pi_circuit as pc
from zkevm_specs_b200.util import FQ, Word, WordOrValue


def load_public_data(z, name):
    d = json.loads(str(z[f"{name}/public_data"]))
    b = d["block"]
    for k in ("bloom", "extra"):
        b[k] = bytes.fromhex(b[k])
    txs = [pc.Transaction(t["nonce"], t["gas_price"], t["gas"], t["from_addr"], t["to_addr"], t["value"], bytes.fromhex(t["data"]),
                          t["tx_sign_hash"]) for t in d["txs"]]
    wds = [pc.Withdrawal(**w) for w in d["withdrawals"]]
    return pc.PublicData(d["chain_id"], pc.Block(**b), d["state_root_prev"], d["block_hashes"], txs, wds)


def cases():
    z = golden_util.load_pi()
    for name in z["names"]:
        name = str(name)
        yield z, name, [int(x) for x in z[f"{name}/params"]]


def test_public_data2witness_equals_the_reference_witness():
    for z, name, (max_txs, max_cd, max_wd) in cases():
        w = pc.public_data2witness(load_public_data(z, name), max_txs, max_cd, max_wd)
        assert w.circuit_len == int(z[f"{name}/circuit_len"][0]) == w.cells.shape[1]
        assert np.array_equal(w.cells, z[f"{name}/rows"]), (name, np.nonzero((w.cells != z[f"{name}/rows"]).any(axis=2)))
        assert np.array_equal(w.keccak_table.matrix(), z[f"{name}/keccak"])
        assert np.array_equal(w.gas_matrix(), z[f"{name}/gas"])
        ff, _ = oracle_lib.check_pi(w.cells, w.keccak_table.matrix(), w.gas_matrix(), w.circuit_len)
        assert (ff == 0xFFFFFFFF).all()
        pc._copy_constraints(w, max_txs, max_cd, max_wd)  # the positive witness satisfies the copy constraints
        assert w.copy_constrains == []
        r = w.row(3)
        w.set_row(3, r)
        assert np.array_equal(w.cells, z[f"{name}/rows"])


@pytest.mark.parametrize("override", [
    lambda w: w.block_table.table.__setitem__(5, WordOrValue(Word(123))),
    lambda w: setattr(w.tx_table.table[5], "tx_id", FQ(123)),
    lambda w: setattr(w.tx_table.table[5], "index", FQ(123)),
    lambda w: setattr(w.tx_table.table[5], "value", WordOrValue(Word(123))),
    lambda w: setattr(w.public_inputs, "pi_keccak", Word(123)),
    lambda w: setattr(w.public_inputs, "state_root", WordOrValue(Word(123))),
    lambda w: setattr(w.public_inputs, "state_root_prev", WordOrValue(Word(123))),
])
def test_copy_constraints_reject_the_reference_negative_overrides(override):
    z, name, (max_txs, max_cd, max_wd) = next(cases())
    w = pc.public_data2witness(load_public_data(z, name), max_txs, max_cd, max_wd)
    override(w)
    with pytest.raises(AssertionError):
        pc._copy_constraints(w, max_txs, max_cd, max_wd)
