"""Pins the CPU oracle's public-inputs-circuit restatement (oracle/pi.c) against vectors produced by the reference's
own check_row under the loop of verify_circuit (tests/golden/pi_*.npz: witnesses from the reference's
public_data2witness + single-cell corruptions of the witness, the keccak table and the calldata gas-cost table)."""
import golden_util
import oracle_lib


def test_oracle_pi_matches_reference_golden():
    classes = oracle_lib.constraint_classes(7)
    n = n_fail = 0
    kinds, ids = set(), set()
    for name, k, R, K, G, clen, exp_row, exp_exc in golden_util.pi_vectors():
        ff, fc = oracle_lib.check_pi(R, K, G, clen)
        row, exc = oracle_lib.first_failure(ff, classes)
        assert (row, exc) == (exp_row, exp_exc), f"{name}[{k}]: oracle {(row, exc)} reference {(exp_row, exp_exc)}"
        n += 1
        n_fail += exp_row >= 0
        kinds.add(exp_exc)
        ids |= {i for i in range(len(ff)) if ff[i] != 0xFFFFFFFF}
    assert n > 700 and n_fail > 300
    assert {"AssertionError", "LookupUnsatFailure"} <= kinds
    assert len(ids) >= 20, sorted(ids)  # most of the 30 constraint ids fire somewhere in the corpus
