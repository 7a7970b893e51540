"""The CPU oracle's restatement of the withdrawal circuit (oracle/withdrawal.c) reproduces every verdict of the
reference (tests/golden/withdrawal.npz: withdrawal_circuit.verify_circuit, :127-201), IndexError cases included."""
import withdrawal_cases as wc


def test_oracle_matches_every_withdrawal_golden():
    n = n_fail = 0
    kinds = set()
    for name, k, w, mx, r, exp_row, exp_exc in wc.vectors():
        got = wc.oracle_verdict(w, mx, r)
        assert got == (exp_row, exp_exc), f"{name}[{k}] oracle {got} reference {(exp_row, exp_exc)}"
        n += 1
        n_fail += exp_row >= 0
        kinds.add(exp_exc)
    assert n >= 400 and n_fail > 300
    assert {"", "AssertionError", "LookupUnsatFailure", "LookupAmbiguousFailure", "IndexError"} <= kinds
