"""Withdrawal circuit host mirror (zkevm_specs_b200.withdrawal_circuit), CPU only: its RLP bytes equal rlp.encode of the
reference's dependency stand-in (oracle/pyshim/rlp), its keccak-table RLC equals the reference's RLC, and the list
indexing quirks of verify_circuit are raised before any device work."""
import importlib.util
import os
import random

import pytest

from zkevm_specs_b200 import withdrawal_circuit as wdc
from zkevm_specs_b200.util import FQ, RLC, Word

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = FQ.field_modulus


def _pyshim_rlp():
    spec = importlib.util.spec_from_file_location("pyshim_rlp", os.path.join(ROOT, "oracle", "pyshim", "rlp", "__init__.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def field_values(rng):
    return [rng.choice([0, 1, 0x7F, 0x80, 0xFF, 0x100, P - 1, rng.randrange(1 << rng.choice([8, 64, 160, 253])) % P])
            for _ in range(4)]


def test_rlp_bytes_equal_rlp_encode():
    rlp = _pyshim_rlp()
    rng = random.Random(1)
    long_payloads = 0
    for _ in range(2000):
        f = field_values(rng)
        enc = wdc.rlp_encode_ints(f)
        assert enc == rlp.encode(f)
        long_payloads += enc[0] == 0xF8
    assert long_payloads > 50


def test_keccak_table_rlc_is_the_reference_rlc():
    rng = random.Random(2)
    r = FQ(rng.randrange(P))
    for _ in range(200):
        enc = wdc.rlp_encode_ints(field_values(rng))
        kt = wdc.KeccakTable()
        kt.add(enc, r)
        row = [t for t in kt.table if t[0] == 1][0]
        acc = 0
        for b in enc:  # Horner over the bytes in order = RLC of the reversed bytes
            acc = (acc * r.n + b) % P
        assert row[1] == FQ(acc) == RLC(bytes(reversed(enc)), r, n_bytes=len(enc)).expr()
        assert row[2] == len(enc)
    assert (FQ(0), FQ(0), FQ(0), Word(0)) in wdc.KeccakTable().table


def test_row_list_quirks_raise_index_error_without_a_device():
    w = wdc.Witness([], wdc.MPTTable(set()), wdc.KeccakTable(), wdc.BlockTable(set()))
    for mx in (0, 1, 3):
        with pytest.raises(IndexError):
            wdc.verify_circuit(w, mx, FQ(5), ctx=object())  # raised before the context is touched
