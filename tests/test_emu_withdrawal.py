"""CPU emulation of the withdrawal circuit's row body (csrc/withdrawal.cu, built for the host by
tests/emu/withdrawal_emu.cc): the same verdict arrays as the oracle (oracle/withdrawal.c) on every golden vector and on
seeded random witnesses, in the canonical and the packed storage instance, whole and in shards; and the streamed RLP
bytes and RLC equal the host mirror's."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import oracle_lib
import withdrawal_cases as wc
from zkevm_specs_b200 import packing
from zkevm_specs_b200 import withdrawal_circuit as wdc
from zkevm_specs_b200.util import FQ, RLC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "emu", "withdrawal_emu.cc")
OUT = os.path.join(ROOT, "tests", "emu", "_build", "libwithdrawalemu.so")
CHALLENGE = np.array([0x1234567, 0x89ABCDEF, 0x13579BDF, 0x02468ACE], dtype=np.uint64)
P = FQ.field_modulus


@pytest.fixture(scope="module")
def lib():
    csrc = os.path.join(ROOT, "zkevm-specs_b200", "csrc")
    deps = [SRC, os.path.join(ROOT, "tests", "emu", "zk_emu.cu")] + [os.path.join(csrc, f) for f in os.listdir(csrc)] + [
        os.path.join(ROOT, "include", f) for f in os.listdir(os.path.join(ROOT, "include"))]
    if not os.path.exists(OUT) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in deps):
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        subprocess.run(["g++", "-x", "c++", "-std=c++17", "-O1", "-fPIC", "-shared", "-D__host__=", "-D__device__=",
                        "-D__forceinline__=inline", "-D__noinline__=__attribute__((noinline))", "-w", "-o", OUT, SRC],
                       check=True)
    return ctypes.CDLL(OUT)


def emu_check(L, rows, keccak, mpt, block, r, mx, row_begin, row_end, row_base=0):
    rows, keccak, mpt, block = [np.ascontiguousarray(a, dtype=np.uint64) for a in (rows, keccak, mpt, block)]
    n = wc.n_constraints()
    ff = np.zeros(n, dtype=np.uint32)
    fc = np.zeros(n, dtype=np.uint64)
    c, p = ctypes.c_uint64, oracle_lib.p64
    rr = np.ascontiguousarray(r, dtype=np.uint64)
    assert L.emu_check_withdrawal(p(rows), c(rows.shape[1]), p(keccak), c(keccak.shape[1]), p(mpt), c(mpt.shape[1]), p(block),
                                  c(block.shape[1]), p(rr), c(mx), c(row_begin), c(row_end), c(row_base), p(CHALLENGE),
                                  ff.ctypes.data_as(oracle_lib.U32P), p(fc)) == 0
    return ff, fc


@pytest.mark.parametrize("packed", [False, True])
def test_emu_matches_oracle_on_goldens(lib, packed):
    ctypes.c_int.in_dll(lib, "g_emu_packed").value = int(packed)
    try:
        n = 0
        for name, k, w, mx, r, exp_row, exp_exc in wc.vectors():
            _, end, _ = wc.plan(w["rows"].shape[1], mx)
            if end == 0:
                continue
            rows = wc.used_rows(w["rows"], mx)
            ff, fc = emu_check(lib, rows, w["keccak"], w["mpt"], w["block"], r, mx, 0, end)
            off, ofc = wc.oracle_check(rows, w["keccak"], w["mpt"], w["block"], r, mx, 0, end)
            assert np.array_equal(ff, off) and np.array_equal(fc, ofc), f"{name}[{k}]"
            assert wc.verdict(ff, mx, w["rows"].shape[1]) == (exp_row, exp_exc), f"{name}[{k}]"
            n += 1
        assert n > 400
    finally:
        ctypes.c_int.in_dll(lib, "g_emu_packed").value = 0


def random_witness(rng: random.Random, n: int, r):
    """n rows from the reference's generator recipe (root = prev + 5), random field widths, some padding-shaped rows;
    tables from the oracle (keccak) and by hand (MPT, block); then random single-cell corruptions"""
    cells, mpt = [], []
    id0, prev = rng.choice([rng.randrange(1 << 64), P - 3]), 0
    for k in range(n):
        i = (id0 + k) % P
        v, a = rng.choice([0, 1, 127, 128, rng.randrange(1 << 64), P - 1]), rng.choice([0, 5, rng.randrange(1 << 160)])
        m = rng.choice([0, 1, rng.randrange(1 << 64), rng.randrange(P)]) if rng.random() < 0.9 else 0
        h = (rng.randrange(1 << 128), rng.randrange(1 << 128))
        root = prev + 5
        cells.append([i, v, a, m, h[0], h[1], root, 0])
        mpt.append([a, 8 if m else 4, i & ((1 << 128) - 1), i >> 128, root, 0, prev, 0, h[0], h[1], 0, 0])
        prev = root
    rows = packing.matrix_from_ints(cells, 8)
    keccak = wc.oracle_keccak_rows(rows, r)
    block = packing.matrix_from_ints([[9, 0, prev, 0]], 4)
    w = {"rows": rows, "keccak": keccak, "mpt": packing.matrix_from_ints(mpt, 12), "block": block}
    for _ in range(rng.randrange(0, 4)):
        t = rng.choice(["rows", "rows", "keccak", "mpt", "block"])
        w[t][rng.randrange(w[t].shape[0]), rng.randrange(w[t].shape[1]), rng.randrange(2)] ^= np.uint64(1 << rng.randrange(8))
    return w


@pytest.mark.parametrize("packed", [False, True])
def test_emu_matches_oracle_on_random_witnesses_and_shards(lib, packed):
    ctypes.c_int.in_dll(lib, "g_emu_packed").value = int(packed)
    rng = random.Random(7 + packed)
    r = oracle_lib.limbs(rng.randrange(P))
    try:
        for t in range(40):
            n = rng.randrange(1, 60)
            w = random_witness(rng, n, r)
            mx = n
            off, ofc = wc.oracle_check(w["rows"], w["keccak"], w["mpt"], w["block"], r, mx)
            ff, fc = emu_check(lib, w["rows"], w["keccak"], w["mpt"], w["block"], r, mx, 0, n)
            assert np.array_equal(ff, off) and np.array_equal(fc, ofc), t
            # shards with halos: local row 0 is global row b - 1 except for the first shard
            acc_ff, acc_fc = np.full_like(ff, 0xFFFFFFFF), np.zeros_like(fc)
            cuts = sorted({0, n, *[rng.randrange(n + 1) for _ in range(3)]})
            for b, e in zip(cuts, cuts[1:]):
                lo, hi = max(b - 1, 0), min(e + 1, n)
                sub = np.ascontiguousarray(w["rows"][:, lo:hi])
                sff, sfc = emu_check(lib, sub, w["keccak"], w["mpt"], w["block"], r, mx, b - lo, e - lo, lo)
                acc_ff, acc_fc = np.minimum(acc_ff, sff), acc_fc + sfc
            assert np.array_equal(acc_ff, off) and np.array_equal(acc_fc, ofc), t
    finally:
        ctypes.c_int.in_dll(lib, "g_emu_packed").value = 0


def test_streamed_rlp_and_rlc_equal_the_host_mirror(lib):
    rng = random.Random(3)
    r = rng.randrange(P)
    widths = [0, 1, 7, 8, 63, 64, 127, 128, 160, 200, 248, 253]
    for _ in range(300):
        f = [rng.choice([0, 1, 0x7F, 0x80, 0xFF, 0x100, P - 1, rng.randrange(1 << rng.choice(widths[1:])) % P]) for _ in range(4)]
        cells = np.ascontiguousarray(np.concatenate([oracle_lib.limbs(v) for v in f]))
        out = np.zeros(140, dtype=np.uint8)
        rlc = np.zeros(4, dtype=np.uint64)
        n = lib.emu_withdrawal_rlp(oracle_lib.p64(cells), oracle_lib.p64(oracle_lib.limbs(r)), out.ctypes.data_as(ctypes.c_void_p),
                                   oracle_lib.p64(rlc))
        enc = wdc.rlp_encode_ints(f)
        assert bytes(out[:n]) == enc
        assert oracle_lib.from_limbs(rlc) == RLC(bytes(reversed(enc)), FQ(r), n_bytes=len(enc)).expr().n
