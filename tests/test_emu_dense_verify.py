"""CPU diff of the typed strip form of the rw table's dense structure verify (lookup.cuh:pos_verify_dense_strip, what
k_pos_verify_dense_typed runs for narrow rw tables) against the row-at-a-time form (pos_verify_dense_row): the same
flag and the same split row on seeded tables with every irregularity the verify has to catch."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "emu", "dense_verify_emu.cc")
OUT = os.path.join(ROOT, "tests", "emu", "_build", "libdenseverify.so")
START, STACK = 1, 8  # rw table tags: Target.Start (the padding rows of the tail), Target.Stack


@pytest.fixture(scope="module")
def lib():
    deps = [SRC, os.path.join(ROOT, "zkevm-specs_b200", "csrc", "lookup.cuh"), os.path.join(ROOT, "zkevm-specs_b200", "csrc", "fr.cuh")]
    if not os.path.exists(OUT) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in deps):
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        subprocess.run(["g++", "-x", "c++", "-std=c++17", "-O1", "-fPIC", "-shared", "-D__host__=", "-D__device__=",
                        "-D__forceinline__=inline", "-D__noinline__=__attribute__((noinline))", "-w", "-o", OUT, SRC],
                       check=True)
    return ctypes.CDLL(OUT)


def verify(lib, counters, tags, wc, has_tail=True):
    """tags: uint8 per row (stored 1 byte per row) or an int (a constant column). -> (row form, strip form)"""
    n = len(counters)
    col = np.zeros((n * wc + 31) // 32 * 32 + 32, dtype=np.uint8)
    col[:n * wc] = np.asarray(counters, dtype=np.uint32 if wc == 4 else np.uint64).view(np.uint8)
    if isinstance(tags, int):
        tag_col, wt = np.zeros(32, dtype=np.uint8), 0
        tag_col[:8] = np.array([tags], dtype=np.uint64).view(np.uint8)
    else:
        tag_col, wt = np.zeros((n + 31) // 32 * 32 + 32, dtype=np.uint8), 1
        tag_col[:n] = tags
    buf = np.ascontiguousarray(np.concatenate([col, tag_col]))
    ok_row = np.zeros(2, dtype=np.uint32)
    ok_strip = np.zeros(2, dtype=np.uint32)
    u32p = ctypes.POINTER(ctypes.c_uint32)
    rc = lib.emu_dense_verify(buf.ctypes.data_as(ctypes.c_void_p), ctypes.c_uint64(0), ctypes.c_uint32(wc),
                              ctypes.c_uint64(len(col)), ctypes.c_uint32(wt), ctypes.c_uint64(n), ctypes.c_int(int(has_tail)),
                              ok_row.ctypes.data_as(u32p), ok_strip.ctypes.data_as(u32p))
    assert rc == 0
    return tuple(ok_row.tolist()), tuple(ok_strip.tolist())


def table(n_head, n_tail, base=1):
    """a regular rw table: a dense head of Stack rows from `base`, then a dense tail of Start rows from 1"""
    counters = np.concatenate([np.arange(base, base + n_head), np.arange(1, 1 + n_tail)]).astype(np.uint64)
    tags = np.concatenate([np.full(n_head, STACK), np.full(n_tail, START)]).astype(np.uint8)
    return counters, tags


def cases(rng):
    """(name, counters, tags, expected (flag, split) or None)"""
    for n_head, n_tail in ((1, 0), (0, 1), (7, 0), (8, 0), (9, 3), (16, 8), (17, 5), (100, 0), (93, 31)):
        c, t = table(n_head, n_tail, base=int(rng.integers(1, 1 << 20)))
        n = n_head + n_tail
        yield f"regular {n_head}+{n_tail}", c, t, (1, 0 if n_head == 0 else (n_head if n_tail else n))
    yield "1-row table", np.array([5], dtype=np.uint64), np.array([STACK], dtype=np.uint8), (1, 1)
    yield "1-row Start table", np.array([5], dtype=np.uint64), np.array([START], dtype=np.uint8), (1, 0)
    yield "empty tail", *table(41, 0), (1, 41)
    yield "Start tail at row 0", *table(0, 23), (1, 0)
    for k in (1, 7, 8, 9, 15, 30):
        c, t = table(33, 12)
        c[k] += np.uint64(1 + rng.integers(3))  # a gap in rw_counter (head)
        yield f"gap at row {k}", c, t, None
        c, t = table(33, 12)
        c[k] = c[k - 1]  # a repeated counter
        yield f"repeated counter at row {k}", c, t, None
        c, t = table(6, 34)
        c[6 + k] += np.uint64(1)  # a gap in the tail
        yield f"tail gap at row {6 + k}", c, t, None
        c, t = table(k, 20)
        t[k + 3] = STACK  # a head row after the tail
        yield f"head row after the tail at {k + 3}", c, t, None
        c, t = table(k + 8, 20)
        c[k + 8] = 0  # tail counters restarting at 0 instead of 1: still one dense tail run
        c[k + 8:] = np.arange(20, dtype=np.uint64)
        yield f"tail from 0 at {k + 8}", c, t, (1, k + 8)
    c, t = table(20, 0)
    c[19] = np.uint64(0xFFFFFFFF)
    yield "counter at the 4-byte limit", c, t, None
    for f in range(120):  # seeded fuzz: random lengths, a few random cell changes
        n_head, n_tail = int(rng.integers(0, 40)), int(rng.integers(0, 20))
        if n_head + n_tail == 0:
            continue
        c, t = table(n_head, n_tail, base=int(rng.integers(1, 1000)))
        for _ in range(int(rng.integers(0, 3))):
            r = int(rng.integers(len(c)))
            if rng.integers(2):
                c[r] = np.uint64(int(c[r]) + int(rng.integers(-2, 3)) if int(c[r]) > 2 else 7)
            else:
                t[r] = START if t[r] == STACK else STACK
        yield f"fuzz {f}", c, t, None


@pytest.mark.parametrize("wc", [4, 8])
def test_emu_typed_dense_verify_equals_row_form(lib, wc):
    rng = np.random.default_rng(11 + wc)
    n_irregular = 0
    for name, c, t, want in cases(rng):
        got_row, got_strip = verify(lib, c, t, wc)
        assert got_strip == got_row, (name, wc, got_row, got_strip)
        if want is not None:
            assert got_row == want, (name, got_row, want)
        n_irregular += got_row[0] == 0
        # the same table without tail tracking (a key set without the tag column) and with the tags as a constant cell
        assert verify(lib, c, t, wc, has_tail=False)[1] == verify(lib, c, t, wc, has_tail=False)[0], name
        for const in (STACK, START):
            got = verify(lib, c, const, wc)
            assert got[1] == got[0], (name, const, got)
    assert n_irregular > 30


def test_emu_typed_dense_verify_wide_counter(lib):
    """an 8-byte counter beyond 2^32 and at 2^64 - 1 (no successor): same verdict in both forms"""
    c, t = table(12, 3, base=(1 << 40) - 5)
    assert verify(lib, c, t, 8) == ((1, 12), (1, 12))
    c = np.array([0xFFFFFFFFFFFFFFFE, 0xFFFFFFFFFFFFFFFF, 0], dtype=np.uint64)
    got = verify(lib, c, np.full(3, STACK, dtype=np.uint8), 8)
    assert got[0] == got[1] and got[0][0] == 0
