"""GPU checks of the EVM check's index phase (api.cu check_evm): one k_pos_prep for the bytecode and rw indexes, the
rw verify next to the step sort, and the hash parts built only after the flags are read back.  Every verdict is
compared with the CPU oracle, across sequences of checks in one context that flip a table between positional and
irregular, so that a stale flag, a stale heads entry or a wrong hash-part state shows up as a wrong verdict."""
import numpy as np
import pytest

import oracle_lib
from zkevm_specs_b200 import native, packing, synth
from zkevm_specs_b200.evm_circuit import main as evm_main
from zkevm_specs_b200.evm_circuit.table import fixed_table_matrix

pytestmark = pytest.mark.gpu

START = 1  # rw table tag of the Start padding rows


def _evm(ctx, S, invalidate):
    if invalidate:
        ctx.invalidate_indexes()
    return ctx.check(native.CIRCUIT_EVM, 0, S.shape[1] - 1, 0, 0)


# rw table storages: narrow counter of 4 bytes (tag column as measured: a constant cell or 1 byte) and the type widths
# (counter 8 bytes, tag 1 byte) take the typed dense verify; 2-byte counters and canonical cells the generic one
RW_STORAGES = ("counter4", "typed", "measured", "canonical")


def _upload_rw(ctx, R, storage):
    if storage == "counter4":  # the bench's layout: counter 4 bytes, every other column at its measured width
        ws = [int(x) for x in packing.pack_matrix(R).widths]
        ws[0] = max(ws[0], 4)
        ctx.upload_table_packed(native.TABLE_RW, packing.pack_matrix(R, widths=ws))
    elif storage == "typed":
        ctx.upload_table_packed(native.TABLE_RW, packing.pack_matrix(R, min_widths=packing.TYPE_WIDTHS["rw_table"]))
    elif storage == "measured":
        ctx.upload_table_packed(native.TABLE_RW, packing.pack_matrix(R))
    else:
        ctx.upload_table(native.TABLE_RW, R)


def _with_start_tail(R, k):
    """R followed by k Start padding rows whose rw_counters restart at 1 (a dense head + a dense tail)"""
    T = np.zeros((R.shape[0], k, 4), dtype=np.uint64)
    T[0, :, 0] = np.arange(1, k + 1, dtype=np.uint64)
    T[2, :, 0] = START
    return np.ascontiguousarray(np.concatenate([R, T], axis=1))


def _assert_oracle(got, want, what):
    ff, fc = got
    off, ofc = want
    assert np.array_equal(ff, off) and np.array_equal(fc, ofc), (what, np.nonzero(ff != off)[0][:8].tolist())


@pytest.mark.parametrize("invalidate", [False, True])
def test_positional_irregular_positional_rw_in_one_context(invalidate):
    """regular rw table, rows permuted, a corrupted value, a dense head + Start tail, regular again: each in every rw
    storage (typed and generic dense verify), every verdict == oracle"""
    fixed = fixed_table_matrix()
    w = synth.evm_trace(300, seed=7)
    S, B, R = w["steps"], w["bytecode"], w["rw"]
    rng = np.random.default_rng(3)
    Rp = np.ascontiguousarray(R[:, rng.permutation(R.shape[1])])
    Rc = R.copy()
    Rc[8, int(rng.integers(R.shape[1])), 0] ^= np.uint64(4)
    Rt = _with_start_tail(R, 37)
    ctx = native.Context(0)
    evm_main.upload_fixed_table(ctx)
    ctx.upload_bytecode_table_from_code(**w["bytecode_src"])
    ctx.upload_columns_packed(native.CIRCUIT_EVM, packing.pack_matrix(S))
    want = {}
    n_fail = 0
    for name, rw in (("regular", R), ("permuted", Rp), ("corrupt", Rc), ("start tail", Rt), ("permuted", Rp), ("regular", R)):
        if name not in want:
            want[name] = oracle_lib.check_evm(S, B, rw, fixed)
        for storage in RW_STORAGES:
            _upload_rw(ctx, rw, storage)
            got = _evm(ctx, S, invalidate)
            _assert_oracle(got, want[name], (name, storage, invalidate))
            # the same tables once more: without invalidate_indexes() the indexes are reused as they are
            _assert_oracle(_evm(ctx, S, invalidate), want[name], (name, storage, invalidate, "again"))
            n_fail += bool((got[0] != native.PASS).any())
    assert n_fail == len(RW_STORAGES)  # the corrupted table fails in every storage; the others pass


def test_duplicate_hash_bytecode_table_between_regular_ones():
    """two contracts with one code hash: the heads build clears the bytecode flag, the hash part is built after the
    read-back; before and after it the regular table takes the positional path again (heads entries reset)"""
    fixed = fixed_table_matrix()
    w = synth.evm_trace(32, seed=4)
    src = w["bytecode_src"]
    n = len(src["code"])
    other = src["code"] ^ np.uint8(1)
    dup = {"code": np.concatenate([src["code"], other]),
           "is_code_bits": np.packbits(np.concatenate([np.unpackbits(src["is_code_bits"], bitorder="little")[:n]] * 2), bitorder="little"),
           "code_offsets": np.array([0, n, 2 * n], dtype=np.uint64),
           "hashes": np.concatenate([src["hashes"], src["hashes"]])}
    second = w["bytecode"].copy()
    second[5, 1:, 0] = other.astype(np.uint64)
    dup_table = np.ascontiguousarray(np.concatenate([w["bytecode"], second], axis=1))
    want_dup = oracle_lib.check_evm(w["steps"], dup_table, w["rw"], fixed)
    want_reg = oracle_lib.check_evm(w["steps"], w["bytecode"], w["rw"], fixed)
    assert (want_dup[0] != native.PASS).any() and (want_reg[0] == native.PASS).all()
    ctx = native.Context(0)
    evm_main.upload_fixed_table(ctx)
    ctx.upload_table_packed(native.TABLE_RW, packing.pack_matrix(w["rw"]))
    ctx.upload_columns_packed(native.CIRCUIT_EVM, packing.pack_matrix(w["steps"]))
    for invalidate in (False, True):
        for step in ("reg-code", "dup-code", "reg-code", "dup-table", "reg-table", "dup-code", "reg-code"):
            kind, how = step.split("-")
            if how == "code":
                ctx.upload_bytecode_table_from_code(**(src if kind == "reg" else dup))
            else:
                ctx.upload_table(native.TABLE_BYTECODE, w["bytecode"] if kind == "reg" else dup_table)
            _assert_oracle(_evm(ctx, w["steps"], invalidate), want_reg if kind == "reg" else want_dup, (step, invalidate))


@pytest.mark.parametrize("permute", [True, False])
def test_copy_check_after_evm_check_shares_the_rw_index(permute):
    """an EVM check over an (irregular or regular) rw table, then a copy-circuit check that looks up the SAME rw index
    without a rebuild: it must find the hash part the EVM check built after its read-back (or the positional path)"""
    fixed = fixed_table_matrix()
    c = synth.copy_events(8, 64, seed=9)
    R = c["rw"]
    order = np.random.default_rng(5).permutation(R.shape[1]) if permute else np.arange(R.shape[1])
    Rp = np.ascontiguousarray(R[:, order])
    Rf = np.ascontiguousarray(c["rw_flags"][order])
    e = synth.evm_trace(64, seed=3)
    ctx = native.Context(0)
    ctx.set_challenge(native.CHALLENGE_KECCAK, packing.cell_to_int(c["r"]))
    evm_main.upload_fixed_table(ctx)
    ctx.upload_bytecode_table_from_code(**e["bytecode_src"])
    ctx.upload_table(native.TABLE_RW, Rp, flags=Rf)
    ctx.upload_table(native.TABLE_TX, c["tx"], flags=c["tx_flags"])
    ctx.upload_columns(native.CIRCUIT_EVM, e["steps"])
    ctx.upload_columns(native.CIRCUIT_COPY, c["copy"], flags=c["copy_flags"])
    for rnd in range(2):
        got = ctx.check(native.CIRCUIT_EVM, 0, e["steps"].shape[1] - 1, 0, 0)
        _assert_oracle(got, oracle_lib.check_evm(e["steps"], e["bytecode"], Rp, fixed), ("evm", permute, rnd))
        v = dict(c)
        v["rw"], v["rw_flags"] = Rp, Rf
        got = ctx.check(native.CIRCUIT_COPY, 0, c["copy"].shape[1], 0, native.FLAG_WRAP)
        want = oracle_lib.check_copy(v, c["r"])
        assert (want[0] == native.PASS).all()
        _assert_oracle(got, want, ("copy", permute, rnd))
    # copy first, then EVM: the copy check builds the index (conditional hash part), the EVM check reuses it
    ctx.invalidate_indexes()
    _assert_oracle(ctx.check(native.CIRCUIT_COPY, 0, c["copy"].shape[1], 0, native.FLAG_WRAP), want, ("copy first", permute))
    got = ctx.check(native.CIRCUIT_EVM, 0, e["steps"].shape[1] - 1, 0, 0)
    _assert_oracle(got, oracle_lib.check_evm(e["steps"], e["bytecode"], Rp, fixed), ("evm after copy", permute))


def test_two_contexts_alternate_like_the_e2e_path():
    """two contexts on two streams, checks alternating with invalidate_indexes(), one regular and one irregular rw
    table: each context keeps its own flags, heads index and hash parts"""
    import torch

    fixed = fixed_table_matrix()
    ws = [synth.evm_trace(200, seed=11), synth.evm_trace(200, seed=12)]
    rng = np.random.default_rng(8)
    rws = [ws[0]["rw"], np.ascontiguousarray(ws[1]["rw"][:, rng.permutation(ws[1]["rw"].shape[1])])]
    wants = [oracle_lib.check_evm(w["steps"], w["bytecode"], r, fixed) for w, r in zip(ws, rws)]
    ctxs = [native.Context(0), native.Context(0)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for ctx, w, r in zip(ctxs, ws, rws):
        evm_main.upload_fixed_table(ctx)
        ctx.upload_bytecode_table_from_code(**w["bytecode_src"])
        ctx.upload_table_packed(native.TABLE_RW, packing.pack_matrix(r))
        ctx.upload_columns_packed(native.CIRCUIT_EVM, packing.pack_matrix(w["steps"]))
    torch.cuda.synchronize()
    for rnd in range(4):
        for k in (0, 1):
            ctxs[k].invalidate_indexes()
            ctxs[k].check_async(native.CIRCUIT_EVM, 0, ws[k]["steps"].shape[1] - 1, 0, 0, streams[k].cuda_stream)
        for k in (0, 1):
            _assert_oracle(ctxs[k].fetch_result(native.CIRCUIT_EVM, streams[k].cuda_stream), wants[k], (rnd, k))
