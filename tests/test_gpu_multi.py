"""Two-GPU test of the C-ABI collective zk_allreduce_results (NCCL all-gather of the result vectors +
fold kernel) through the library's own communicator plumbing (zk_nccl_unique_id / zk_nccl_comm_init):
row-sharded EVM steps and state rows, sharded + reduced == whole circuit on one GPU == oracle.
Needs 2 GPUs; skipped on a machine with fewer."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = textwrap.dedent(
    """
    import os, sys
    sys.path.insert(0, os.path.join(%r, "tests")); sys.path.insert(0, %r)
    import numpy as np, torch, torch.distributed as dist
    import oracle_lib
    from zkevm_specs_b200 import native, packing, synth
    from zkevm_specs_b200.evm_circuit.table import fixed_table_matrix
    dist.init_process_group("gloo")                       # only ships the 128-byte NCCL id
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(rank)
    ctx = native.Context(rank)
    box = [ctx.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    ctx.nccl_init(world, rank, box[0])
    # ---- EVM steps: two corruptions, one per shard
    w = synth.evm_trace(64, seed=11)
    S = w["steps"].copy()
    n = S.shape[1] - 1
    S[9, n - 20, 0] += np.uint64(1)     # gas corruption in the last shard
    S[1, 5, 0] += np.uint64(1)          # rw_counter corruption in rank 0's shard
    fixed = fixed_table_matrix()
    lo, hi = rank * n // world, (rank + 1) * n // world
    ctx.upload_table(native.TABLE_FIXED, fixed)
    ctx.upload_bytecode_table_from_code(**w["bytecode_src"])
    ctx.upload_table_packed(native.TABLE_RW, packing.pack_matrix(w["rw"]))
    ctx.upload_columns(native.CIRCUIT_EVM, np.ascontiguousarray(S[:, lo : hi + 1]))
    ctx.check_async(native.CIRCUIT_EVM, 0, hi - lo, lo, 0)
    ctx.allreduce_results(native.CIRCUIT_EVM)
    ff, fc = ctx.fetch_result(native.CIRCUIT_EVM)
    whole, wc = oracle_lib.check_evm(S, w["bytecode"], w["rw"], fixed)
    assert np.array_equal(ff, whole), (rank, ff[ff != whole], whole[ff != whole])
    assert np.array_equal(fc, wc)
    assert (whole != 0xFFFFFFFF).sum() >= 2
    # ---- state rows: halos on both sides, one corruption per shard
    st = synth.state_rows(1 << 12, seed=5)
    R = st["rows"].copy()
    nr = R.shape[1]
    R[50, 100, 0] ^= np.uint64(1)       # value.lo of row 100
    R[50, nr - 7, 0] ^= np.uint64(1)
    b, e = rank * nr // world, (rank + 1) * nr // world
    idx = np.arange(b - 1, e + 1) %% nr
    ctx.upload_table(native.TABLE_MPT, st["mpt"])
    ctx.upload_columns(native.CIRCUIT_STATE, np.ascontiguousarray(R[:, idx]), flags=st["flags"][idx])
    ctx.check_async(native.CIRCUIT_STATE, 1, 1 + e - b, b - 1, 0)
    ctx.allreduce_results(native.CIRCUIT_STATE)
    ff, fc = ctx.fetch_result(native.CIRCUIT_STATE)
    whole, wc = oracle_lib.check_state(R, st["flags"], st["mpt"])
    assert np.array_equal(ff, whole), (rank, np.nonzero(ff != whole))
    assert np.array_equal(fc, wc)
    assert (whole != 0xFFFFFFFF).any()
    ctx.nccl_destroy()
    if rank == 0:
        print("OK")
    dist.destroy_process_group()
    """
)


@pytest.mark.gpu
def test_c_abi_collective_two_gpus(tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % (ROOT, ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29541", str(script)],
                         capture_output=True, text=True, env=env, timeout=900)
    assert out.returncode == 0 and "OK" in out.stdout, out.stdout[-2000:] + out.stderr[-3000:]
