"""Withdrawal circuit on one GPU: device witness assignment, lookup-index build and check kernel, at the sizes given.

    python tools/bench_withdrawal.py [--rows 20 22] [--max16] [--reps 7] [--label NAME]

Prints one JSON line per size.  Every number is measured in this run:
- assign_ms: zk_assign_withdrawal_circuit (records host -> device, RLP, Keccak-256, RLC, the 8-cell rows and the keccak
  table), host clock around the call and a device synchronise, median of --reps;
- index_ms / check_ms: zk_enable_timing events of a zk_check_async with the indexes dropped first (keccak 5-column,
  MPT 12-column, block 3-column), median of --reps;
- rows_per_s: rows / check_ms;
- algo_bytes_per_row: the 8 row cells plus the looked-up keccak row (5 cells) and MPT row (12 cells), 32 B each;
- hbm_fraction: algo_bytes_per_row * rows / check time over 7.7 TB/s (HGX B200 data sheet, one GPU) — the memory bound;
  a fraction well below 1 means the kernel is bound by something else (its Fr arithmetic and probe latency);
- gpu, power_limit, sm_clock: nvidia-smi, read in the same run.
At --max16 (MAX_WITHDRAWALS = 16, the per-payload cap on Ethereum) the figures are end-to-end latencies of one assign
and one check (launch-bound), not rates.  The working set at 2^20 rows is ~0.8 GB, well past the 126 MB L2."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from zkevm_specs_b200 import native, synth  # noqa: E402

HBM_BPS = 7.7e12
ALGO_BYTES_PER_ROW = (8 + 5 + 12) * 32


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, pl, sm, smax = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": pl, "sm_clock": sm, "sm_clock_max": smax}


def run(log_n, max16, reps, label):
    n = 16 if max16 else 1 << log_n
    ctx = native.Context(0)
    ctx.set_challenge(native.CHALLENGE_KECCAK, 0x0DDBA11CAFE + n)
    s = synth.withdrawals(n, n, seed=log_n, ctx=ctx)  # assigns, uploads the MPT and block tables
    ctx.enable_timing(True)

    def sync():
        torch.cuda.synchronize()

    assign = []
    for k in range(reps + 2):
        sync()
        t0 = time.perf_counter()
        ctx.assign_withdrawal_circuit(s["records"], n)
        sync()
        assign.append((time.perf_counter() - t0) * 1e3)
    idx, chk, e2e = [], [], []
    ff = None
    for k in range(reps + 2):
        ctx.invalidate_indexes()
        sync()
        t0 = time.perf_counter()
        ctx.check_async(native.CIRCUIT_WITHDRAWAL, 0, n, 0, 0)
        ff, _ = ctx.fetch_result(native.CIRCUIT_WITHDRAWAL)
        e2e.append((time.perf_counter() - t0) * 1e3)
        a, b = ctx.last_timing()
        idx.append(a)
        chk.append(b)
    assert (ff == native.PASS).all(), native.first_failure(ff, native.CIRCUIT_WITHDRAWAL)
    med = lambda v: float(np.median(v[2:]))  # noqa: E731  (the first two passes warm up)
    out = {"label": label, "rows": n, "assign_ms": med(assign), "index_ms": med(idx), "check_ms": med(chk),
           "check_e2e_ms": med(e2e), "reps": reps, "spread_check_ms": float(np.ptp(chk[2:])), **gpu_info()}
    if max16:
        out["note"] = "MAX_WITHDRAWALS = 16: end-to-end latencies, launch-bound; no rate is stated"
    else:
        out.update({"rows_per_s": n / (out["check_ms"] * 1e-3), "algo_bytes_per_row": ALGO_BYTES_PER_ROW,
                    "hbm_fraction": ALGO_BYTES_PER_ROW * n / (out["check_ms"] * 1e-3) / HBM_BPS,
                    "bound": "memory: algorithmic bytes over 7.7 TB/s"})
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="*", default=[20, 22], help="log2 of the row counts")
    ap.add_argument("--max16", action="store_true", help="also run MAX_WITHDRAWALS = 16")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--label", default=os.environ.get("ZKCHECK_LIB", "in-tree"))
    a = ap.parse_args()
    for log_n in a.rows:
        print(json.dumps(run(log_n, False, a.reps, a.label)), flush=True)
    if a.max16:
        print(json.dumps(run(0, True, a.reps, a.label)), flush=True)


if __name__ == "__main__":
    main()
