#!/usr/bin/env python
"""bench.py — constraint-rows/sec of the zkevm-specs hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload W] [--scaling S]
                    [--dump-outputs DIR]

Main line (the bench contract): workload `evm` = BASELINE cfg2's generator scaled to the metric's 2^20
rows — per GPU 2^18 groups `PUSH32 b, PUSH32 a, {ADD,SUB,MUL,DIV,MOD}, POP` = 2^20 execution steps,
17.8 M bytecode-table rows, 1.57 M rw-table rows, fixed table 224,490 rows (synthetic, seeded).
One "step" of the bench = one pass of the whole hot path over that witness: build the lookup indexes
of the bytecode / rw tables on the device, then check every execution step.
  value    : rows/s with all inputs resident in HBM (CUDA events on the launching stream)
  e2e      : rows/s through the C-ABI with HOST (pinned) buffers: H2D of tables + steps, index build,
             check, D2H of the result vector, all inside the timed region
  roofline : algorithmic bytes of the check phase / its device time vs MEASURED_PEAKS.json, next to the
             honest denominators: stored bytes (what sits in HBM) and DRAM traffic (ncu capture of THIS
             build, profiles/, matched by source hash — null when the sources changed since the capture)
  cpu_baseline : the CPU oracle (a C port of the reference algorithm; the reference itself is pure
             Python and absent on this box) on a bounded sample of the same workload
Extra objects on the same line (`--no-extras` skips them; they are not inside the main timed region):
  typed          : the same check with data-independent column widths (packing.TYPE_WIDTHS)
  circuits       : BASELINE cfg3 (state 2^18 rows), cfg4's copy circuit (2^20 rows), the bytecode circuit
                   (2^19 rows) and the public-inputs circuit (64 txs, 2^18 calldata bytes: 2.9e5 rows) on
                   canonical 32-byte cells, each with its own roofline
  strong_scaling : ONE 2^20-step witness split over the N ranks (tables replicated, step shards with
                   a halo step, one collective) — north_star's "2^20-row witness at 1/2/4/8 B200"
  block_trace    : the realistic variant — ONE whole-block trace (4,096 transactions over 1,024 contracts: BeginTx ..
                   STOP, EndTx each, EndBlock last) checked with the first / last step flags
  assign         : witness assignment on the device (bytecode 2^19 / state 2^18 / copy 2^20 rows from their compact host
                   inputs) and the check of the narrow rows it leaves
  cfg4 / cfg5    : copy circuit 2^20 rows and the super circuit (evm + state + copy + bytecode, 2^22 rows
                   in total) row-sharded over the N ranks
Multi-GPU (torchrun): rows are sharded, tables replicated, then ONE collective on the result vectors
(zk_allreduce_results: NCCL all-gather + fold); main line scaling "weak" (own 2^20-step shard per rank).
"""
import argparse
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only, and a benchmark run leaves nothing in it

N_CELLS_STEP, N_CELLS_RW, N_CELLS_BYTECODE = 13, 14, 6
DTYPE = "u64 limbs (BN254 Fr, 254-bit modular)"


class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons through NVML while the timed region runs (NVML is
    initialised in the constructor, before the region; one sample is taken at start and one at
    stop so that even a 10 ms region is covered)"""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self._stop_evt = index, [], set(), threading.Event()
        self.max_mhz, self._nv, self._h, self._names = None, None, None, {}
        try:
            import pynvml as nv

            nv.nvmlInit()
            self._nv, self._h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
            self._names = {
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            }
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def _sample(self):
        nv = self._nv
        if nv is None:
            return
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
            for bit, nm in self._names.items():
                if r & bit:
                    self.reasons.add(nm)
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def run(self):
        while not self._stop_evt.is_set():
            self._sample()
            time.sleep(0.005)

    def stop(self):
        self._sample()  # still under load: the caller stops the sampler before synchronising
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def algorithmic_bytes(n_steps, n_rw, n_bytecode, n_constraints):
    """SURVEY.md §8d: every witness/table cell once at canonical 32 B; fixed table excluded."""
    return 32 * (n_steps * N_CELLS_STEP + n_rw * N_CELLS_RW + n_bytecode * N_CELLS_BYTECODE) + 4 * n_constraints


def source_hash() -> str:
    """hash of the CUDA sources: ties a profiles/ capture to the build it was taken from"""
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "zkevm-specs_b200", "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(csrc, f), "rb").read())
    return h.hexdigest()[:16]


def load_capture():
    """profiles/current_capture.json: {"source_hash", "dram_bytes_per_check", "kernels": {...}} written by
    tools/traffic_from_ncu.py from an `ncu --set full` capture of this command; used only when its
    source_hash matches the sources on disk"""
    try:
        c = json.load(open(os.path.join(ROOT, "profiles", "current_capture.json")))
        return c if c.get("source_hash") == source_hash() else None
    except Exception:  # noqa: BLE001
        return None


def _cpu_port_worker(args):
    sample_groups, seed = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    from zkevm_specs_b200 import synth
    from zkevm_specs_b200.evm_circuit.table import fixed_table_matrix

    w = synth.evm_trace(sample_groups, seed=seed)
    fixed = fixed_table_matrix()
    oracle_lib.lib()
    t0 = time.perf_counter()
    ff, _ = oracle_lib.check_evm(w["steps"], w["bytecode"], w["rw"], fixed)
    dt = time.perf_counter() - t0
    assert (ff == 0xFFFFFFFF).all(), "oracle rejected the synthetic witness"
    return w["n_steps"], dt


def cpu_port(sample_groups: int, seed: int, threads: int):
    """time the CPU oracle (C port of the reference algorithm) on a bounded sample.  threads > 1:
    that many processes each check their own sample of the same size concurrently (the reference
    has no parallelism of its own; rows are independent, so this is how it would use the cores);
    returns (total rows, wall seconds of the slowest worker)"""
    if threads <= 1:
        return _cpu_port_worker((sample_groups, seed))
    import multiprocessing as mp

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib

    oracle_lib.lib()  # build once before forking
    with mp.get_context("fork").Pool(threads) as pool:
        res = pool.map(_cpu_port_worker, [(sample_groups, seed + k) for k in range(threads)])
    # generation time is outside; use the max of the measured check times (they overlap)
    return sum(r[0] for r in res), max(r[1] for r in res)


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's algorithm on the host cores.  The reference is pure
    Python and /root/reference is absent on the GPU box, so this times the C port (oracle/) with
    one process per core (rows are independent: that is how the reference would use the cores).
    A step = every core checks its own bounded sample of the cfg2 trace; the sample is sized from
    a calibration step so that the K timed steps end within ~2 minutes."""
    if rank != 0:
        return
    import multiprocessing as mp

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib

    oracle_lib.lib()  # build once before forking
    cores = os.cpu_count() or 1
    with mp.get_context("fork").Pool(cores) as pool:
        def step(groups, seed0):
            res = pool.map(_cpu_port_worker, [(groups, seed0 + k) for k in range(cores)])
            return sum(r[0] for r in res), max(r[1] for r in res)

        n, dt = step(256, 2)  # calibration (also the first warm-up)
        rate = n / dt  # rows/s over all cores
        budget = min(3.0, 120.0 / max(1, args.steps))  # seconds per timed step
        sample_groups = int(min(args.ref_groups, max(64, rate * budget / cores / 4)))
        for _ in range(max(0, args.warmup - 1)):
            step(sample_groups, 2)
        rows = secs = 0.0
        for k in range(args.steps):
            n, dt = step(sample_groups, 2 + k)
            rows += n
            secs += dt
    v = rows / secs
    line = {
        "impl": "reference", "metric": "constraint-rows/sec", "value": v, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
        "data": "synthetic",
        "config": {"workload": f"evm_circuit ADD/SUB/MUL/DIV/MOD trace (cfg2 generator), bounded sample: {cores} x "
                               f"{4 * sample_groups} steps per bench step (same generator as the CUDA arm)", "seed": 2},
        "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port",
                         "sample": f"{cores} processes x {4 * sample_groups} steps each per bench step, C oracle incl. "
                                   "sorted-index build of all tables"},
        "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


class Harness:
    """device context + timing helpers shared by every workload of one rank"""

    def __init__(self, rank, world, local):
        import torch
        import torch.distributed as dist

        from zkevm_specs_b200 import native

        self.torch, self.dist, self.native = torch, dist, native
        self.rank, self.world, self.local = rank, world, local
        torch.cuda.set_device(local)
        if world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        self.ctx = native.Context(local)
        self.stream = torch.cuda.current_stream().cuda_stream
        if world > 1:  # the library's own communicator (zk_nccl_*): id drawn on rank 0, shipped through torch
            box = [self.ctx.nccl_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            self.ctx.nccl_init(world, rank, box[0])
        self.peak = 6650.0
        self.peak_source = "fallback 6.65 TB/s"
        try:
            self.peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
            self.peak_source = "MEASURED_PEAKS.json (burst copy)"
        except Exception:  # noqa: BLE001
            pass

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def timed(self, fn, k):
        """device time of k calls of fn, barrier + synchronize on both sides, max over ranks (ms)"""
        torch = self.torch
        self.sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        self.sync_all()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device=f"cuda:{self.local}")
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def check_pass(self, circuit):
        ff, _ = self.ctx.fetch_result(circuit, self.stream)
        assert (ff == self.native.PASS).all(), f"witness rejected: {self.native.first_failure(ff, circuit)}"

    def phases(self, circuit, row_begin, row_end, row_base, flags, reps):
        """(index build ms, check ms) of one check, device-timed inside the library, mean of reps"""
        ctx = self.ctx
        ctx.enable_timing(True)
        idx, chk = [], []
        for _ in range(reps):
            ctx.invalidate_indexes()
            ctx.check_async(circuit, row_begin, row_end, row_base, flags, self.stream)
            a, b = ctx.last_timing()
            idx.append(a)
            chk.append(b)
        ctx.enable_timing(False)
        return float(np.mean(idx)), float(np.mean(chk))

    def sharded_pass(self, circuit, row_begin, row_end, row_base, flags, reps):
        """whole pass of one (sharded) circuit: index builds + check + the one collective; returns ms per pass,
        max over ranks"""
        ctx = self.ctx

        def one():
            ctx.invalidate_indexes()
            ctx.check_async(circuit, row_begin, row_end, row_base, flags, self.stream)
            if self.world > 1:
                ctx.allreduce_results(circuit, self.stream)

        for _ in range(3):
            one()
        self.check_pass(circuit)
        return self.timed(one, reps) / reps


def dump_outputs(out_dir, first_fail, fail_count):
    """the result vectors of the last timed step, as a caller of the check receives them, in float64 (exact: first_fail
    holds rows < 2^32, fail_count row counts < 2^53)"""
    assert (fail_count < (1 << 53)).all()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "first_fail.npy"), first_fail.astype(np.float64))
    np.save(os.path.join(out_dir, "fail_count.npy"), fail_count.astype(np.float64))


def shard(n, rank, world):
    b = n * rank // world
    return b, n * (rank + 1) // world


def take_rows(m, idx):
    return np.ascontiguousarray(np.take(m, idx, axis=1))


def roofline_of(h, chk_ms, bytes_alg, stored=None, **extra):
    ach = bytes_alg / (chk_ms / 1e3) / 1e9
    d = {"bound": "hbm", "achieved": ach, "peak": h.peak, "unit": "GB/s", "frac": ach / h.peak, "traffic": None,
         "kernel_ms": chk_ms, "algorithmic_bytes": int(bytes_alg), "peak_source": h.peak_source}
    if stored is not None:
        d["stored_bytes"] = int(stored)
        d["stored_frac"] = stored / (chk_ms / 1e3) / 1e9 / h.peak
    d.update(extra)
    return d


# ------------------------------------------------------------------------------------------------
# row circuits (canonical storage), optionally row-sharded over the ranks
def bench_state(h, n_rows, reps, seed=3):
    from zkevm_specs_b200 import synth
    native = h.native
    w = synth.state_rows(n_rows, seed=seed)
    n = w["rows"].shape[1]
    h.ctx.upload_table(native.TABLE_MPT, w["mpt"], stream=h.stream)
    b, e = shard(n, h.rank, h.world)
    if h.world == 1:
        h.ctx.upload_columns(native.CIRCUIT_STATE, w["rows"], flags=w["flags"], stream=h.stream)
        rng = (0, n, 0, native.FLAG_WRAP)
    else:  # rows b-1 .. e (rotations -1, +1), wrapping at the ends of the circuit
        idx = np.arange(b - 1, e + 1) % n
        h.ctx.upload_columns(native.CIRCUIT_STATE, take_rows(w["rows"], idx), flags=w["flags"][idx], stream=h.stream)
        rng = (1, 1 + e - b, b - 1, 0)
    ms = h.sharded_pass(native.CIRCUIT_STATE, *rng, reps)
    i_ms, c_ms = h.phases(native.CIRCUIT_STATE, *rng, min(reps, 10))
    byt = 32 * ((e - b) * 57 + w["mpt"].shape[1] * 12)
    return {"circuit": "state", "rows": n, "rows_per_gpu": e - b, "ms_per_pass": ms, "rows_per_s": n / (ms / 1e3),
            "index_ms": i_ms, "roofline": roofline_of(h, c_ms, byt, kernel="k_check_state<L_CANON>")}


def bench_copy(h, n_events, length, reps, seed=4):
    from zkevm_specs_b200 import synth
    native = h.native
    w = synth.copy_events(n_events, length, seed=seed)
    n = w["copy"].shape[1]
    ctx = h.ctx
    ctx.set_challenge(native.CHALLENGE_KECCAK, sum(int(w["r"][k]) << (64 * k) for k in range(4)))
    ctx.upload_table(native.TABLE_RW, w["rw"], flags=w["rw_flags"], stream=h.stream)
    ctx.upload_table(native.TABLE_BYTECODE, w["bytecode"], stream=h.stream)
    ctx.upload_table(native.TABLE_TX, w["tx"], flags=w["tx_flags"], stream=h.stream)
    b, e = shard(n, h.rank, h.world)
    if h.world == 1:
        ctx.upload_columns(native.CIRCUIT_COPY, w["copy"], flags=w["copy_flags"], stream=h.stream)
        rng = (0, n, 0, native.FLAG_WRAP)
    else:  # rows b .. e+1 (rotations +1, +2)
        idx = np.arange(b, e + 2) % n
        ctx.upload_columns(native.CIRCUIT_COPY, take_rows(w["copy"], idx), flags=w["copy_flags"][idx], stream=h.stream)
        rng = (0, e - b, b, 0)
    ms = h.sharded_pass(native.CIRCUIT_COPY, *rng, reps)
    i_ms, c_ms = h.phases(native.CIRCUIT_COPY, *rng, min(reps, 10))
    byt = 32 * ((e - b) * 20 + w["rw"].shape[1] * 14 + w["tx"].shape[1] * 5)
    return {"circuit": "copy", "rows": n, "rows_per_gpu": e - b, "rw_rows": int(w["rw"].shape[1]), "tx_rows": int(w["tx"].shape[1]),
            "ms_per_pass": ms, "rows_per_s": n / (ms / 1e3), "index_ms": i_ms,
            "roofline": roofline_of(h, c_ms, byt, kernel="k_check_copy_small<L_CANON> (+ k_check_copy_general over deferred warps)")}


def bench_bytecode(h, k, reps):
    from zkevm_specs_b200 import synth
    native = h.native
    w = synth.bytecode_circuit_rows(k, 8)
    n = w["rows"].shape[1]
    ctx = h.ctx
    ctx.set_challenge(native.CHALLENGE_KECCAK, sum(int(w["r"][k_]) << (64 * k_) for k_ in range(4)))
    ctx.upload_table(native.TABLE_PUSH, w["push"], stream=h.stream)
    ctx.upload_table(native.TABLE_KECCAK, w["keccak"], stream=h.stream)
    b, e = shard(n, h.rank, h.world)
    if h.world == 1:
        ctx.upload_columns(native.CIRCUIT_BYTECODE, w["rows"], stream=h.stream)
        rng = (0, n, 0, native.FLAG_WRAP)
    else:  # rows b .. e (rotation +1)
        idx = np.arange(b, e + 1) % n
        ctx.upload_columns(native.CIRCUIT_BYTECODE, take_rows(w["rows"], idx), stream=h.stream)
        rng = (0, e - b, b, 0)
    ms = h.sharded_pass(native.CIRCUIT_BYTECODE, *rng, reps)
    i_ms, c_ms = h.phases(native.CIRCUIT_BYTECODE, *rng, min(reps, 10))
    return {"circuit": "bytecode", "rows": n, "rows_per_gpu": e - b, "ms_per_pass": ms, "rows_per_s": n / (ms / 1e3),
            "index_ms": i_ms, "roofline": roofline_of(h, c_ms, 32 * (e - b) * 12, kernel="k_check_bytecode<L_CANON>")}


def bench_pi(h, max_txs, max_calldata, max_wd, reps, seed=7):
    """public-inputs circuit (pi_circuit.check_row): one row per raw public-input byte, row-sharded over the ranks"""
    from zkevm_specs_b200 import pi_circuit as pc
    from zkevm_specs_b200 import synth
    native, ctx = h.native, h.ctx
    t0 = time.perf_counter()
    w = pc.public_data2witness(synth.pi_public_data(max_txs * 3 // 4, max_calldata, max_wd, seed=seed), max_txs, max_calldata, max_wd)
    gen_s = time.perf_counter() - t0
    n = w.cells.shape[1]
    K, G = w.keccak_table.matrix(), w.gas_matrix()
    ctx.set_challenge(native.CHALLENGE_PI_KECCAK, pc.keccak_rand.n)
    ctx.set_challenge(native.CHALLENGE_PI_BYTE_BASE, pc.byte_pow_base.n)
    ctx.set_challenge(native.PARAM_PI_CIRCUIT_LEN, w.circuit_len)
    ctx.upload_table(native.TABLE_KECCAK, K, stream=h.stream)
    ctx.upload_table(native.TABLE_CALLDATA_GAS, G, stream=h.stream)
    b, e = shard(n, h.rank, h.world)
    if h.world == 1:
        ctx.upload_columns(native.CIRCUIT_PI, w.cells, stream=h.stream)
        rng = (0, n, 0, native.FLAG_WRAP)
    else:  # rows b .. e (rotation +1)
        ctx.upload_columns(native.CIRCUIT_PI, take_rows(w.cells, np.arange(b, e + 1) % n), stream=h.stream)
        rng = (0, e - b, b, 0)
    ms = h.sharded_pass(native.CIRCUIT_PI, *rng, reps)
    i_ms, c_ms = h.phases(native.CIRCUIT_PI, *rng, min(reps, 10))
    byt = 32 * ((e - b) * 28 + K.shape[1] * 5 + G.shape[1] * 3)
    return {"circuit": "pi", "rows": n, "rows_per_gpu": e - b, "gas_table_rows": int(G.shape[1]), "ms_per_pass": ms,
            "rows_per_s": n / (ms / 1e3), "index_ms": i_ms, "host_generate_s": gen_s,
            "roofline": roofline_of(h, c_ms, byt, kernel="k_check_pi<L_CANON>")}


def bench_assign(h, reps):
    """witness assignment on the device (SURVEY.md 8(f)-3): per circuit, the time from the compact HOST inputs (raw code /
    15 operation cells / copy events + bytes, pinned) to the resident witness, and the check of the narrow rows it leaves"""
    import torch
    from zkevm_specs_b200 import assign, packing, synth
    native, ctx, stream = h.native, h.ctx, h.stream
    out = {}

    def timed_pair(assign_fn, circuit, n, flags):
        for _ in range(2):
            assign_fn()
        a_ms = h.timed(assign_fn, reps) / reps
        ctx.check_async(circuit, 0, n, 0, flags, stream)
        h.check_pass(circuit)
        i_ms, c_ms = h.phases(circuit, 0, n, 0, flags, min(reps, 10))
        return a_ms, c_ms

    b = synth.bytecode_circuit_rows(19, 8)
    src = assign.bytecode_src(b["codes"])
    ctx.set_challenge(native.CHALLENGE_KECCAK, b["r_int"])
    ctx.upload_table(native.TABLE_PUSH, b["push"], stream=stream)
    ctx.upload_table(native.TABLE_KECCAK, b["keccak"], stream=stream)
    pin = {k: torch.from_numpy(v).pin_memory() for k, v in src.items()}
    a_ms, c_ms = timed_pair(lambda: ctx.assign_bytecode_circuit(19, **{k: v.numpy() for k, v in pin.items()}, stream=stream),
                            native.CIRCUIT_BYTECODE, 1 << 19, native.FLAG_WRAP)
    out["bytecode"] = {"rows": 1 << 19, "assign_ms": a_ms, "check_narrow_ms": c_ms, "h2d_bytes": int(sum(v.nbytes for v in src.values())),
                       "canonical_bytes": 32 * 12 << 19}
    s = synth.state_rows(1 << 18, seed=3)
    pm = packing.pack_matrix(assign.state_ops_from_rows(s["rows"]))
    pm.buf = torch.from_numpy(pm.buf).pin_memory().numpy()
    ctx.upload_table(native.TABLE_MPT, s["mpt"], stream=stream)
    a_ms, c_ms = timed_pair(lambda: ctx.assign_state_circuit(pm, flags=s["flags"], stream=stream), native.CIRCUIT_STATE, 1 << 18,
                            native.FLAG_WRAP)
    out["state"] = {"rows": 1 << 18, "assign_ms": a_ms, "check_narrow_ms": c_ms, "h2d_bytes": int(pm.nbytes), "canonical_bytes": 32 * 57 << 18}
    w = synth.copy_events(512, 1024)
    n = w["copy"].shape[1]
    ctx.set_challenge(native.CHALLENGE_KECCAK, w["r_int"])
    ctx.upload_table(native.TABLE_RW, w["rw"], flags=w["rw_flags"], stream=stream)
    ctx.upload_table(native.TABLE_BYTECODE, w["bytecode"], stream=stream)
    ctx.upload_table(native.TABLE_TX, w["tx"], flags=w["tx_flags"], stream=stream)
    ev, data = torch.from_numpy(w["events"]).pin_memory().numpy(), torch.from_numpy(w["data"]).pin_memory().numpy()
    a_ms, c_ms = timed_pair(lambda: ctx.assign_copy_circuit(ev, data, stream=stream), native.CIRCUIT_COPY, n, native.FLAG_WRAP)
    out["copy"] = {"rows": n, "assign_ms": a_ms, "check_narrow_ms": c_ms, "h2d_bytes": int(ev.nbytes + data.nbytes), "canonical_bytes": 32 * 20 * n}
    return out


def bench_block(h, n_txs, groups, n_contracts, reps, seed=6):
    """the realistic variant: ONE whole-block trace (synth.block_trace: BeginTx .. STOP, EndTx per transaction over
    `n_contracts` contracts, EndBlock last) checked with the first / last step flags; step-sharded over the ranks"""
    from zkevm_specs_b200 import packing, synth
    native, ctx, stream = h.native, h.ctx, h.stream
    t0 = time.perf_counter()
    w = synth.block_trace(n_txs, groups, n_contracts, seed=seed)
    gen_s = time.perf_counter() - t0
    n = w["n_steps"]
    b, e = shard(n, h.rank, h.world)
    ctx.upload_bytecode_table_from_code(**w["bytecode_src"], stream=stream)
    ctx.upload_table_packed(native.TABLE_RW, packing.pack_matrix(w["rw"]), flags=w["rw_flags"], stream=stream)
    ctx.upload_columns_packed(native.CIRCUIT_EVM, packing.pack_matrix(take_rows(w["steps"], np.arange(b, e + 1))), stream=stream)
    ctx.upload_table(native.TABLE_TX, w["tx"], flags=w["tx_flags"], stream=stream)
    ctx.upload_table(native.TABLE_BLOCK, w["block"], flags=w["block_flags"], stream=stream)
    ctx.upload_table(native.TABLE_WITHDRAWAL, w["wd"], stream=stream)
    flags = (native.FLAG_EVM_FIRST_STEP if b == 0 else 0) | (native.FLAG_EVM_LAST_STEP if e == n else 0)
    ms = h.sharded_pass(native.CIRCUIT_EVM, 0, e - b, b, flags, reps)
    i_ms, c_ms = h.phases(native.CIRCUIT_EVM, 0, e - b, b, flags, min(reps, 10))
    states = np.bincount(w["steps"][0, :n, 0].astype(np.int64), minlength=64)
    for t_, c_ in ((native.TABLE_TX, 5), (native.TABLE_BLOCK, 4)):
        ctx.upload_table(t_, np.zeros((c_, 0, 4), dtype=np.uint64), stream=stream)
    return {"workload": f"whole-block trace: {n_txs} transactions over {n_contracts} contracts of {68 * groups + 1} bytes, "
                        "verify_steps(begin_with_first_step, end_with_last_step) as ONE trace",
            "steps": n, "steps_per_gpu": e - b, "rw_rows": int(w["rw"].shape[1]), "bytecode_rows": int(w["bytecode"].shape[1]),
            "tx_level_steps": int(states[1] + states[2] + states[3] + states[4]), "ms_per_pass": ms, "rows_per_s": n / (ms / 1e3),
            "index_build_ms": i_ms, "check_ms": c_ms, "host_generate_s": gen_s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--groups", type=int, default=1 << 18, help="trace groups per GPU (4 steps each)")
    ap.add_argument("--ref-groups", type=int, default=1 << 12)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip typed / circuits / strong_scaling / cfg4 / cfg5")
    ap.add_argument("--workload", choices=["evm", "state", "copy", "bytecode", "block", "pi", "assign"], default="evm",
                    help="evm: the bench contract's line.  state / copy / bytecode: only that row circuit (canonical "
                         "storage; for profiling), printed as a JSON line of its own")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="main line under torchrun: weak = every rank checks its own 2^20-step witness; strong = ONE "
                         "2^20-step witness split over the ranks")
    ap.add_argument("--storage", choices=["adaptive", "typed", "packed", "canonical"], default="adaptive",
                    help="adaptive: the packer's default — every column at its measured minimal width, constant "
                         "columns stored once (packing.pack_matrix); typed (= packed): data-independent widths by "
                         "column type (packing.TYPE_WIDTHS); both through zk_upload_*_packed.  canonical: 32-byte "
                         "cells through zk_upload_*")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result vectors of the last one (first_fail.npy, "
                         "fail_count.npy; float64) to DIR; inputs are seeded, so runs with the same arguments compare "
                         "output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "evm"):
        ap.error("--dump-outputs applies to the main line: --impl ours --workload evm")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    h = Harness(rank, world, local)
    native, ctx, stream, dist = h.native, h.ctx, h.stream, h.dist
    from zkevm_specs_b200 import packing, synth
    from zkevm_specs_b200.evm_circuit.table import fixed_table_matrix

    if args.workload != "evm":
        reps = max(3, min(args.steps, 20))
        if args.workload == "block":
            h.ctx.upload_table(native.TABLE_FIXED, fixed_table_matrix(), stream=stream)
        d = {"state": lambda: bench_state(h, 1 << 18, reps), "copy": lambda: bench_copy(h, 512, 1024, reps),
             "bytecode": lambda: bench_bytecode(h, 19, reps), "pi": lambda: bench_pi(h, 64, 1 << 18, 16, reps), "assign": lambda: bench_assign(h, reps), "block": lambda: bench_block(h, 4096, 64, 1024, reps)}[args.workload]()
        if rank == 0:
            print(json.dumps({"workload": args.workload, "n_gpus": world, "storage": "canonical", **d}))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- synthetic witness ---------------------------------------------------------------------
    # weak: per rank its own row shard, own seed.  strong: every rank generates the SAME 2^20-step
    # witness (tables replicated) and uploads only its step shard + the halo step.
    strong = args.scaling == "strong" and world > 1
    t0 = time.perf_counter()
    w = synth.evm_trace(args.groups, seed=2 + (0 if strong else rank))
    gen_s = time.perf_counter() - t0
    n_total = w["n_steps"]
    sb, se = shard(n_total, rank, world) if strong else (0, n_total)
    n_steps = se - sb
    fixed = fixed_table_matrix()
    n_rw, n_bc = w["rw"].shape[1], w["bytecode"].shape[1]
    n_constraints = ctx.n_constraints(native.CIRCUIT_EVM)
    ctx.upload_table(native.TABLE_FIXED, fixed, stream=stream)  # circuit constant: uploaded once
    steps_m = w["steps"] if not strong else take_rows(w["steps"], np.arange(sb, se + 1))
    row_base = sb if strong else rank * n_steps
    if args.storage == "packed":
        args.storage = "typed"
    host_pack_ms = None
    if args.storage in ("adaptive", "typed"):
        t0 = time.perf_counter()
        if args.storage == "typed":
            packed = {"steps": packing.pack_matrix(steps_m, min_widths=packing.TYPE_WIDTHS["evm_steps"]),
                      "bytecode": packing.pack_matrix(w["bytecode"], min_widths=packing.TYPE_WIDTHS["bytecode_table"]),
                      "rw": packing.pack_matrix(w["rw"], min_widths=packing.TYPE_WIDTHS["rw_table"])}
            fmt = "packed columns, data-independent type widths (packing.TYPE_WIDTHS)"
        else:
            packed = {"steps": packing.pack_matrix(steps_m), "rw": packing.pack_matrix(w["rw"])}
            fmt = ("steps / rw table: packed columns, measured minimal width per column, constant columns stored "
                   "once (packing.pack_matrix default; the packing scan is host preparation, outside the timed "
                   "region: host_pack_ms).  bytecode table: the raw code bytes + 1 is_code bit per byte + 1 hash per "
                   "contract, unrolled on the device (zk_upload_bytecode_table_from_code = Bytecode.table_assignments, "
                   "typing.py:390-427), inside the timed region")
        host_pack_ms = 1e3 * (time.perf_counter() - t0)
        pinned = {k: torch.from_numpy(pm.buf).pin_memory() for k, pm in packed.items()}
        h2d_bytes = sum(pm.nbytes for pm in packed.values())
        src = None
        if "bytecode" not in packed:
            src = w["bytecode_src"]
            pinned["code"] = torch.from_numpy(src["code"]).pin_memory()
            pinned["bits"] = torch.from_numpy(src["is_code_bits"]).pin_memory()
            h2d_bytes += src["code"].nbytes + src["is_code_bits"].nbytes + src["code_offsets"].nbytes + src["hashes"].nbytes
        stored = sum(pm.nbytes for pm in packed.values()) + (42 * n_bc if src is not None else 0)
        widths = {k: [int(x) for x in pm.widths] for k, pm in packed.items()}
        if src is not None:
            widths["bytecode"] = [16, 16, 1, 4, 1, 4]  # written by k_bytecode_table_expand
        storage = {"format": fmt, "widths": widths, "stored_bytes": stored}

        def upload_inputs(ctx=ctx, stream=stream):
            if src is not None:
                ctx.upload_bytecode_table_from_code(src["code"], src["is_code_bits"], src["code_offsets"], src["hashes"],
                                                    stream=stream, ptrs=(pinned["code"].data_ptr(), pinned["bits"].data_ptr()))
            else:
                ctx.upload_table_packed(native.TABLE_BYTECODE, packed["bytecode"], stream=stream,
                                        host_ptr=pinned["bytecode"].data_ptr())
            ctx.upload_table_packed(native.TABLE_RW, packed["rw"], stream=stream, host_ptr=pinned["rw"].data_ptr())
            ctx.upload_columns_packed(native.CIRCUIT_EVM, packed["steps"], stream=stream, host_ptr=pinned["steps"].data_ptr())
    else:
        pinned = {"steps": torch.from_numpy(steps_m).pin_memory(), "bytecode": torch.from_numpy(w["bytecode"]).pin_memory(),
                  "rw": torch.from_numpy(w["rw"]).pin_memory()}
        h2d_bytes = 32 * ((n_steps + 1) * N_CELLS_STEP + n_rw * N_CELLS_RW + n_bc * N_CELLS_BYTECODE)
        storage = {"format": "canonical 32-byte cells", "stored_bytes": h2d_bytes}

        def upload_inputs(ctx=ctx, stream=stream):
            ctx.upload_table_ptr(native.TABLE_BYTECODE, n_bc, 6, pinned["bytecode"].data_ptr(), stream)
            ctx.upload_table_ptr(native.TABLE_RW, n_rw, 14, pinned["rw"].data_ptr(), stream)
            ctx.upload_columns_ptr(native.CIRCUIT_EVM, n_steps + 1, 13, pinned["steps"].data_ptr(), stream)

    def hot_path(ctx=ctx, stream=stream):
        """index builds + check of every step; + the one collective when sharded"""
        ctx.invalidate_indexes()
        ctx.check_async(native.CIRCUIT_EVM, 0, n_steps, row_base, 0, stream)
        if world > 1:
            ctx.allreduce_results(native.CIRCUIT_EVM, stream)

    upload_inputs()
    for _ in range(args.warmup):
        hot_path()
    h.check_pass(native.CIRCUIT_EVM)

    sampler = ClockSampler(local)
    sampler.start()
    launches0 = ctx.launch_count()
    ms = h.timed(hot_path, args.steps)
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *ctx.fetch_result(native.CIRCUIT_EVM, stream))
    rows_per_step = n_total if strong else world * n_steps
    value = rows_per_step * args.steps / (ms / 1e3)

    # ---- roofline of the check phase, device-timed per launch inside the library ----------------
    idx_ms, chk = h.phases(native.CIRCUIT_EVM, 0, n_steps, row_base, 0, min(args.steps, 50))
    bytes_alg = algorithmic_bytes(n_steps, n_rw, n_bc, n_constraints)
    cap = load_capture() if (args.groups == (1 << 18) and args.storage == "adaptive" and not strong) else None
    roofline = roofline_of(h, chk, bytes_alg, stored=storage["stored_bytes"],
                           kernel="evm check phase: k_evm_classify + k_evm_scatter + k_evm_push_pos + k_evm_gadget<MUL|ADD|POP, POS>",
                           index_build_ms=idx_ms, achieved_stored_gbs=storage["stored_bytes"] / (chk / 1e3) / 1e9,
                           note="frac uses SURVEY.md 8(d)'s canonical bytes (every cell at 32 B); the kernels read the "
                                "narrow stored columns, so stored_frac / dram_frac are the figures that bound them — they "
                                "are latency- / issue-bound, not byte-bound (profiles/README.md)")
    if cap:
        roofline["traffic"] = cap["dram_bytes_per_check"]
        roofline["dram_frac"] = cap["dram_bytes_per_check"] / (chk / 1e3) / 1e9 / h.peak
        roofline["ncu"] = {k: cap[k] for k in ("capture", "kernels", "kernel_ms_sum") if k in cap}

    # ---- e2e: host buffers through the C-ABI, copies inside the timed region --------------------
    # Every step ships its inputs from pinned host memory, builds the indexes, checks, and reads the result
    # vector back.  `serial`: one context, step k+1 starts when step k's result is on the host (latency of
    # one check).  `value`: the throughput of a STREAM of checks — two contexts on two streams alternate, so
    # step k+1's host->device copies run under step k's kernels (the copy engine never waits for the SMs).
    e2e = None
    if not args.no_e2e:
        def e2e_step():
            upload_inputs()
            hot_path()
            ctx.fetch_result(native.CIRCUIT_EVM, stream)

        e2e_step()
        k_e2e = max(4, min(args.steps, 20))
        ms_serial = h.timed(e2e_step, k_e2e)
        ctx2 = native.Context(local)
        s2 = torch.cuda.Stream()
        stream2 = s2.cuda_stream
        ctx2.upload_table(native.TABLE_FIXED, fixed, stream=stream2)
        if world > 1:
            box = [ctx2.nccl_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            ctx2.nccl_init(world, rank, box[0])
        lanes = [(ctx, stream), (ctx2, stream2)]

        def pipelined(k):
            def run():
                upload_inputs(*lanes[0])
                for i in range(k):
                    cur, nxt = lanes[i % 2], lanes[(i + 1) % 2]
                    if i + 1 < k:
                        upload_inputs(*nxt)  # enqueued before the (briefly host-blocking) check of `cur`
                    hot_path(*cur)
                    ff, _ = cur[0].fetch_result(native.CIRCUIT_EVM, cur[1])
                    assert (ff == native.PASS).all()
            return run

        pipelined(2)()
        torch.cuda.synchronize()
        ms_e2e = h.timed(pipelined(k_e2e), 1)
        if world > 1:
            ctx2.nccl_destroy()
        ctx2.close()
        e2e = {"value": rows_per_step * k_e2e / (ms_e2e / 1e3), "unit": "rows/s", "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": n_constraints * 12, "steps": k_e2e, "ms_per_step": ms_e2e / k_e2e,
               "mode": "stream of checks, double-buffered: two contexts / two streams alternate, every step's H2D + "
                       "index build + check + D2H inside the timed region",
               "serial": {"value": rows_per_step * k_e2e / (ms_serial / 1e3), "ms_per_step": ms_serial / k_e2e,
                          "mode": "one context, one stream: copy, then check, then read back"},
               "host_pack_ms": host_pack_ms, "host_generate_ms": 1e3 * gen_s,
               "note": "host_pack_ms (numpy scan of the canonical matrices into narrow columns) and host_generate_ms are "
                       "host preparation done once, outside the timed region"}

    # ---- extras ------------------------------------------------------------------------------------
    extras = {}
    if not args.no_extras:
        reps = max(3, min(args.steps, 20))
        if args.storage == "adaptive" and not strong:  # data-independent widths, same witness
            tp = {"steps": packing.pack_matrix(w["steps"], min_widths=packing.TYPE_WIDTHS["evm_steps"]),
                  "rw": packing.pack_matrix(w["rw"], min_widths=packing.TYPE_WIDTHS["rw_table"])}
            ctx.upload_table_packed(native.TABLE_RW, tp["rw"], stream=stream)
            ctx.upload_columns_packed(native.CIRCUIT_EVM, tp["steps"], stream=stream)
            for _ in range(3):
                hot_path()
            h.check_pass(native.CIRCUIT_EVM)
            t_ms = h.timed(hot_path, reps) / reps
            ti, tc = h.phases(native.CIRCUIT_EVM, 0, n_steps, row_base, 0, reps)
            extras["typed"] = {"value": world * n_steps / (t_ms / 1e3), "ms_per_step": t_ms, "kernel_ms": tc, "index_build_ms": ti,
                               "stored_bytes": int(tp["steps"].nbytes + tp["rw"].nbytes + 42 * n_bc),
                               "widths": {k: [int(x) for x in pm.widths] for k, pm in tp.items()}}
            del tp
        # ONE 2^20-step witness over the N ranks (at N = 1 this is the main line's workload)
        if world > 1 and not strong:
            ws = synth.evm_trace(args.groups, seed=2)
            b, e = shard(ws["n_steps"], rank, world)
            ctx.upload_bytecode_table_from_code(**ws["bytecode_src"], stream=stream)
            ctx.upload_table_packed(native.TABLE_RW, packing.pack_matrix(ws["rw"]), stream=stream)
            ctx.upload_columns_packed(native.CIRCUIT_EVM, packing.pack_matrix(take_rows(ws["steps"], np.arange(b, e + 1))), stream=stream)
            s_ms = h.sharded_pass(native.CIRCUIT_EVM, 0, e - b, b, 0, reps)
            si, sc = h.phases(native.CIRCUIT_EVM, 0, e - b, b, 0, reps)
            extras["strong_scaling"] = {"rows": ws["n_steps"], "rows_per_gpu": e - b, "ms_per_pass": s_ms,
                                        "rows_per_s": ws["n_steps"] / (s_ms / 1e3), "index_build_ms": si, "check_ms": sc,
                                        "collective_and_launch_ms": s_ms - si - sc,
                                        "bounded_by": max((("index build of the replicated tables", si), ("check kernels", sc),
                                                           ("collective + launch gaps", s_ms - si - sc)), key=lambda x: x[1])[0]}
            del ws
        else:
            extras["strong_scaling"] = {"rows": n_total, "rows_per_gpu": n_steps, "ms_per_pass": ms / args.steps,
                                        "rows_per_s": value, "index_build_ms": idx_ms, "check_ms": chk}
        extras["block_trace"] = bench_block(h, 4096, 64, 1024, reps)
        # row circuits on canonical cells: cfg3, cfg4 (copy 2^20 rows, sharded over the ranks), bytecode 2^19
        circuits = [bench_state(h, 1 << 18, reps), bench_copy(h, 512, 1024, reps), bench_bytecode(h, 19, reps),
                    bench_pi(h, 64, 1 << 18, 16, reps)]
        extras["circuits"] = circuits
        if world == 1:
            extras["assign"] = bench_assign(h, reps)
        extras["cfg4"] = {"copy_rows": circuits[1]["rows"], "rows_per_s": circuits[1]["rows_per_s"], "ms_per_pass": circuits[1]["ms_per_pass"],
                          "sharding": f"copy rows over {world} rank(s), halos +1/+2, rw / tx tables replicated"}
        # cfg5: super circuit = evm 2^20 + state 2^21 + copy 2^19 + bytecode 2^19 rows (2^22 in total), every circuit
        # row-sharded over the ranks, each against its own tables (state's rw encoding differs: SURVEY.md A.2)
        st5 = bench_state(h, 1 << 21, max(3, reps // 2))
        cp5 = bench_copy(h, 256, 1024, reps)
        evm_ms = extras["strong_scaling"]["ms_per_pass"]
        tot_rows = n_total + st5["rows"] + cp5["rows"] + circuits[2]["rows"]
        tot_ms = evm_ms + st5["ms_per_pass"] + cp5["ms_per_pass"] + circuits[2]["ms_per_pass"]
        extras["cfg5"] = {"rows": int(tot_rows), "ms": tot_ms, "rows_per_s": tot_rows / (tot_ms / 1e3),
                          "parts_ms": {"evm": evm_ms, "state": st5["ms_per_pass"], "copy": cp5["ms_per_pass"],
                                       "bytecode": circuits[2]["ms_per_pass"]},
                          "state_roofline_frac": st5["roofline"]["frac"], "copy_roofline_frac": cp5["roofline"]["frac"]}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        n, dt = cpu_port(args.ref_groups, 2, cores)
        cpu = {"value": n / dt, "unit": "rows/s", "cores": cores, "kind": "port",
               "sample": f"{cores} processes x {n // cores} steps of the same generator, C oracle incl. sorted-index build"}

    if rank == 0:
        line = {
            "metric": "constraint-rows/sec", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": f"evm_circuit ADD/SUB/MUL/DIV/MOD trace (cfg2 generator), {n_steps} steps per GPU",
                       "steps_per_gpu": n_steps, "rw_rows": n_rw, "bytecode_rows": n_bc, "fixed_rows": int(fixed.shape[1]),
                       "parallelism": f"row-shard x{world}, tables replicated, 1 collective (zk_allreduce_results)",
                       "l2": "inputs larger than L2 (%.2f GB stored per GPU)" % (storage["stored_bytes"] / 1e9),
                       "storage": storage, "source_hash": source_hash(),
                       "timed_region": "lookup-index build of bytecode+rw tables, then step check"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            **extras,
        }
        print(json.dumps(line))
    if world > 1:
        ctx.nccl_destroy()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
