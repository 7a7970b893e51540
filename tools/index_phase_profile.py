"""torch.profiler kernel list of the EVM check on bench.py's main-line workload (2^20 steps, packed rw table and
steps, bytecode table unrolled on the device): per-kernel device times of one pass from the trace, the stream each
kernel ran on, and how long the rw index verify overlapped k_evm_classify.

    python tools/index_phase_profile.py OUT_DIR [passes]

Writes OUT_DIR/index_phase_trace.json (chrome trace) and prints the kernel list of the last profiled pass."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from zkevm_specs_b200 import native, packing, synth  # noqa: E402
from zkevm_specs_b200.evm_circuit.table import fixed_table_matrix  # noqa: E402


def main():
    out = sys.argv[1]
    passes = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    os.makedirs(out, exist_ok=True)
    w = synth.evm_trace(1 << 18, seed=2)
    n = w["n_steps"]
    ctx = native.Context(0)
    stream = torch.cuda.Stream()
    s = stream.cuda_stream
    ctx.upload_table(native.TABLE_FIXED, fixed_table_matrix(), stream=s)
    ctx.upload_bytecode_table_from_code(**w["bytecode_src"], stream=s)
    ctx.upload_table_packed(native.TABLE_RW, packing.pack_matrix(w["rw"]), stream=s)
    ctx.upload_columns_packed(native.CIRCUIT_EVM, packing.pack_matrix(w["steps"]), stream=s)

    def one_pass():
        ctx.invalidate_indexes()
        ctx.check_async(native.CIRCUIT_EVM, 0, n, 0, 0, s)

    for _ in range(5):
        one_pass()
    stream.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(passes):
            one_pass()
            stream.synchronize()
    path = os.path.join(out, "index_phase_trace.json")
    prof.export_chrome_trace(path)
    ev = json.load(open(path))["traceEvents"]
    dev = [e for e in ev if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset") and "dur" in e]
    dev.sort(key=lambda e: e["ts"])
    # passes are separated by the host synchronise: split at the prep kernel that starts each pass
    starts = [i for i, e in enumerate(dev) if e["name"].startswith("void zk::k_pos_prep") or e["name"].startswith("zk::k_pos_prep")]
    last = dev[starts[-1]:] if starts else dev
    t0 = last[0]["ts"]
    print("GPU:", torch.cuda.get_device_name(0))
    print("%-10s %-10s %-8s %s" % ("start_us", "dur_us", "stream", "kernel / copy"))
    for e in last:
        print("%-10.1f %-10.2f %-8s %s" % (e["ts"] - t0, e["dur"], e.get("args", {}).get("stream", "?"), e["name"][:110]))
    end = max(e["ts"] + e["dur"] for e in last)
    print("pass: %.1f us from the prep kernel to the last kernel's end" % (end - t0))
    ver = [e for e in last if "k_pos_verify" in e["name"]]
    cls = [e for e in last if "k_evm_classify" in e["name"]]
    for v in ver:
        for c in cls:
            ov = min(v["ts"] + v["dur"], c["ts"] + c["dur"]) - max(v["ts"], c["ts"])
            print("overlap of %s (stream %s) with k_evm_classify (stream %s): %.2f us" % (
                v["name"].split("(")[0][-40:], v.get("args", {}).get("stream"), c.get("args", {}).get("stream"), max(ov, 0.0)))
    names = sorted({e["name"].split("(")[0] for e in dev})
    print("hash-index kernels in the profiled passes:", [x for x in names if "k_index_build" in x or "k_slots_clear" in x])
    sizes = sorted({e.get("args", {}).get("bytes") for e in dev if e.get("cat") == "gpu_memset"}, key=str)
    print("k_set_u32 launches:", [x for x in names if "k_set_u32" in x], "| memsets:", sum(1 for e in dev if e.get("cat") == "gpu_memset"),
          "of sizes (bytes)", sizes)


if __name__ == "__main__":
    main()
