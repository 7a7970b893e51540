#!/bin/bash
# round-3 call A: the index phase off the EVM check's critical path (k_pos_prep, typed dense verify, rw verify next to
# the step sort, hash parts after the flag read-back).  GPU tests, smoke, byte-identical outputs against the parent
# commit's library, base / new / ZKCHECK_INDEX_OVERLAP=0 alternated three times, full bench lines of base and new,
# the torch.profiler kernel list, memcheck of the new GPU test file.
# Needs build/base/libzkcheck.so (parent commit) and build/new/libzkcheck.so (this tree), both built for sm_100a.
O=${1:?usage: bash $0 OUT_DIR}
mkdir -p $O
BASE=$PWD/build/base/libzkcheck.so
NEW=$PWD/build/new/libzkcheck.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/a_gpu.txt; cat $O/a_gpu.txt
export ZKCHECK_LIB=$NEW
timeout 1500 python -m pytest tests -m gpu -q > $O/a_gpu_tests.log 2>&1; echo "pytest rc=$?"; grep -n "passed\|failed" $O/a_gpu_tests.log | tail -2; grep -n "^FAILED\|^E   " $O/a_gpu_tests.log | head -12
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/a_smoke.log 2>&1; echo "smoke rc=$?"; tail -2 $O/a_smoke.log
for arm in base new; do
  L=$BASE; [ $arm = new ] && L=$NEW
  ZKCHECK_LIB=$L timeout 600 python bench.py --steps 5 --warmup 2 --no-extras --no-cpu-baseline --no-e2e --dump-outputs $O/a_dump_$arm > /dev/null 2> $O/a_dump_$arm.err; echo "dump $arm rc=$?"
done
cmp $O/a_dump_base/first_fail.npy $O/a_dump_new/first_fail.npy && cmp $O/a_dump_base/fail_count.npy $O/a_dump_new/fail_count.npy && echo "outputs byte-identical"
for rep in 1 2 3; do
  for arm in base new overlap0; do
    L=$BASE; [ $arm != base ] && L=$NEW
    OV=1; [ $arm = overlap0 ] && OV=0
    ZKCHECK_LIB=$L ZKCHECK_INDEX_OVERLAP=$OV timeout 600 python bench.py --no-extras --no-cpu-baseline > $O/a_ab_${arm}_$rep.json 2> $O/a_ab_${arm}_$rep.err
    python - <<PY
import json
d=json.loads(open("$O/a_ab_${arm}_$rep.json").read().strip().splitlines()[-1]); r=d["roofline"]
print("$arm $rep ms/step %.4f index %.4f check %.4f e2e %s" % (d["ms_per_step"], r["index_build_ms"], r["kernel_ms"], d.get("e2e", {}).get("value")))
PY
  done
done
timeout 300 python tools/index_phase_profile.py $O 3 > $O/a_profile.txt 2>&1; echo "profile rc=$?"; cat $O/a_profile.txt | tail -40
for arm in base new; do
  L=$BASE; [ $arm = new ] && L=$NEW
  ZKCHECK_LIB=$L timeout 900 python bench.py --no-cpu-baseline > $O/a_full_$arm.json 2> $O/a_full_$arm.err; echo "full $arm rc=$?"
  python - <<PY
import json
d=json.loads(open("$O/a_full_$arm.json").read().strip().splitlines()[-1])
ss=d.get("strong_scaling"); bt=d.get("block_trace", {})
print("$arm full: ms/step", d["ms_per_step"], "e2e", d["e2e"]["value"], "block ms/pass", bt.get("ms_per_pass"), "strong", json.dumps(ss)[:300])
PY
done
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 9 python -m pytest tests/test_gpu_index_phase.py -q -p no:cacheprovider > $O/a_sanitizer_memcheck_index_phase.log 2>&1; echo "memcheck rc=$?"; grep -n "passed\|failed\|ERROR SUMMARY" $O/a_sanitizer_memcheck_index_phase.log | tail -3
