#!/bin/bash
# round-4 call A: the withdrawal circuit (csrc/withdrawal.cu).  GPU tests (the whole -m gpu suite), smoke, byte-identical
# bench.py outputs against the parent commit's library, bench.py main line alternated base / new three times,
# tools/bench_withdrawal.py at 2^20 and 2^22 rows and at MAX_WITHDRAWALS = 16 with the one-limb-product RLC (new) and the
# Horner-chain RLC (-DZK_WD_HORNER) alternated twice, and a compute-sanitizer memcheck of tests/test_gpu_withdrawal.py
# where the tool exists.  Needs build/base/libzkcheck.so (parent commit), build/new/libzkcheck.so (this tree) and
# build/horner/libzkcheck.so (this tree, -DZK_WD_HORNER), all built for sm_100a.
O=${1:?usage: bash $0 OUT_DIR}
mkdir -p $O
BASE=$PWD/build/base/libzkcheck.so
NEW=$PWD/build/new/libzkcheck.so
HORNER=$PWD/build/horner/libzkcheck.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/a_gpu.txt; cat $O/a_gpu.txt
export ZKCHECK_LIB=$NEW
timeout 1200 python -m pytest tests -m gpu -q -p no:cacheprovider > $O/a_gpu_tests.log 2>&1; echo "pytest rc=$?"; grep -n "passed\|failed" $O/a_gpu_tests.log | tail -2; grep -n "^FAILED\|^E   " $O/a_gpu_tests.log | head -12
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/a_smoke.log 2>&1; echo "smoke rc=$?"; tail -2 $O/a_smoke.log
for arm in base new; do
  L=$BASE; [ $arm = new ] && L=$NEW
  ZKCHECK_LIB=$L timeout 600 python bench.py --dump-outputs $O/a_dump_$arm --no-extras --no-cpu-baseline > $O/a_dump_$arm.json 2> $O/a_dump_$arm.err; echo "dump $arm rc=$?"
done
cmp $O/a_dump_base/first_fail.npy $O/a_dump_new/first_fail.npy && cmp $O/a_dump_base/fail_count.npy $O/a_dump_new/fail_count.npy && echo "outputs byte-identical"
for rep in 1 2 3; do
  for arm in base new; do
    L=$BASE; [ $arm = new ] && L=$NEW
    ZKCHECK_LIB=$L timeout 600 python bench.py --no-extras --no-cpu-baseline > $O/a_ab_${arm}_$rep.json 2> $O/a_ab_${arm}_$rep.err
    python - <<PY
import json
d=json.loads(open("$O/a_ab_${arm}_$rep.json").read().strip().splitlines()[-1]); r=d["roofline"]
print("$arm $rep ms/step %.4f index %.4f check %.4f e2e %s" % (d["ms_per_step"], r["index_build_ms"], r["kernel_ms"], d.get("e2e", {}).get("value")))
PY
  done
done
for rep in 1 2; do
  for arm in new horner; do
    L=$NEW; [ $arm = horner ] && L=$HORNER
    ZKCHECK_LIB=$L timeout 900 python tools/bench_withdrawal.py --rows 20 22 --max16 --label $arm >> $O/a_bench_withdrawal.jsonl 2> $O/a_bench_withdrawal_${arm}_$rep.err; echo "bench_withdrawal $arm $rep rc=$?"
  done
done
cat $O/a_bench_withdrawal.jsonl
if command -v compute-sanitizer > /dev/null; then
  timeout 900 compute-sanitizer --tool memcheck --error-exitcode 9 python -m pytest tests/test_gpu_withdrawal.py -q -p no:cacheprovider -k "golden or assignment or reference" > $O/a_sanitizer_memcheck_withdrawal.log 2>&1; echo "memcheck rc=$?"; grep -n "passed\|failed\|ERROR SUMMARY" $O/a_sanitizer_memcheck_withdrawal.log | tail -3
else
  echo "compute-sanitizer: not on this machine" | tee $O/a_sanitizer_memcheck_withdrawal.log
fi
