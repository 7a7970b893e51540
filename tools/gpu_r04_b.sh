#!/bin/bash
# round-4 call B: bench.py against the parent commit.  The parent's tree (its Python package and bench.py, with its
# library) runs from build/base_tree, this tree with build/new/libzkcheck.so: --dump-outputs of both, compared byte for
# byte, then the main line alternated base / new three times.  Needs build/base_tree (git archive of the parent commit
# with its libzkcheck.so in the package directory) and build/new/libzkcheck.so, both built for sm_100a.
O=${1:?usage: bash $0 OUT_DIR}
mkdir -p $O
ROOT=$PWD
BASE_TREE=$ROOT/build/base_tree
NEW=$ROOT/build/new/libzkcheck.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/b_gpu.txt; cat $O/b_gpu.txt
run_bench() {  # arm, output file, extra args
  if [ $1 = base ]; then
    (cd $BASE_TREE && ZKCHECK_LIB=$BASE_TREE/zkevm-specs_b200/libzkcheck.so timeout 600 python bench.py "${@:3}") > $2 2> $2.err
  else
    ZKCHECK_LIB=$NEW timeout 600 python bench.py "${@:3}" > $2 2> $2.err
  fi
  echo "$1 rc=$?"
}
for arm in base new; do
  run_bench $arm $O/b_dump_$arm.json --dump-outputs $ROOT/$O/b_dump_$arm --no-extras --no-cpu-baseline
done
cmp $O/b_dump_base/first_fail.npy $O/b_dump_new/first_fail.npy && cmp $O/b_dump_base/fail_count.npy $O/b_dump_new/fail_count.npy && echo "outputs byte-identical"
for rep in 1 2 3; do
  for arm in base new; do
    run_bench $arm $O/b_ab_${arm}_$rep.json --no-extras --no-cpu-baseline
    python - <<PY
import json
d=json.loads(open("$O/b_ab_${arm}_$rep.json").read().strip().splitlines()[-1]); r=d["roofline"]
print("$arm $rep ms/step %.4f index %.4f check %.4f e2e %s" % (d["ms_per_step"], r["index_build_ms"], r["kernel_ms"], d.get("e2e", {}).get("value")))
PY
  done
done
