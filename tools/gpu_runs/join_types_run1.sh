#!/bin/bash
# join types, run 1: the launch profile of q3 / q5 / q8 before and after, the new join-type tests, the whole -m gpu suite,
# smoke(), tools/join_types_bench.py, and bench.py's `queries` for the previous commit (_parent/, built from it) and this
# one, alternately
export RUN_OUT=${RUN_OUT:-out}
O=$RUN_OUT/join_types_run1; mkdir -p $O
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > $O/card.txt; cat $O/card.txt
timeout 300 python tools/launch_profile.py --root _parent --out $O/profile_parent.json > /dev/null 2> $O/profile_parent.err; tail -2 $O/profile_parent.err
timeout 300 python tools/launch_profile.py --out $O/profile_branch.json > /dev/null 2> $O/profile_branch.err; tail -2 $O/profile_branch.err
cmp $O/profile_parent.json $O/profile_branch.json && echo "launch profiles identical"
cp $O/profile_parent.json tests/golden/launch_profile_q3_q5_q8.json
timeout 900 python -m pytest tests/test_gpu_join_types.py -m gpu -q -x > $O/pytest_join_types.log 2>&1; tail -15 $O/pytest_join_types.log
timeout 600 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" > $O/smoke.txt 2>&1; tail -2 $O/smoke.txt
timeout 600 python tools/join_types_bench.py --out $O/join_types_bench.json > /dev/null 2> $O/join_types_bench.err; cat $O/join_types_bench.json; tail -3 $O/join_types_bench.err
for i in 1 2; do
  timeout 400 python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline > $O/bench_branch_$i.json 2> $O/bench_branch_$i.err
  (cd _parent && timeout 400 python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline) > $O/bench_parent_$i.json 2> $O/bench_parent_$i.err
done
python - <<'PY'
import json, os
O = os.environ.get("RUN_OUT", "out") + "/join_types_run1"
for arm in ("branch", "parent"):
    for i in (1, 2):
        try:
            d = json.loads([l for l in open(f"{O}/bench_{arm}_{i}.json") if l.startswith("{")][-1])
            q = d.get("queries", {})
            print(arm, i, "value", d.get("value"), {k: (q[k]["ms"], q[k]["ms_best"], q[k]["kernel_launches"]) for k in ("q3", "q5", "q8") if k in q}, d.get("parity_check"))
        except Exception as e:
            print(arm, i, "no result", e)
PY
timeout 1500 python -m pytest tests -m gpu -q > $O/pytest_all.log 2>&1; tail -4 $O/pytest_all.log
