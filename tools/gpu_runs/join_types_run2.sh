#!/bin/bash
# join types, run 2: the join-type tests after fixing two of the test's own checks (schema slicing; Inner's row order
# with duplicate keys is the build's, so the two entry points are compared byte for byte only where keys are unique)
O=${RUN_OUT:-out}/join_types_run2; mkdir -p $O
timeout 900 python -m pytest tests/test_gpu_join_types.py -m gpu -q > $O/pytest_join_types.log 2>&1; tail -6 $O/pytest_join_types.log
timeout 600 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" > $O/smoke.txt 2>&1; tail -2 $O/smoke.txt
