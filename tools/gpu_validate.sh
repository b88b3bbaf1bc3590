#!/bin/bash
# usage (GPU box): tools/gpu_validate.sh <tag> [extra kbench variants...]
# The whole -m gpu tier, smoke(), the default bench line and the launch-policy sweep of the CURRENT build.
tag=$1; shift
mkdir -p gpurun_out
timeout 1200 python -m pytest tests -x -q -m gpu > gpurun_out/${tag}_pytest.log 2>&1
tail -4 gpurun_out/${tag}_pytest.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 900 python bench.py > gpurun_out/${tag}_bench_full.log 2> gpurun_out/${tag}_bench.err
tail -c 600 gpurun_out/${tag}_bench_full.log; tail -3 gpurun_out/${tag}_bench.err
timeout 600 python tools/tail_policy_sweep.py 14000,18944,25000,65536,80776,113664,131072,262144,257328,524288 0,1 \
  > gpurun_out/${tag}_policy_sweep.jsonl 2> gpurun_out/${tag}_policy_sweep.err
cat gpurun_out/${tag}_policy_sweep.jsonl; tail -3 gpurun_out/${tag}_policy_sweep.err
for v in "$@"; do timeout 120 build/kbench/$v 20 3 >> gpurun_out/${tag}_kbench.jsonl 2>&1; done
for v in "$@"; do timeout 120 build/kbench/$v 20 3 >> gpurun_out/${tag}_kbench.jsonl 2>&1; done
[ -f gpurun_out/${tag}_kbench.jsonl ] && cut -c1-400 gpurun_out/${tag}_kbench.jsonl
