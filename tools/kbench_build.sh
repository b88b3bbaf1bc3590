#!/bin/bash
# Build kbench from several checkouts in parallel, for an A/B of the pairing kernels:
#   tools/kbench_build.sh parent:/path/to/parent/checkout new:.
# Each name:tree compiles tree/tools/kbench.cu (with that tree's kernels) into build/kbench/name.
mkdir -p build/kbench
for spec in "$@"; do
  name="${spec%%:*}"; tree="${spec#*:}"
  ( nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xptxas -v -DSY_VARIANT="\"$name\"" \
      -o build/kbench/$name "$tree/tools/kbench.cu" > build/kbench/$name.log 2>&1 \
    && grep -A2 "k_miller\|k_final_exp" build/kbench/$name.log | grep "stack\|Used" | tr '\n' ' ' | sed "s/^/$name: /" && echo ) &
done
wait
