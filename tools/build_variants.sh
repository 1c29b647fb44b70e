#!/bin/bash
# Alternate builds of libpp2d.so for tuning experiments: name=flags ...
# usage: bash tools/build_variants.sh "cs16=-DPP2D_CS_BATCH=16" "evm128=-DPP2D_EVM=128"
cd "$(dirname "$0")/.."
mkdir -p build/variants
for spec in "$@"; do
  name=${spec%%=*}; flags=${spec#*=}
  /usr/local/cuda/bin/nvcc -std=c++17 -O3 -lineinfo -gencode arch=compute_100a,code=sm_100a \
    -Xcompiler -fPIC -Xcompiler -fopenmp -shared -I include $flags -Xptxas -v \
    -o build/variants/libpp2d_$name.so path_planning_2d_b200/csrc/mdp.cu \
    path_planning_2d_b200/csrc/pomdp.cu path_planning_2d_b200/csrc/pbvi.cu path_planning_2d_b200/csrc/sim.cu -ldl -lgomp 2> build/variants/$name.ptxas.log &
done
wait
for spec in "$@"; do name=${spec%%=*}; echo "== $name"; grep -A2 "mdp_sweep_kernelILi2ELi2ELb0ELb0" build/variants/$name.ptxas.log | grep -E "registers|spill"; done
