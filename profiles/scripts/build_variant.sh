#!/bin/bash
# A/B kernel variants: recompiles the tick kernels + C-ABI host code with extra -D flags into
# dnn-mppi-mpc_b200/mppi_b200/libmppi_b200_<name>.so (the other objects come from the default build).
# Usage: profiles/scripts/build_variant.sh <name> "<-D flags>"; run with MPPI_B200_LIB=<that .so>
set -e
cd "$(dirname "$0")/../../dnn-mppi-mpc_b200/csrc"
name=$1; flags=$2; files=${3:-"mppi_kernels mppi_api"}      # third argument: the translation units to recompile
mkdir -p build_$name
NV="nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -ccbin /usr/bin/g++ $flags"
objs=""
for f in mppi_kernels mppi_api mppi_mlp mppi_mlp_traj mppi_topn mppi_spline mppi_probe; do
    unit=$f
    [[ $f == mppi_mlp_traj ]] && unit=mppi_mlp          # mppi_mlp_traj.cu compiles mppi_mlp.cu again: same flags for both
    if [[ " $files " == *" $unit "* || " $files " == *" $f "* ]]; then $NV -c $f.cu -o build_$name/$f.o & objs="$objs build_$name/$f.o"; else objs="$objs build/$f.o"; fi
done
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ../mppi_b200/libmppi_b200_$name.so $objs -ldl
echo built $name
