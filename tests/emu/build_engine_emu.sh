#!/bin/bash
# Builds tests/emu/engine_emu.so: the library's host logic (capi.cu, engine.cu) and its general-N kernels, hostified
# (hostify.py) and compiled for the CPU on top of the warp emulator and the fake CUDA runtime.  The lane family (N <= 16)
# is left out (lane_stubs.cpp): every batch takes the team kernels.
#
# LANE=1 builds tests/emu/engine_emu_lane.so instead: the same library with the lane family (lane_kernels.cuh,
# lane_dispatch.cu and the sixteen instantiations of lane_inst_{a..f}.cu) in place of the stubs, so that batches with
# N <= 16 run the lane kernels as the GPU build does.  Its objects go to _gen/lane/, apart from the default build's.
set -e
HERE=$(cd "$(dirname "$0")" && pwd)
ROOT=$(cd "$HERE/../.." && pwd)
GEN="$HERE/_gen"
SO="$HERE/engine_emu.so"
if [ "${LANE:-0}" = 1 ]; then
    GEN="$HERE/_gen/lane"
    SO="$HERE/engine_emu_lane.so"
fi
mkdir -p "$GEN"
INC="-I${CUDA_HOME:-/usr/local/cuda}/include -I$ROOT/bhmm_b200/csrc -I$HERE"
UNITS="capi engine certify team_kernels panel_kernels lane_viterbi scan_kernels frame_kernels sample_kernels transfer"
if [ "${LANE:-0}" = 1 ]; then
    # the instantiation units include "lane_kernels.cuh" by a quoted name: the hostified header next to them is found first
    python "$HERE/hostify.py" "$ROOT/bhmm_b200/csrc/lane_kernels.cuh" > "$GEN/lane_kernels.cuh"
    UNITS="$UNITS lane_dispatch lane_inst_a lane_inst_b lane_inst_c lane_inst_d lane_inst_e lane_inst_f"
fi
OBJS=""
for f in $UNITS; do
    python "$HERE/hostify.py" "$ROOT/bhmm_b200/csrc/$f.cu" > "$GEN/$f.cpp"
    g++ -O1 -std=c++17 -fPIC -w $INC -DPANEL_HOST_EMU=1 -include "$HERE/cuda_fake.h" -c "$GEN/$f.cpp" -o "$GEN/$f.o" &
    OBJS="$OBJS $GEN/$f.o"
done
g++ -O1 -std=c++17 -fPIC -w $INC -c "$HERE/cuda_fake.cpp" -o "$GEN/cuda_fake.o" &
OBJS="$OBJS $GEN/cuda_fake.o"
if [ "${LANE:-0}" != 1 ]; then
    g++ -O1 -std=c++17 -fPIC -w $INC -include "$HERE/cuda_fake.h" -c "$HERE/lane_stubs.cpp" -o "$GEN/lane_stubs.o" &
    OBJS="$OBJS $GEN/lane_stubs.o"
fi
wait
g++ -shared -o "$SO" $OBJS -lpthread
echo "$SO"
