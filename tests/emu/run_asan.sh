#!/bin/bash
# The emulated panel-family tests under AddressSanitizer: any access of a kernel outside the caller's (numpy) buffers aborts.
# Builds the emulator library with -fsanitize=address into a scratch copy of the test (the repo copy stays untouched).
#   bash tests/emu/run_asan.sh          # ~25 minutes
set -e
ROOT=$(cd "$(dirname "$0")/../.." && pwd)
W=$(mktemp -d)
mkdir -p "$W/emu"
cp "$ROOT/tests/test_panel_emulated_cpu.py" "$ROOT/tests/test_panel_family_emulated_cpu.py" "$ROOT/tests/conftest.py" "$W/"
cp "$ROOT/tests/emu/panel_emu.cpp" "$ROOT/tests/emu/warp_emu.h" "$W/emu/"
sed -i "s|ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))|ROOT = '$ROOT'|" "$W/conftest.py"
sed -i "s|os.path.join(HERE, '..', 'bhmm_b200'|os.path.join('$ROOT', 'bhmm_b200'|g" "$W/test_panel_emulated_cpu.py"
sed -i "s|#include \"../../bhmm_b200/csrc/panel_kernels.cu\"|#include \"$ROOT/bhmm_b200/csrc/panel_kernels.cu\"|" "$W/emu/panel_emu.cpp"
g++ -O1 -g -fsanitize=address -fno-omit-frame-pointer -std=c++17 -shared -fPIC -w -I"${CUDA_HOME:-/usr/local/cuda}/include" \
    -o "$W/emu/panel_emu.so" "$W/emu/panel_emu.cpp"
cd "$W"
LD_PRELOAD=$(gcc -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0:detect_stack_use_after_return=0 \
    python -m pytest test_panel_emulated_cpu.py test_panel_family_emulated_cpu.py -x -q -p no:cacheprovider

# ---- part 2: the whole library (host logic + hostified kernels + fake CUDA runtime) under AddressSanitizer: the library's
# own "device" allocations (workspace carving, partial-statistics rows, flag maps) are checked too.  ~3 minutes.
E="$W/engine"
mkdir -p "$E/emu"
INC="-I${CUDA_HOME:-/usr/local/cuda}/include -I$ROOT/bhmm_b200/csrc -I$ROOT/tests/emu"
for f in capi engine certify team_kernels panel_kernels lane_viterbi scan_kernels frame_kernels sample_kernels transfer; do
    python "$ROOT/tests/emu/hostify.py" "$ROOT/bhmm_b200/csrc/$f.cu" > "$E/$f.cpp"
    g++ -O1 -g -fsanitize=address -fno-omit-frame-pointer -std=c++17 -fPIC -w $INC -DPANEL_HOST_EMU=1 \
        -include "$ROOT/tests/emu/cuda_fake.h" -c "$E/$f.cpp" -o "$E/$f.o" &
done
g++ -O1 -g -fsanitize=address -std=c++17 -fPIC -w $INC -c "$ROOT/tests/emu/cuda_fake.cpp" -o "$E/cuda_fake.o" &
g++ -O1 -g -fsanitize=address -std=c++17 -fPIC -w $INC -include "$ROOT/tests/emu/cuda_fake.h" -c "$ROOT/tests/emu/lane_stubs.cpp" -o "$E/lane_stubs.o" &
wait
g++ -shared -fsanitize=address -o "$E/emu/engine_emu.so" "$E"/*.o
cp "$ROOT/tests/emu/engine_emu_driver.py" "$E/emu/"
sed -i "s|ROOT = os.path.dirname(os.path.dirname(HERE))|ROOT = '$ROOT'|" "$E/emu/engine_emu_driver.py"
cd "$E/emu"
for mode in 0 1 2; do
    LD_PRELOAD=$(gcc -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0:detect_stack_use_after_return=0 \
        BHMM_B200_PANEL=$mode BHMM_B200_CHASE_TILED=1 python engine_emu_driver.py 32,40,40 21,40,40 s32 l8 v10 w32 w40 | grep -v " ok " || true
done
echo "engine under ASan: done (no AddressSanitizer report above = clean)"

# ---- part 3: the library with the lane family (engine_emu_lane.so, build_engine_emu.sh LANE=1) under AddressSanitizer: one
# E-step and Gibbs sweep for the N whose lane groups pad rows (9, 10, 11, 13, 14, 15) and for N = 1 and 16.  ~2 minutes.
L="$W/lane"
mkdir -p "$L"
python "$ROOT/tests/emu/hostify.py" "$ROOT/bhmm_b200/csrc/lane_kernels.cuh" > "$L/lane_kernels.cuh"
for f in capi engine certify team_kernels panel_kernels lane_viterbi scan_kernels frame_kernels sample_kernels transfer \
         lane_dispatch lane_inst_a lane_inst_b lane_inst_c lane_inst_d lane_inst_e lane_inst_f; do
    python "$ROOT/tests/emu/hostify.py" "$ROOT/bhmm_b200/csrc/$f.cu" > "$L/$f.cpp"
    g++ -O1 -g -fsanitize=address -fno-omit-frame-pointer -std=c++17 -fPIC -w $INC -DPANEL_HOST_EMU=1 \
        -include "$ROOT/tests/emu/cuda_fake.h" -c "$L/$f.cpp" -o "$L/$f.o" &
done
g++ -O1 -g -fsanitize=address -std=c++17 -fPIC -w $INC -c "$ROOT/tests/emu/cuda_fake.cpp" -o "$L/cuda_fake.o" &
wait
g++ -shared -fsanitize=address -o "$L/engine_emu_lane.so" "$L"/*.o
LD_PRELOAD=$(gcc -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0:detect_stack_use_after_return=0 \
    BHMM_EMU_LIB="$L/engine_emu_lane.so" BHMM_B200_EXACT_SCAN=0 \
    python "$ROOT/tests/emu/lane_emu_driver.py" 1,9,10,11,13,14,15,16 estep gibbs | grep -v " ok " || true
echo "lane family under ASan: done (no AddressSanitizer report above = clean)"
