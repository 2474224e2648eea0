// tests/emu/lane_stubs.cpp -- the default emulator build (engine_emu.so) leaves the lane family (lane_kernels.cuh, N <= 16)
// out: batches are reported as unsupported by it, so the engine takes the general-N team path, which the other emulated
// tests rely on.  engine_emu_lane.so (build_engine_emu.sh with LANE=1) links the real lane kernels instead of this file.
#include "../../bhmm_b200/csrc/kernels.h"

int lane_blocks_per_sm(int, int) { return 1; }
int lane_threads() { return 128; }
int launch_lane_sum_moments(const double*, int, int, double*, cudaStream_t) { return BHMM_ERR_UNSUPPORTED; }
bool lane_supported(int, int) { return false; }
int lane_blocks(int) { return 1; }
int launch_lane(const LaneArgs&, const LaneHostParams&, int, int, int, cudaStream_t) { return BHMM_ERR_UNSUPPORTED; }
int launch_add_gamma0(const Chains&, int, int, const double*, double*, cudaStream_t) { return BHMM_ERR_UNSUPPORTED; }
