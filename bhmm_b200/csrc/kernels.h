// bhmm_b200/csrc/kernels.h -- internal launch interface between the C ABI (capi.cu) and the kernels.
#pragma once
#include "common.cuh"

struct FwdArgs {
    Chains ch;
    Emission em;
    int N;
    int cpb;                 // chains per block (filled by the launcher)
    const double* A;         // (N,N) row-major, device
    const double* pi;        // (N), device
    double* alpha;           // (rows,N) row-major output, or NULL
    double* chain_ll;        // per chain: sum of log c_t over the chain's own frames
    double* hand_used;       // (n_chains_total, N): alpha_{t0-1} the chain was started from
    double* hand_end;        // (n_chains_total, N): the chain's own last alpha row
};

struct BwdArgs {
    Chains ch;
    Emission em;
    int N;
    int cpb;
    int grid;                // STATS: number of blocks (= rows of `partials`)
    const double* A;
    double* beta;            // literal backward: (rows,N) output
    const double* alpha;     // STATS: (rows,N) forward variables
    double* gamma;           // STATS: optional (rows,N) state probabilities output
    double* Bnum;            // STATS + EM_DISC: (N,M) B-numerator, accumulated with atomics
    double* partials;        // STATS: (grid, N*N+4N) per-block partial statistics
    double* hand_used;       // (n_chains_total, N): beta_e the chain entered with (e = first frame after the chain)
    double* hand_end;        // (n_chains_total, N): the chain's own beta at its first frame
};

struct VitArgs {
    Emission em;
    int N;
    int cpb;
    int K;                   // trajectories
    const long long* offsets;  // (K+1) row offsets, device
    const double* A;
    const double* pi;
    void* backptr;           // (rows, N) uint8 (N <= 256) or uint16
    int* path;               // (rows) int32 output
};

// Time-chunked Viterbi (panel_kernels.cu:k_viterbi_chain32): the chains of a long trajectory run their max-product
// recursions in parallel after a warm-up, hand-overs are certified like the forward filter's, and every decision's margin
// between best and second-best candidate is tracked so that the certified hand-over tolerance cannot have changed it.
struct VitChainArgs {
    Chains ch;
    Emission em;
    int N;
    const double* A;
    const double* pi;
    void* backptr;           // (rows, N) uint8 shifted back-pointer map (CHASE layout of k_viterbi_team)
    double* hand_used;       // (n_chains_total, N): normalised max-product vector at t0-1 the chain was started from
    double* hand_end;        // (n_chains_total, N): the chain's vector at its last frame
    unsigned* flagmap;       // (rows) one word per row of the map: bit j set = the decision stored in F[row][j] had a
                             // relative margin below margin_min (only decisions ON the resolved path matter)
    double margin_min;
};

// ---- lane family (lane_kernels.cu): one thread per chain, N <= LANE_MAX_N
constexpr int LANE_MAX_N = 16;
template <int N>
struct LaneParams {          // passed by value as a __grid_constant__ kernel parameter (constant-bank operands)
    double A[N * N];
    double pi[N];
    double mu[N];
    double isg[N];           // 1 / (sqrt(2) sigma)
    double nrm[N];           // log(1 / (sqrt(2 pi) sigma))
    double nrml[N];          // 1 / (sqrt(2 pi) sigma)   (comparison build LANE_FOLD_NRM=0 only)
};
struct LaneHostParams {      // HOST pointers
    const double* A;
    const double* pi;
    const double* mu;
    const double* sigma;
};
struct LaneArgs {
    Chains ch;
    const double* obs;       // EM_GAUSS: (rows)
    const int* sym;          // EM_DISC : (rows)
    const double* Bt;        // EM_DISC : (M,N)
    int M;
    int ignore_outliers;
    double* alpha_il;        // interleaved forward variables: [chain/32][frame][state/2][chain%32] double2
    int Lmax;                // frames per chain slot in alpha_il (= chunk)
    double* alpha_rm;        // row-major (rows,N) forward variables (LANE_FORWARD_ROWMAJOR)
    double* chain_ll;
    double* hand_used;       // forward or backward hand-over buffers, depending on the kernel
    double* hand_end;
    double* g0buf;           // (n_chains, N): gamma at frame 0 of the chains that start a trajectory
    double* partials;        // (blocks, N*N+4N)
    double* Bnum;
    double* gamma;           // optional (rows,N)
    // ---- forward-filter / backward-sample (LANE_SAMPLE_MAP / LANE_SAMPLE_FIX)
    const double* u_row;     // optional (rows) uniforms, one per frame; NULL: Philox4x32-10 keyed by (seed, sweep, row)
    unsigned long long seed, sweep;
    int* path;               // (rows) int32 sampled states
    unsigned char* smap;     // (n_chains, N): state at the chain's first frame for every entering state
    const int* enter;        // (n_chains): state at the frame after the chain (LANE_SAMPLE_FIX)
    int* coal;               // (n_chains): frame at which the chain's hypothetical paths coalesced (t0-1: never)
    long long* counts;       // device int64 [C (N*N) | n0 (N) | frames per state (N)], accumulated with atomics
    int* err;
};
enum { LANE_FORWARD = 0, LANE_FORWARD_ROWMAJOR = 1, LANE_BACKWARD_STATS = 2, LANE_SAMPLE_MAP = 3, LANE_SAMPLE_FIX = 4,
       LANE_QUERY_BLOCKS = 5 };
// resident blocks per SM of the most register-hungry lane kernel for this N (occupancy API); sizes the chain count
int lane_blocks_per_sm(int N, int em);
int lane_threads();
int launch_lane_sum_moments(const double* partials, int rows, int N, double* sums, cudaStream_t st);
bool lane_supported(int N, int em);
int lane_blocks(int n_chains);
int launch_lane(const LaneArgs& a, const LaneHostParams& hp, int N, int em, int what, cudaStream_t st);
int launch_add_gamma0(const Chains& ch, int n_total, int N, const double* g0buf, double* stats, cudaStream_t st);

void team_shape(int N, int* threads, int* cpb);
int launch_forward_team(const FwdArgs& a, int em, cudaStream_t st);
int launch_backward_team(const BwdArgs& a, int em, bool stats, cudaStream_t st);
int backward_stats_grid(int N, int n_chains);
int launch_viterbi_team(const VitArgs& a, int em, cudaStream_t st);

// ---- panel family (panel_kernels.cu): FP64 tensor pipe, 8 chains per warp (N = 32) or per block (32 < N <= 104);
// the default for 17 <= N <= 104 (BHMM_B200_PANEL=0 turns it off)
bool panel_enabled(int N);
void panel_shape(int N, int* threads, int* chains_per_row);
int panel_stats_rows(int N, int n_chains);   // rows of `partials` a statistics launch over n_chains writes
bool panel_forward_ok(const FwdArgs& a, int em);
bool panel_backward_ok(const BwdArgs& a, int em);
int launch_forward_panel(const FwdArgs& a, int em, cudaStream_t st);
int launch_backward_stats_panel(const BwdArgs& a, int em, cudaStream_t st);
bool panel_viterbi_ok(int N);                // 32 < N <= 104: Viterbi with the matrix column in registers
int launch_viterbi_panel(const VitArgs& a, int em, cudaStream_t st);
// ---- exact time-parallel chain starts (scan_kernels.cu): transfer operators per chain + a scan over them, N <= 32
bool exact_scan_ok(int N);
size_t exact_scan_bytes(int n_chains, int N);
int launch_exact_scan(const Chains& all, int n_total, const Emission& em, int emkind, const double* dA, int N, int dir,
                      double* he, double* ops, cudaStream_t st);
bool lane_viterbi_ok(int N);                 // N <= 16: the chunked Viterbi runs one thread per chain (lane_viterbi.cu)
int launch_viterbi_chain_lane(const VitChainArgs& a, int em, cudaStream_t st);
bool panel_viterbi_chain_ok(int N);          // N <= 32: time-chunked Viterbi for trajectories cut into chains
int launch_viterbi_chain(const VitChainArgs& a, int em, cudaStream_t st);
// counter += number of decisions ON the resolved paths whose margin was flagged (0: the paths are certified)
int launch_viterbi_path_flags(const unsigned* flagmap, const int* path, const long long* offsets, int K, long long rows,
                              int* counter, cudaStream_t st);

// ---- frame-parallel kernels (frame_kernels.cu)
int launch_gaussian_pobs(const double* obs, const double* mu, const double* sigma, int N, long long rows,
                         int ignore_outliers, double* pobs, cudaStream_t st);
int launch_discrete_pobs(const int* sym, const double* Bt, int N, int M, long long rows, int ignore_outliers,
                         double* pobs, cudaStream_t st);
int launch_state_probabilities(const double* alpha, const double* beta, int N, long long rows, double* gamma,
                               cudaStream_t st);
// column sums of a (rows,N) table; scratch holds blocks*N doubles
int launch_state_counts(const double* gamma, int N, long long rows, double* counts, double* scratch, int* blocks,
                        cudaStream_t st);
int state_counts_blocks(long long rows);
// literal transition_counts for ONE trajectory of T frames; scratch holds blocks*N*N doubles
int launch_transition_counts(const double* alpha, const double* beta, const double* A, const double* pobs, int N,
                             int T, double* C, double* scratch, cudaStream_t st);
int transition_counts_blocks(int T);
int launch_update_pout(const int* sym, const double* w, long long rows, int N, int M, double* pout, cudaStream_t st);
int launch_mstep_hmm(const double* stats, const double* mu_old, int N, int gauss, double mincount, double* out, cudaStream_t st);
int launch_mstep_rows(const double* Bnum, int N, int M, double* B, double* Bt, cudaStream_t st);
int launch_transpose(const double* in, int R, int Cc, double* out, cudaStream_t st);

// ---- certification of chain hand-overs (certify.cu)
// dir = +1 forward (chain c against c-1), -1 backward (chain c against c+1).
// out[0] = number of failing chains, out[1] = bits of the largest mismatch seen, out[2] = largest estimate of the
// warm-up length a hand-over needs (frames) to reach `tol`; fail_list receives the ids of the chains whose mismatch
// exceeds max(tol, tol_fail).
int launch_certify(const Chains& ch, int n_total, int N, int dir, const double* hand_used, const double* hand_end,
                   double tol, double tol_fail, int* fail_list, unsigned long long* out, cudaStream_t st);
// deterministic reduction of the E-step: stats = [loglik | gamma0 (N) | C (N*N) | sum gamma | sum gamma d | sum gamma d^2]
int launch_finalize_stats(const double* partials, int grid, const double* chain_ll, int n_chains, const double* A,
                          int N, double* stats, cudaStream_t st);

// ---- forward-filter / backward-sample and path statistics (sample_kernels.cu)
// choice table F[row][s'] = state drawn at `row` given the next frame's state s' and the frame's uniform.
int launch_sample_table(const double* alpha, const double* A, const double* u, const long long* offsets, int K,
                        int N, long long rows, unsigned char* F, int* err, cudaStream_t st);
// philox variant: uniforms generated on device from (seed, row)
int launch_sample_table_philox(const double* alpha, const double* A, unsigned long long seed, unsigned long long ctr,
                               const long long* offsets, int K, int N, long long rows, unsigned char* F, int* err,
                               cudaStream_t st);
// segment table `seg` has the chain-table layout (row0, len, t0, T), ordered by (trajectory, t0)
int launch_chase(const unsigned char* F, const Chains& seg, int N, unsigned char* seg_map, int* seg_enter, int* path,
                 cudaStream_t st);
// link step alone (lane-family sampler): enter[c] = state at the frame after chain c
int launch_chase_link(const Chains& seg, int N, const unsigned char* seg_map, int* seg_enter, cudaStream_t st);
int launch_path_stats(const int* path, const double* obs, const long long* offsets, int K, int N, long long rows,
                      long long* Cint, long long* n0, long long* cnt, double* so, double* soo, cudaStream_t st);
int launch_symbol_histogram(const int* path, const int* sym, long long rows, int N, int M, long long* hist,
                            cudaStream_t st);
// ---- synthetic trajectories (sample_kernels.cu).  `seg` is the segment table in REVERSED time order (t0 counted from the
// trajectory's end, see k_gen_map); cum0 (N) and cumA (N,N) are the cumulative tables; seg_start[c] >= 0 fixes the first
// state of segment c (NULL: drawn from cum0).  whole: every segment is a whole trajectory, the map and link steps are skipped.
int launch_generate_states(const Chains& seg, int N, const double* cum0, const double* cumA, const int* seg_start,
                           unsigned long long seed, bool whole, unsigned char* seg_map, int* seg_enter, int* states,
                           cudaStream_t st);
// one observation per frame from its state; a state outside [0, N) sets *err = BHMM_ERR_INVALID
int launch_emit_gaussian(const int* states, long long rows, int N, const double* mu, const double* sigma,
                         unsigned long long seed, double* obs, int* err, cudaStream_t st);
int launch_emit_discrete(const int* states, long long rows, int N, int M, const double* cumB, unsigned long long seed,
                         int* obs, int* err, cudaStream_t st);
