/*
 * include/bhmm_b200.h -- C ABI of libbhmm_b200.so, the B200 (sm_100a) implementation of the bhmm HMM
 * dynamic-programming hot path.
 *
 * Plain C: pointers and sizes only, no torch / numpy types.  Three groups of entry points:
 *
 *  (1) HOST-pointer drop-ins.  Same argument lists, layouts (C-contiguous float64, (T,N) time-major, int32 paths)
 *      and meaning as the functions the reference's Cython wrappers bind, so a maintainer can point
 *      bhmm/hidden/impl_c/hidden.pyx at them by changing the `cdef extern` block (INTEGRATION.md).  They copy
 *      the inputs to the GPU, run the kernels, copy the outputs back and return when the host arrays are valid.
 *
 *        reference symbol (bhmm/hidden/impl_c/_hidden.h)           replacement
 *        ---------------------------------------------------------------------------------------------
 *        double _forward(alpha,A,pobs,pi,N,T)            :10-16    bhmm_b200_forward
 *        void   _backward(beta,A,pobs,N,T)               :18-23    bhmm_b200_backward
 *        void   _computeGamma(gamma,alpha,beta,N,T)      :25-30    bhmm_b200_state_probabilities
 *               (dead in C; live numpy code is bhmm/hidden/api.py:133-188)
 *        (numpy) state_counts, bhmm/hidden/api.py:191-211          bhmm_b200_state_counts
 *        int    _compute_transition_counts(C,A,pobs,alpha,beta,N,T) :38-45   bhmm_b200_transition_counts
 *        int    _compute_viterbi(path,A,pobs,pi,N,T)     :47-52    bhmm_b200_viterbi
 *        int    _sample_path(path,alpha,A,pobs,N,T)      :54-60    bhmm_b200_sample_path
 *        void   set_seed(seed)                           :63       bhmm_b200_set_seed
 *        void   _p_obs(o,mus,sigmas,N,T,p)   output_models/impl_c/_gaussian.h:5   bhmm_b200_gaussian_p_obs
 *        void   _update_pout(obs,weights,T,N,M,pout)  output_models/impl_c/_discrete.c:1  bhmm_b200_discrete_update_pout
 *
 *      Functions that return double/void in the reference keep that shape; their status is read with
 *      bhmm_b200_last_error().  Nothing here ever calls exit() (the reference does, _hidden.c:299-304).
 *
 *  (2) DEVICE-pointer variants (suffix _dev) of the same functions for callers whose arrays already live in
 *      GPU memory (torch tensors: pass tensor.data_ptr()).  `stream` is a cudaStream_t passed as void*.
 *
 *  (3) The batched, device-resident engine (bhmm_b200_batch_*): all trajectories of a data set stay on the GPU,
 *      one call runs a whole E-step (emission + forward + backward + statistics), a Viterbi pass or a Gibbs
 *      hidden-path sweep over every trajectory.  This is what MaximumLikelihoodEstimator._forward_backward
 *      (maximum_likelihood.py:221-282) and BayesianHMMSampler._updateHiddenStateTrajectories
 *      (bayesian_sampling.py:283-331) loop over, one trajectory at a time, in the reference.
 *
 * There is no CPU fallback: every entry point fails with BHMM_B200_ERR_CUDA when no device is usable.
 */
#ifndef BHMM_B200_H
#define BHMM_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BHMM_B200_OK 0
#define BHMM_B200_ERR_INVALID 1
#define BHMM_B200_ERR_NO_MEM 2         /* == _BHMM_ERR_NO_MEM (bhmm/hidden/impl_c/_hidden.h:5) -> MemoryError */
#define BHMM_B200_ERR_SAMPLE 3         /* no state could be drawn (p not normalisable) */
#define BHMM_B200_ERR_CUDA 4
#define BHMM_B200_ERR_UNSUPPORTED 5
#define BHMM_B200_ERR_NOT_CERTIFIED 6  /* chain hand-overs could not be certified (never observed; see DESIGN.md) */

/* ---- library state ------------------------------------------------------------------------------ */
int bhmm_b200_last_error(void);                 /* status of the last call made by this thread */
const char* bhmm_b200_last_error_string(void);
const char* bhmm_b200_version(void);
int bhmm_b200_device_count(void);
/* Counters of kernels launched by this library since load (bench.py reports them as gpu_launches). */
unsigned long long bhmm_b200_launch_count(void);
/* Time-chunking policy of the literal API: frames per chain and warm-up frames (0 = automatic). */
void bhmm_b200_set_chunking(int chunk, int warm);
/* Relative hand-over tolerance used by the certification (default 1e-13). */
void bhmm_b200_set_certify_tolerance(double tol);
/* E-step hand-overs whose mismatch exceeds max(certification tolerance, this) are repaired (default 1e-11); below it a
 * mismatch above the certification tolerance only lengthens the next warm-up.  0 = repair everything above the
 * certification tolerance (round-1 behaviour). */
void bhmm_b200_set_repair_tolerance(double tol);
/* Extra safety margin of the adaptive warm-up length (added to the factors 1.12 / 1.15 by which the warm-up is kept above the
 * measured need).  A failed certification costs a repair sweep on ONE rank and a wait on all the others, so a job on W ranks
 * wants failures W times rarer than a single process does: bhmm_b200.dist.tune_for_world() sets 0.04 log2(W). */
void bhmm_b200_set_warm_margin(double extra);
/* Diagnostics of the last chunked call: info[0]=chains, [1]=chunk, [2]=warm, [3]=fix-up sweeps (fwd),
 * [4]=fix-up sweeps (bwd), [5]=largest hand-over mismatch fwd, [6]= ... bwd, [7]=chains re-run. */
void bhmm_b200_last_info(double info[8]);

/* ---- (1) host-pointer drop-ins ------------------------------------------------------------------ */
double bhmm_b200_forward(double* alpha, const double* A, const double* pobs, const double* pi, int N, int T);
void bhmm_b200_backward(double* beta, const double* A, const double* pobs, int N, int T);
int bhmm_b200_state_probabilities(double* gamma, const double* alpha, const double* beta, int N, int T);
int bhmm_b200_state_counts(double* counts, const double* gamma, int N, int T);
int bhmm_b200_transition_counts(double* C, const double* A, const double* pobs, const double* alpha,
                                const double* beta, int N, int T);
int bhmm_b200_viterbi(int* path, const double* A, const double* pobs, const double* pi, int N, int T);
/* Uniforms come from the library's restatement of glibc srand()/rand() (r = rand()/(RAND_MAX+1.0)), so a
 * given seed reproduces the reference's draws; pobs is accepted and ignored like in the reference. */
int bhmm_b200_sample_path(int* path, const double* alpha, const double* A, const double* pobs, int N, int T);
void bhmm_b200_set_seed(int seed);              /* seed >= 0: srand(seed); seed < 0: srand(time(NULL)) */
/* Same with caller-supplied uniforms in draw order (u[0] is used for t = T-1). */
int bhmm_b200_sample_path_u(int* path, const double* alpha, const double* A, const double* u, int N, int T);
/* Fills n uniforms of the emulated glibc stream after srand(seed) (does not touch the library's stream). */
void bhmm_b200_glibc_uniforms(int seed, long n, double* u);

void bhmm_b200_gaussian_p_obs(const double* o, const double* mus, const double* sigmas, int N, int T, double* p);
/* p_obs followed by the outlier rule of OutputModel._handle_outliers (outputmodel.py:119-131). */
int bhmm_b200_gaussian_p_obs_outliers(const double* o, const double* mus, const double* sigmas, int N, int T,
                                      int ignore_outliers, double* p);
int bhmm_b200_discrete_p_obs(const int* obs, const double* B, int N, int M, int T, int ignore_outliers, double* p);
void bhmm_b200_discrete_update_pout(const int* obs, const double* weights, int T, int N, int M, double* pout);

/* ---- (2) device-pointer variants ---------------------------------------------------------------- */
int bhmm_b200_forward_dev(double* d_alpha, const double* d_A, const double* d_pobs, const double* d_pi, int N,
                          int T, double* logprob_host, void* stream);
int bhmm_b200_backward_dev(double* d_beta, const double* d_A, const double* d_pobs, int N, int T, void* stream);
int bhmm_b200_state_probabilities_dev(double* d_gamma, const double* d_alpha, const double* d_beta, int N, int T,
                                      void* stream);
int bhmm_b200_state_counts_dev(double* d_counts, const double* d_gamma, int N, int T, void* stream);
int bhmm_b200_transition_counts_dev(double* d_C, const double* d_A, const double* d_pobs, const double* d_alpha,
                                    const double* d_beta, int N, int T, void* stream);
int bhmm_b200_viterbi_dev(int* d_path, const double* d_A, const double* d_pobs, const double* d_pi, int N, int T,
                          void* stream);
int bhmm_b200_sample_path_dev(int* d_path, const double* d_alpha, const double* d_A, const double* d_u, int N,
                              int T, void* stream);
int bhmm_b200_gaussian_p_obs_dev(const double* d_o, const double* d_mus, const double* d_sigmas, int N, int T,
                                 int ignore_outliers, double* d_p, void* stream);
int bhmm_b200_discrete_p_obs_dev(const int* d_obs, const double* d_B, int N, int M, int T, int ignore_outliers,
                                 double* d_p, void* stream);

/* ---- (3) batched device-resident engine --------------------------------------------------------- */
typedef struct bhmm_b200_batch bhmm_b200_batch;

/* offsets: host array of K+1 row offsets of the concatenated trajectories (offsets[0]=0, offsets[K]=rows).
 * chunk / warm: frames per chain and warm-up frames (0 = automatic).  Scratch memory (forward variables,
 * chain tables, partial statistics) is allocated by the library unless a workspace is attached. */
int bhmm_b200_batch_create(bhmm_b200_batch** out, const long long* offsets, int K, int N, int chunk, int warm);
/* Time-sharded trajectories (SURVEY 8e, C5: one trajectory too long for one GPU): this batch OWNS only the frames
 * [own_lo[k], own_hi[k]) of trajectory k -- statistics, log-likelihood and outputs cover exactly those -- and the
 * frames around the range are a halo on which the chains next to its borders warm up (forward: from before own_lo,
 * backward: from after own_hi).  The hand-overs at the borders cannot be certified inside one batch:
 * bhmm_b200_batch_border_handovers returns, for trajectory k after an E-step, four N-vectors (host) --
 *   [0] the forward vector the first owned chain started from   (warmed-up alpha at frame own_lo-1)
 *   [1] the forward vector at the last owned frame              (alpha at own_hi-1)
 *   [2] the backward vector the last owned chain started from   (warmed-up beta at frame own_hi)
 *   [3] the backward vector at the first owned frame            (beta at own_lo)
 * -- so that the caller compares [0] with the previous shard's [1] and [2] with the next shard's [3]
 * (bhmm_b200.engine.TimeShardedTrajectories does, component-wise and relatively, with the engine's tolerance).
 * Viterbi and hidden-path sampling return BHMM_B200_ERR_UNSUPPORTED on such a batch unless their time-shard phases are set
 * (bhmm_b200_batch_set_viterbi_phase, bhmm_b200_batch_set_gibbs_phase). */
int bhmm_b200_batch_create_ranges(bhmm_b200_batch** out, const long long* offsets, const long long* own_lo,
                                  const long long* own_hi, int K, int N, int chunk, int warm);
int bhmm_b200_batch_border_handovers(const bhmm_b200_batch* b, int k, double* out);
/* Exact shard borders, for models whose filter does not forget its start within the halo (the border vectors then disagree).
 * The recursions are linear maps, so a shard's owned frames of trajectory k reduce to two N x N operators:
 *   forward  F_k = prod_{t = own_lo}^{own_hi - 1} (A D_t):  alpha_{own_hi - 1} ~ alpha_{own_lo - 1} . F_k
 *   backward B_k = prod_{f = own_lo + 1}^{own_hi} (A D_f):  beta_{own_lo}     ~ B_k . beta_{own_hi}
 * with D_t = diag(p(o_t | state)).  bhmm_b200_shard_operators_* write them to d_out, device (K, 2, N, N + 1) doubles: row i of
 * [0] = [row i of F_k, normalised to sum one | log of its scale], [1] the same for B_k; the identity with zero log-scales where
 * the shard owns no frame of trajectory k.  B_k reads frame own_hi, so a trajectory that continues after the owned range
 * needs at least one halo frame after it; an owned range that ends with the local trajectory is taken to end the trajectory
 * (its backward operator is not used).  N > 128 returns BHMM_B200_ERR_UNSUPPORTED, a batch without owned ranges
 * BHMM_B200_ERR_INVALID.  About N times the work of a forward pass.
 * The caller gathers all shards' operators together with their border vectors [1] and [3] (an all_gather of
 * K * 2 * N * (N + 1) doubles per shard), composes the exact alpha at own_lo - 1 from the first owner's [1] left to right and the
 * exact beta at own_hi from the last owner's [3] right to left (engine.compose_shard_operators), and hands them to the shard
 * with bhmm_b200_batch_set_border_starts (host N-vectors; NULL keeps the halo warm-up on that side, both NULL clear the
 * trajectory's starts).  The next E-steps start the first owned chain's forward recursion and the last owned chain's backward
 * recursion from them until they are cleared.  Rejected with BHMM_B200_ERR_INVALID: a batch without owned ranges, k out of
 * range, a shard that owns no frame of trajectory k, vectors with a NaN, negative or infinite component or no positive one, a
 * forward start where the owned range begins at local frame 0 and a backward start where it ends with the local trajectory. */
int bhmm_b200_shard_operators_gaussian(bhmm_b200_batch* b, const double* d_obs, const double* A, const double* pi,
                                       const double* means, const double* sigmas, int ignore_outliers, double* d_out,
                                       void* stream);
int bhmm_b200_shard_operators_discrete(bhmm_b200_batch* b, const int* d_obs, const double* A, const double* pi,
                                       const double* B, int M, int ignore_outliers, double* d_out, void* stream);
int bhmm_b200_batch_set_border_starts(bhmm_b200_batch* b, int k, const double* fwd, const double* bwd);
/* The warm-up adaptation policy of the batch engine as a plain host function (no device needed; used by the tests):
 * next warm-up length from the current one, the certification's need estimate (w log tol / log m), the largest
 * hand-over mismatch m of the pass and whether the pass failed; state[2] = {remembered need, passes since confirmed}. */
int bhmm_b200_adapt_warm(int current, double need, double worst, int failed, int warm_min, int warm_cap, double* state);
void bhmm_b200_batch_destroy(bhmm_b200_batch* b);
int bhmm_b200_batch_replan(bhmm_b200_batch* b, int chunk, int warm);
/* 1 when the batch runs the small-N one-thread-per-chain kernels (N <= 16), 0 for the general-N team kernels.
 * The environment variable BHMM_B200_FAMILY=team forces the latter at creation time. */
int bhmm_b200_batch_uses_lane_kernels(const bhmm_b200_batch* b);
/* Chains that fill the GPU exactly once for this state count (resident blocks of the statistics kernel x chains per block);
 * 0 without a device.  Callers that cut a data set into groups (engine.SubBatchedTrajectories) size the groups in multiples
 * of it so that no round of the persistent kernels runs mostly empty. */
int bhmm_b200_wave_chains(int N);
/* How many times the exact transfer-operator scan (scan_kernels.cu) replaced the certified warm-up starts of this batch's
 * chains since it was created: the fallback for models whose filter does not forget its start (N <= 32). */
double bhmm_b200_batch_scan_count(const bhmm_b200_batch* b);
/* Diagnostic: the hand-over vectors of the last pass, (chains, N) doubles each (host buffers): the vector every chain was
 * started from and the vector it computed at its own border; dir > 0 forward, dir < 0 backward. */
int bhmm_b200_batch_debug_handovers(const bhmm_b200_batch* b, int dir, double* used, double* end);
/* Switch a batch between the lane kernels (lane != 0; N <= 16 only) and the general-N team / panel kernels, re-plan its
 * chains and invalidate the workspace layout (query bhmm_b200_batch_workspace_bytes and attach again).  Used for models the
 * lane kernels refuse (a Gaussian sigma below 1e-100). */
int bhmm_b200_batch_set_family(bhmm_b200_batch* b, int lane);
/* Viterbi-only batch: the workspace holds no (rows, N) forward variables -- observations, uint8 back-pointer map and path
 * only (N + 4 + 8 bytes per frame instead of 9 N + 12) -- so that one very long trajectory (C5: 1e9 frames x 32 states = 44 GB)
 * fits one GPU for bhmm_b200_viterbi_*; E-step and sampling calls on such a batch return BHMM_B200_ERR_UNSUPPORTED.  Call
 * it right after bhmm_b200_batch_create, before bhmm_b200_batch_workspace_bytes / attach_workspace.  (The reference has no
 * counterpart: compute_viterbi_paths, maximum_likelihood.py:332-352, keeps every trajectory's (T, N) table in host memory.) */
int bhmm_b200_batch_set_viterbi_only(bhmm_b200_batch* b, int on);
size_t bhmm_b200_batch_workspace_bytes(const bhmm_b200_batch* b);
int bhmm_b200_batch_attach_workspace(bhmm_b200_batch* b, void* d_workspace, size_t bytes);
/* info[0]=chains, [1]=chunk, [2]=warm, [3]=fwd fix-up sweeps, [4]=bwd fix-up sweeps, [5]=worst fwd mismatch,
 * [6]=worst bwd mismatch, [7]=chains re-run, of the last engine call on this batch. */
void bhmm_b200_batch_info(const bhmm_b200_batch* b, double info[8]);
/* Per-kernel device timing of the E-step (CUDA events on the launching stream): ms[0] = forward kernel incl.
 * certification, ms[1] = backward+statistics kernel, ms[2] = from the first to the last of those events. */
int bhmm_b200_batch_set_profiling(bhmm_b200_batch* b, int on);
void bhmm_b200_batch_kernel_ms(const bhmm_b200_batch* b, double ms[4]);
int bhmm_b200_stats_len_gaussian(int N);        /* 1 + N + N*N + 3N */
int bhmm_b200_stats_len_discrete(int N);        /* 1 + N + N*N + N  (B-numerator is separate) */

/* One Baum-Welch E-step over all trajectories (maximum_likelihood.py:383-385 + :271-282 + the data passes of
 * OutputModel.estimate).  d_obs: device (rows) float64.  A, pi, means, sigmas: HOST arrays.
 * d_stats (device, bhmm_b200_stats_len_gaussian(N) doubles) receives
 *    [ loglik | gamma0_sum (N) | C (N*N) | sum_t gamma (N) | sum_t gamma*(o-mu) (N) | sum_t gamma*(o-mu)^2 (N) ]
 * with mu the CURRENT means (shifted moments; the host M-step recentres them, see estimators/).
 * d_gamma: optional device (rows,N) output of the state probabilities (NULL to keep them on chip). */
int bhmm_b200_estep_gaussian(bhmm_b200_batch* b, const double* d_obs, const double* A, const double* pi,
                             const double* means, const double* sigmas, int ignore_outliers, double* d_gamma,
                             double* d_stats, void* stream);
/* Discrete output model: d_obs device (rows) int32, B host (N,M).  d_stats = [loglik|gamma0|C|sum gamma];
 * d_Bnum device (N,M) receives the B numerator sum_t gamma[t,i]*[o_t == m] (_update_pout). */
int bhmm_b200_estep_discrete(bhmm_b200_batch* b, const int* d_obs, const double* A, const double* pi,
                             const double* B, int M, int ignore_outliers, double* d_gamma, double* d_stats,
                             double* d_Bnum, void* stream);
/* Viterbi paths of all trajectories (maximum_likelihood.py:332-352); d_path device (rows) int32. */
int bhmm_b200_viterbi_gaussian(bhmm_b200_batch* b, const double* d_obs, const double* A, const double* pi,
                               const double* means, const double* sigmas, int ignore_outliers, int* d_path,
                               void* stream);
int bhmm_b200_viterbi_discrete(bhmm_b200_batch* b, const int* d_obs, const double* A, const double* pi,
                               const double* B, int M, int ignore_outliers, int* d_path, void* stream);
/* Viterbi of trajectories that are cut in TIME across devices (SURVEY 8e, C5).  A shard is a batch with owned ranges
 * (bhmm_b200_batch_create_ranges) whose local trajectories END with their owned range: halo frames before it, none after.
 * phase 1: bhmm_b200_viterbi_* only builds the back-pointer map of the owned frames (chain-parallel, hand-overs inside the
 * shard certified; the border hand-over is exported by bhmm_b200_batch_border_handovers, rows 0 and 1, for the caller to
 * compare across shards).  phase 2: only resolves the path, ending in the state set by
 * bhmm_b200_batch_set_viterbi_end_state (the state of trajectory k at its last local frame, i.e. path[own_lo - 1] of the
 * shard that owns the following frames; -1 = this shard holds the trajectory's end).  phase 0 (default) does both.
 * d_path is filled for the local rows; rows before own_lo - 1 are meaningless.  N <= 128 (BHMM_B200_PANEL=0: none); a path
 * through a decision whose margin is below the certified tolerance returns BHMM_B200_ERR_NOT_CERTIFIED.  For 32 < N <= 128
 * the near-tie flags take ceil(N / 32) words per frame, and a Viterbi-only shard sizes its chains to that kernel's wave. */
int bhmm_b200_batch_set_viterbi_phase(bhmm_b200_batch* b, int phase);
int bhmm_b200_batch_set_viterbi_end_state(bhmm_b200_batch* b, int k, int state);
/* One Gibbs hidden-path sweep (bayesian_sampling.py:283-331): emission + forward + backward sampling of every
 * trajectory, then the path statistics of generic_hmm.py:297-334,398-431.  Uniforms: d_u (device, one per row,
 * u[row] is the draw of that frame) or, when d_u is NULL, device Philox4x32-10 keyed by (seed, sweep).
 * d_counts (device int64): [ C (N*N) | n0 (N) | frames per state (N) ];  d_sums (device float64, may be NULL for
 * discrete): [ sum o (N) | sum o^2 (N) ] per state. */
int bhmm_b200_gibbs_gaussian(bhmm_b200_batch* b, const double* d_obs, const double* A, const double* pi,
                             const double* means, const double* sigmas, int ignore_outliers, const double* d_u,
                             unsigned long long seed, unsigned long long sweep, int* d_path, long long* d_counts,
                             double* d_sums, double* loglik_host, void* stream);
int bhmm_b200_gibbs_discrete(bhmm_b200_batch* b, const int* d_obs, const double* A, const double* pi,
                             const double* B, int M, int ignore_outliers, const double* d_u,
                             unsigned long long seed, unsigned long long sweep, int* d_path, long long* d_counts,
                             double* loglik_host, void* stream);
/* Gibbs hidden-path sweep of trajectories cut in TIME across devices.  A sampling shard is a batch with owned ranges whose
 * local trajectories END with their owned range (halo frames before it, none after), on the team / panel family
 * (bhmm_b200_batch_set_family(b, 0); N <= 256).  Given the uniforms, the draw at frame t is a function s_t = F_t(s_{t+1}) of the
 * next state only, so the shard's owned frames of trajectory k reduce to one map of N states: from the state at the frame
 * after the local end to the state at the first owned frame.
 *   phase 1: bhmm_b200_gibbs_* runs the forward filter (warm-up on the halo), the table of the owned rows and those maps;
 *            bhmm_b200_batch_gibbs_shard_map copies map k (N bytes) to the host.  The forward border vectors are in
 *            bhmm_b200_batch_border_handovers, rows 0 and 1, for the caller to compare across shards.
 *   phase 2: bhmm_b200_gibbs_* links and replays the owned frames from the states set by
 *            bhmm_b200_batch_set_gibbs_enter_state (state of trajectory k at the frame after its local end; -1 = the shard
 *            holds the trajectory's end) and returns the statistics of the owned frames: the transition out of the last owned
 *            frame into the entering state belongs to this shard, n0 is counted only where local frame 0 is the
 *            trajectory's frame 0, the log-likelihood covers the owned frames.  Summed over shards they are the statistics
 *            of the whole trajectories.  d_path is filled for the owned rows only.
 *   phase 0 (default): whole trajectories only; a batch with owned ranges is refused.
 * bhmm_b200_batch_set_philox_rows: frame t of local trajectory k draws the Philox row base[k] + t (NULL: the batch row), so
 * that a shard draws the uniforms of the rows its frames have in the unsharded batch.  bhmm_b200_batch_set_gibbs_borders:
 * per trajectory, flag 1 = the trajectory continues after the local end (its last owned row is an ordinary row), flag 2 =
 * local frame 0 is the trajectory's frame 0 (NULL: flag 2 for every trajectory).  Bad phases, flags, states, a right halo
 * and phase 2 before phase 1 are rejected with BHMM_B200_ERR_INVALID. */
int bhmm_b200_batch_set_gibbs_phase(bhmm_b200_batch* b, int phase);
int bhmm_b200_batch_set_philox_rows(bhmm_b200_batch* b, const long long* base);
int bhmm_b200_batch_set_gibbs_borders(bhmm_b200_batch* b, const int* flags);
int bhmm_b200_batch_set_gibbs_enter_state(bhmm_b200_batch* b, int k, int state);
int bhmm_b200_batch_gibbs_shard_map(const bhmm_b200_batch* b, int k, unsigned char* out);
/* Per-state symbol histogram of sampled paths (DiscreteOutputModel.sample's bincount, discrete.py:240-245):
 * d_hist (device int64, N*M) += [path==i][obs==m]. */
int bhmm_b200_path_symbol_histogram(const int* d_path, const int* d_obs, long long rows, int N, int M,
                                    long long* d_hist, void* stream);

/* M-step on the device from the (all-reduced) packed statistics of bhmm_b200_estep_* (SURVEY 8f N1; replaces the host
 * arithmetic of maximum_likelihood.py:284-330 on the non-reversible branch: estimate_P -> C / rowsum,
 * _tmatrix_disconnected.py:110-115; pi = gamma0 / sum, :318-320; GaussianOutputModel.estimate gaussian.py:214-272 via the
 * shifted moments).  d_means_old: the means the E-step ran with (NULL for a discrete model: no Gaussian part).
 * d_out (device, N*N + 3N + 2 doubles) = [A | pi | means | sigmas | flags | loglik]; flags counts C entries <= mincount (+1 each:
 * the caller must use the general-connectivity estimator instead) and sigmas below machine epsilon (+1024 each). */
int bhmm_b200_mstep_dev(const double* d_stats, const double* d_means_old, int N, double mincount, double* d_out,
                        void* stream);
/* DiscreteOutputModel.estimate's normalisation (discrete.py:214-215): d_B (N,M) = d_Bnum / rowsum; d_Bt (M,N), optional,
 * receives the transposed table. */
int bhmm_b200_mstep_discrete_dev(const double* d_Bnum, int N, int M, double* d_B, double* d_Bt, void* stream);

/* ---- synthetic trajectories (HMM.generate_synthetic_*, bhmm/hmm/generic_hmm.py:433-589) --------------------------
 * Hidden states of K trajectories (host offsets as in bhmm_b200_batch_create) drawn by exact time-parallel forward
 * simulation of the chain, then one observation per frame.  The stream: with row the frame's index in the call and
 * U(seed, c, row) the 53-bit uniform of Philox4x32-10 (key = seed, counter = (row, c)),
 *   s_0 = start[k], or the smallest i with U(seed, 0, row) < cum0[i];   s_t = smallest i with U(seed, 0, row) < cumA[s_{t-1}][i]
 * where the cumulative tables are sequential float64 sums of the rows of p0 / A, set to exactly 1.0 from the last
 * positive entry on.  Only comparisons are involved, so the states do not depend on the device or on `segment` (frames
 * per time-parallel segment, 0 = automatic).  A and p0 are HOST arrays (p0 may be NULL when start is given); d_states
 * (device, rows int32) receives the states; the workspace (device) holds bhmm_b200_generate_workspace_bytes bytes
 * (0: invalid arguments).  N <= 256; every trajectory has 1 to 2^31 - 1 frames. */
size_t bhmm_b200_generate_workspace_bytes(const long long* offsets, int K, int N, int segment);
int bhmm_b200_generate_states(int* d_states, const long long* offsets, int K, int N, const double* A, const double* p0,
                              const int* start, unsigned long long seed, int segment, void* d_workspace, size_t bytes,
                              void* stream);
/* Observations of d_states (device, rows int32; a state outside [0, N) fails with BHMM_B200_ERR_INVALID).
 * Gaussian: Box-Muller on the Philox block (seed, counter (row, 1)): u1 = ((bits of words 0,1 >> 11) + 1) 2^-53,
 * u2 = (bits of words 2,3 >> 11) 2^-53, o = means[s] + sigmas[s] sqrt(-2 log u1) cospi(2 u2); d_obs device float64.
 * Discrete: o = smallest m with U(seed, 1, row) < cumB[s][m]; B host (N, M); d_obs device int32. */
int bhmm_b200_emit_gaussian(double* d_obs, const int* d_states, long long rows, int N, const double* means,
                            const double* sigmas, unsigned long long seed, void* stream);
int bhmm_b200_emit_discrete(int* d_obs, const int* d_states, long long rows, int N, int M, const double* B,
                            unsigned long long seed, void* stream);

/* ---- (4) the estimators' one-off transfers -------------------------------------------------------- */
/* The reference estimators take a LIST of host arrays (maximum_likelihood.py:60-144, bayesian_sampling.py:60-150) and return
 * one hidden-state path per trajectory (maximum_likelihood.py:332-352).  upload_ragged concatenates K pageable host arrays
 * (srcs[k], nbytes[k] bytes each) into device memory at d_dst; download_ragged cuts device memory back into K host arrays.
 * `threads` worker threads (0 = automatic) each drive two pinned staging slots and a copy stream, so the host-side copy
 * (which is also what first touches a fresh destination's pages) runs in parallel with the DMA.  `stream` is synchronised
 * before the transfer starts (work queued on it may still use the buffers); both calls return when the data has arrived. */
int bhmm_b200_upload_ragged(void* d_dst, const void* const* srcs, const long long* nbytes, int K, int threads, void* stream);
int bhmm_b200_download_ragged(void* const* dsts, const void* d_src, const long long* nbytes, int K, int threads,
                              void* stream);
/* Write-touches every page of a fresh host allocation (threads = 0: two threads); host code only.  The estimators call it from a
 * helper thread on the array that will receive the paths, so that the page faults happen while the GPU is busy. */
int bhmm_b200_prefault(void* p, long long nbytes, int threads);
/* Tuning knobs of the two calls above (measurement scripts): staging slot size in KiB (0 = keep; default 2048, or
 * BHMM_B200_STAGE_KB) and streaming stores for the host-side copy on / off (negative = keep; default on, or
 * BHMM_B200_NT_COPY=0).  The pinned staging slots are released and re-created by the next transfer. */
int bhmm_b200_transfer_config(int stage_kb, int nt_copy);

#ifdef __cplusplus
}
#endif
#endif /* BHMM_B200_H */
