// bhmm_b200/csrc/tmatrix_kernels.cu -- reversible transition matrices from a count matrix, for N <= 128, in one thread block:
//   k_tmatrix_reversible   the detailed-balance maximum-likelihood estimate of the EM M-step
//                          (util/tmatrix.py:transition_matrix_reversible, reached through estimate_P);
//   k_sample_reversible    one draw from the reversible posterior of the Gibbs sweep (util/tmatrix.py:sample_P_reversible).
// Both run the same strong-connectivity check and the same fixed point (rev_connected / rev_fixed_point).  Every sum runs in
// a fixed order and there are no floating-point atomics, so identical inputs give bit-identical outputs on every rank.
//
// Shared memory holds one N x N array M (128 KB at N = 128): the counts C on entry, then Csym = C + C^T.  The fixed point
// never stores X: x_ij = csym_ij / (q_i + q_j) with q_i = c_i / x_i is a function of the N values q, so thread i recomputes
// row i of X from column i of Csym (equal to row i, and free of bank conflicts) and keeps only its row sum.
#include "host_common.h"
#include "philox.cuh"

namespace {

constexpr int TM_MAX_N = 128;
constexpr int TM_WORDS = TM_MAX_N / 32;

// Is the directed graph {i -> j : C_ij > thr} one strongly connected set?  Forward and backward reachability from state 0
// on bit rows, at most N frontier steps.  Thread i owns state i; blockDim.x is a multiple of 32 and at least N.  Reads
// C = M (row-major, shared); block-uniform result.
__device__ bool rev_connected(const double* M, int N, double thr, unsigned* fwd, unsigned* bwd)
{
    const int i = threadIdx.x, lane = i & 31, warp = i >> 5;
    unsigned row[TM_WORDS] = {0u, 0u, 0u, 0u}, col[TM_WORDS] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int w = 0; w < TM_WORDS; ++w)        // unrolled: the bit words stay in registers
        for (int j = 32 * w; j < min(N, 32 * w + 32) && i < N; ++j) {
            if (M[i * N + j] > thr) row[w] |= 1u << (j & 31);     // i -> j
            if (M[j * N + i] > thr) col[w] |= 1u << (j & 31);     // j -> i
        }
    bool f = i == 0, b = i == 0;              // reached from 0 / reaches 0
    for (;;) {
        const unsigned fw = __ballot_sync(0xffffffffu, f), bw = __ballot_sync(0xffffffffu, b);
        if (lane == 0) { fwd[warp] = fw; bwd[warp] = bw; }
        __syncthreads();
        bool nf = f, nb = b;
#pragma unroll
        for (int w = 0; w < TM_WORDS; ++w) {
            nf |= (col[w] & fwd[w]) != 0u;
            nb |= (row[w] & bwd[w]) != 0u;
        }
        const bool changed = nf != f || nb != b;
        f = nf;
        b = nb;
        if (!__syncthreads_or(changed)) break;   // the barrier also orders this step's reads before the next step's writes
    }
    return !__syncthreads_or(i < N && !(f && b));
}

// The fixed point of transition_matrix_reversible.  On entry M holds C; on return M holds Csym = C + C^T, and for thread i
// (< N): crow = c_i = sum_j C_ij, q[i] = c_i / pi_i of the last update, s = sum_j x_ij of the last update, pi = s / total,
// total = sum_ij x_ij.  The iteration: x_ij <- csym_ij / (q_i + q_j) (0 where the denominator is not positive), normalised
// to sum 1, until max_i |pi_new - pi_old| < maxerr or maxiter (>= 1) updates.  Returns the number of updates.
__device__ int rev_fixed_point(double* M, int N, int maxiter, double maxerr, double* q, double* sh_s, double& crow,
                               double& s, double& pi, double& total)
{
    const int i = threadIdx.x;
    crow = 0.0;
    if (i < N)
        for (int j = 0; j < N; ++j) crow += M[i * N + j];
    __syncthreads();
    if (i < N) {
        for (int j = i + 1; j < N; ++j) {
            const double v = M[i * N + j] + M[j * N + i];
            M[i * N + j] = v;
            M[j * N + i] = v;
        }
        M[i * N + i] += M[i * N + i];
    }
    __syncthreads();
    s = 0.0;
    if (i < N)
        for (int j = 0; j < N; ++j) s += M[j * N + i];
    sh_s[i] = s;
    __syncthreads();
    total = 0.0;
    for (int k = 0; k < N; ++k) total += sh_s[k];
    pi = s / total;
    int it = 0;
    while (it < maxiter) {
        if (i < N) q[i] = crow / pi;
        __syncthreads();
        s = 0.0;
        if (i < N) {
            const double qi = q[i];
            for (int j = 0; j < N; ++j) {
                const double d = qi + q[j];
                s += d > 0.0 ? M[j * N + i] / d : 0.0;
            }
        }
        sh_s[i] = s;
        __syncthreads();
        total = 0.0;
        for (int k = 0; k < N; ++k) total += sh_s[k];
        const double pn = s / total;
        const double err = fabs(pn - pi);
        pi = pn;
        ++it;
        if (!__syncthreads_or(i < N && !(err < maxerr))) break;
    }
    return it;
}

__device__ __forceinline__ double rev_x(const double* M, const double* q, int N, int i, int j)
{
    const double d = q[i] + q[j];
    return d > 0.0 ? M[j * N + i] / d : 0.0;
}

// EM M-step, run after k_mstep_hmm (with mincount < 0, so that its flags count collapsed sigmas only) on the same `out`
// = [A | pi | means | sigmas | flags | loglik]: A becomes the reversible MLE; with `stationary`, pi becomes its stationary
// vector (the normalised row sums of X).  flags += 1 when C thresholded at `mincount` is not one strongly connected set (A
// and pi are then left as k_mstep_hmm wrote them).  iters (optional) receives the number of fixed-point updates.
__global__ void k_tmatrix_reversible(const double* __restrict__ stats, int N, double mincount, int stationary, int maxiter,
                                     double maxerr, double* __restrict__ out, int* __restrict__ iters)
{
    extern __shared__ double M[];
    __shared__ double q[TM_MAX_N], sh_s[TM_MAX_N];
    __shared__ unsigned fwd[TM_WORDS], bwd[TM_WORDS];
    const int i = threadIdx.x;
    if (N == 1) {
        if (i == 0) {
            out[0] = 1.0;
            if (stationary) out[1] = 1.0;
            if (iters) *iters = 0;
        }
        return;
    }
    const double* Cm = stats + 1 + N;
    for (int k = i; k < N * N; k += blockDim.x) M[k] = Cm[k];
    __syncthreads();
    if (!rev_connected(M, N, mincount, fwd, bwd)) {
        if (i == 0) {
            out[(long long)N * N + 3 * N] += 1.0;
            if (iters) *iters = 0;
        }
        return;
    }
    double crow, s, pi, total;
    const int it = rev_fixed_point(M, N, maxiter, maxerr, q, sh_s, crow, s, pi, total);
    if (i < N) {
        sh_s[i] = s;
        if (stationary) out[(long long)N * N + i] = pi;
    }
    __syncthreads();
    // T_ij = x_ij / s_i, thread j writes column j (coalesced)
    if (i < N)
        for (int r = 0; r < N; ++r) out[(long long)r * N + i] = rev_x(M, q, N, r, i) / sh_s[r];
    if (i == 0 && iters) *iters = it;
}

// One reversible posterior draw (sample_P_reversible's chain, updates of disjoint rows run at the same time).
//
// Start: the reversible MLE of C = counts + prior (threshold 0 for connectivity, maxiter / maxerr as the host calls it),
// X = pi_i T_ij = x_ij / total (symmetric bit for bit), scaled so that its weights on the pattern {i <= j : x_ij > 0} sum to
// the pattern's size.  Storage: X in the upper triangle of M (diagonal included), Csym below it, c_ii in a register.
//
// A sweep is 1 + R rounds, R = N - 1 (N even) or N (N odd), with a barrier after each:
//   round 0       thread i updates x_ii (it touches row i only);
//   round 1 + r   round r of the circle-method matching of P = R + 1 players (player P - 1 fixed, a player N is a bye):
//                 slot 0 pairs (r, P - 1), slot k in 1 .. P/2 - 1 pairs ((r + k) mod (P - 1), (r - k) mod (P - 1)); thread
//                 k updates x_ij of its pair i < j, which touches rows i and j only.
// Every pair of the pattern is visited once per sweep, and the updates of one round depend on disjoint rows and commute, so
// the chain is the host's in another scan order with the same stationary law.  The row sums are recomputed after each sweep.
// Uniforms of the update in (sweep, round, slot): the Philox block (key, counter (row = round << 32 | slot, ctr = sweep))
// gives the Box-Muller normal of the proposal x' = x exp(0.5 z); the block (key, (row, ctr = 1 << 32 | sweep)) gives the
// acceptance uniform u.  Accept when log u < dlog, dlog as in sample_P_reversible.
// Output: T = X / rows, mu = rows / sum(rows); status 1 (T, mu untouched) when C is not strongly connected.
__global__ void k_sample_reversible(const long long* __restrict__ counts, const double* __restrict__ prior, int N, int nsweeps,
                                    unsigned long long key, int maxiter, double maxerr, double* __restrict__ T,
                                    double* __restrict__ mu, int* __restrict__ status)
{
    extern __shared__ double M[];
    __shared__ double q[TM_MAX_N], sh_s[TM_MAX_N], rows[TM_MAX_N], crows[TM_MAX_N];
    __shared__ int cnt[TM_MAX_N];
    __shared__ unsigned fwd[TM_WORDS], bwd[TM_WORDS];
    const int i = threadIdx.x;
    if (N == 1) {
        if (i == 0) { T[0] = 1.0; mu[0] = 1.0; *status = 0; }
        return;
    }
    for (int k = i; k < N * N; k += blockDim.x) M[k] = (double)counts[k] + prior[k];
    __syncthreads();
    if (!rev_connected(M, N, 0.0, fwd, bwd)) {
        if (i == 0) *status = 1;
        return;
    }
    double crow, s, pi, total;
    rev_fixed_point(M, N, maxiter, maxerr, q, sh_s, crow, s, pi, total);
    // the start: row i of X into the upper triangle (thread i alone touches it), then its share of the pattern's weight
    const double cii = 0.5 * M[i < N ? i * N + i : 0];         // Csym_ii = 2 c_ii exactly
    double part = 0.0;
    int np = 0;
    if (i < N) {
        crows[i] = crow;
        for (int j = i; j < N; ++j) {
            const double x = rev_x(M, q, N, i, j) / total;
            M[i * N + j] = x;
            if (x > 0.0) { part += x; ++np; }
        }
    }
    sh_s[i] = part;
    cnt[i] = np;
    __syncthreads();
    double wsum = 0.0;
    int npat = 0;
    for (int k = 0; k < N; ++k) { wsum += sh_s[k]; npat += cnt[k]; }
    const double scale = (double)npat / wsum;
    if (i < N)
        for (int j = i; j < N; ++j) M[i * N + j] *= scale;
    __syncthreads();
    auto row_sum = [&](int a) {
        double r = 0.0;
        for (int j = 0; j < a; ++j) r += M[j * N + a];
        for (int j = a; j < N; ++j) r += M[a * N + j];
        return r;
    };
    if (i < N) rows[i] = row_sum(i);
    __syncthreads();

    const int R = (N & 1) ? N : N - 1, P = R + 1;
    const double sigma = 0.5;
    for (int sw = 0; sw < nsweeps; ++sw) {
        for (int round = 0; round <= R; ++round) {
            int a = -1, b = -1;
            if (round == 0) {
                if (i < N) a = b = i;
            } else if (i < P / 2) {
                const int r = round - 1;
                a = i == 0 ? r : (r + i) % (P - 1);
                b = i == 0 ? P - 1 : (r - i + P - 1) % (P - 1);
                if (a > b) { const int t = a; a = b; b = t; }
                if (b >= N) a = -1;                                  // the bye
            }
            if (a >= 0 && M[a * N + b] > 0.0) {
                const long long prow = ((long long)round << 32) | (unsigned)i;
                const double z = philox_normal(key, (unsigned long long)sw, prow);
                const double u = philox_uniform(key, (1ULL << 32) | (unsigned long long)sw, prow);
                const double old = M[a * N + b];
                const double nw = __dmul_rn(old, exp(__dmul_rn(sigma, z)));
                const double d = __dadd_rn(nw, -old);
                const double lr = log(nw / old);
                const double ra = __dadd_rn(rows[a], d);
                double dlog;
                double rb = 0.0;
                if (a == b) {
                    dlog = __dadd_rn(__dmul_rn(cii, lr), -__dmul_rn(crows[a], log(ra / rows[a])));
                } else {
                    rb = __dadd_rn(rows[b], d);
                    dlog = __dadd_rn(__dadd_rn(__dmul_rn(M[b * N + a], lr), -__dmul_rn(crows[a], log(ra / rows[a]))),
                                     -__dmul_rn(crows[b], log(rb / rows[b])));
                }
                dlog = __dadd_rn(dlog, __dadd_rn(lr, -d));
                if (log(u) < dlog) {
                    M[a * N + b] = nw;
                    rows[a] = ra;
                    if (a != b) rows[b] = rb;
                }
            }
            __syncthreads();
        }
        if (i < N) rows[i] = row_sum(i);
        __syncthreads();
    }
    double rtot = 0.0;
    for (int k = 0; k < N; ++k) rtot += rows[k];
    if (i < N) {
        mu[i] = rows[i] / rtot;
        for (int r = 0; r < N; ++r) T[(long long)r * N + i] = (r <= i ? M[r * N + i] : M[i * N + r]) / rows[r];
    }
    if (i == 0) *status = 0;
}

inline int tm_threads(int N) { return ((N + 31) / 32) * 32; }

template <class K>
int tm_smem(K* kernel, int N, size_t& smem)
{
    smem = sizeof(double) * (size_t)N * N;
    if (smem > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return BHMM_OK;
}

int launch_tmatrix_reversible(const double* stats, int N, double mincount, int stationary, int maxiter, double maxerr,
                              double* out, int* iters, cudaStream_t st)
{
    if (N < 1 || N > TM_MAX_N) return BHMM_ERR_UNSUPPORTED;
    size_t smem;
    const int rc = tm_smem(k_tmatrix_reversible, N, smem);
    if (rc != BHMM_OK) return rc;
    k_tmatrix_reversible<<<1, tm_threads(N), smem, st>>>(stats, N, mincount, stationary, maxiter, maxerr, out, iters);
    return BHMM_OK;
}

int launch_sample_reversible(const long long* counts, const double* prior, int N, int nsweeps, unsigned long long key,
                             double* T, double* mu, int* status, cudaStream_t st)
{
    if (N < 1 || N > TM_MAX_N) return BHMM_ERR_UNSUPPORTED;
    size_t smem;
    const int rc = tm_smem(k_sample_reversible, N, smem);
    if (rc != BHMM_OK) return rc;
    // the fixed point as sample_P_reversible calls transition_matrix_reversible: maxiter 1e6, maxerr 1e-12
    k_sample_reversible<<<1, tm_threads(N), smem, st>>>(counts, prior, N, nsweeps, key, 1000000, 1e-12, T, mu, status);
    return BHMM_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI (include/bhmm_b200.h).  It lives with its kernels, so that the library's other units do not depend on this one.
extern "C" int bhmm_b200_mstep_reversible_dev(const double* d_stats, const double* d_means_old, int N, double mincount,
                                              int stationary, int maxiter, double maxerr, double* d_out, int* d_iters,
                                              void* stream)
{
    if (!d_stats || !d_out || N < 1 || maxiter < 1) {
        bhmm_set_error(BHMM_ERR_INVALID, "mstep_reversible: null pointer, N < 1 or maxiter < 1");
        return BHMM_ERR_INVALID;
    }
    if (N > TM_MAX_N) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "mstep_reversible: N > 128"); return BHMM_ERR_UNSUPPORTED; }
    // pi, means, sigmas and the collapsed-sigma flags of the non-reversible M-step; mincount < 0 keeps empty counts out of
    // its flags (the reversible estimator needs strong connectivity, not positive entries)
    RC_TRY(launch_mstep_hmm(d_stats, d_means_old, N, d_means_old != nullptr, -1.0, d_out, (cudaStream_t)stream));
    RC_TRY(launch_tmatrix_reversible(d_stats, N, mincount, stationary != 0, maxiter, maxerr, d_out, d_iters,
                                     (cudaStream_t)stream));
    LAUNCHED(2);
    CUDA_TRY(cudaGetLastError());
    return BHMM_OK;
}

extern "C" int bhmm_b200_sample_tmatrix_reversible_dev(const long long* d_counts, const double* d_prior, int N, int nsweeps,
                                                       unsigned long long key, double* d_T, double* d_mu, int* d_status,
                                                       void* stream)
{
    if (!d_counts || !d_prior || !d_T || !d_mu || !d_status || N < 1 || nsweeps < 0) {
        bhmm_set_error(BHMM_ERR_INVALID, "sample_tmatrix_reversible: null pointer, N < 1 or nsweeps < 0");
        return BHMM_ERR_INVALID;
    }
    if (N > TM_MAX_N) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "sample_tmatrix_reversible: N > 128"); return BHMM_ERR_UNSUPPORTED; }
    RC_TRY(launch_sample_reversible(d_counts, d_prior, N, nsweeps, key, d_T, d_mu, d_status, (cudaStream_t)stream));
    LAUNCHED(1);
    CUDA_TRY(cudaGetLastError());
    return BHMM_OK;
}
