// bhmm_b200/csrc/scan_kernels.cu -- the EXACT time-parallel start of chains: transfer operators of the chains and a scan over
// them (north star (4): "a time-parallel associative scan over scaled transition-emission matrix products"; SURVEY 7.3-1b).
//
// The default way to start a chain in the middle of a trajectory is a warm-up whose result is certified afterwards
// (certify.cu).  That relies on the filter forgetting its start; a model that does not (a nearly reducible transition
// matrix with uninformative emissions) fails the certification for most chains, and the repair -- re-running failed chains
// from their neighbour's exact value, sweep after sweep -- degenerates to the sequential recursion.  This file is the
// fallback that stays parallel: the scaled recursions of _forward / _backward (_hidden.c:40-64, :92-108) are linear maps, so
//   forward :  alpha_{e-1}  ~  alpha_{t0-1} . M_c ,   M_c = prod_{t = t0}^{e-1} (A D_t)        (row vector times matrix)
//   backward:  beta_{t0}    ~  B_c . beta_e ,         B_c = prod_{f = t0+1}^{e} (A D_f)        (matrix times column vector)
// with D_t = diag(p_t).  k_chain_operator builds every chain's operator by running the N unit vectors through the chain at
// once (row i in warp i, one normalisation per row and frame, the scales kept as logarithms): N times the work of a vector
// pass, in parallel over chains.  k_scan_starts then walks the chains of each trajectory ONCE, composing the exact hand-over
// vectors from the one exact end the normal pass produced (the first chain started from pi, the last from beta = 1/N), and
// writes them where a pass with Chains.exact = 1 reads its starts.  N <= 32 here, 32 < N <= 128 in the wide variants below.
//
// Every kernel here is templated on the semiring SR.  SR_SUM is the sum-product of the E-step.  SR_MAX is the max-product of
// Viterbi (_hidden.c:229-265): the recursion delta_t(j) = p_j max_i delta_{t-1}(i) A_ij, normalised to sum one per frame, is
// linear in the max-times semiring, so the same operators, scan and composition carry over with the inner sum replaced by a
// max.  Row normalisation, log-scales, the exp(L - Lmax) weights, rows that drop out and the outlier rule stay as they are
// (every step is homogeneous in a positive scalar in both semirings).  The operators carry values only: back-pointers and the
// first-maximum tie rule stay in the Viterbi chain kernels, which re-run from the exact starts.  SR_MAX runs forward only.
#include <algorithm>

#include "common.cuh"
#include "kernels.h"

namespace {

constexpr unsigned FULLM = 0xffffffffu;

// acc (+) a (x) b: a fused multiply-add in the sum-product semiring, max(acc, a b) in the max-product one (a compare and a
// select: every value here is non-negative, and a NaN product is ignored as fmax would)
template <int SR>
__device__ __forceinline__ double sr_acc(double acc, double a, double b)
{
    if (SR == SR_SUM) return fma(a, b, acc);
    const double h = a * b;
    return h > acc ? h : acc;
}

// Backward scan, chain c: B_c maps the exact vector after it to zero.  The trajectory then has probability zero (a frame no
// state can emit, the outlier rule off: the reference's log-likelihood is -inf), and the exact beta is zero on chain c and every
// chain before it in the run: that is what the exact pass starts them from.  Left as they were, these starts would come from the
// failed warm-up pass, and the backward pass after the scan has no repair of its own.
__device__ __forceinline__ void scan_zero_backward(const Chains& ch, int n_total, int N, int c, int j, double* he)
{
    auto follows = [&](int a, int b) { return b < n_total && a >= 0 && ch.t0[b] != 0 && ch.row0[a] + ch.len[a] == ch.row0[b]; };
    for (; c > 0 && follows(c, c + 1) && follows(c - 1, c); --c)
        if (j < N) he[(long long)c * N + j] = 0.0;
}

template <int EM, int SR>
__global__ void __launch_bounds__(1024) k_chain_operator(Chains ch, Emission em, const double* __restrict__ A, int N, int dir,
                                                         double* __restrict__ ops, double* __restrict__ lscale)
{
    extern __shared__ double As[];                          // A (N x N), row-major
    for (int k = threadIdx.x; k < N * N; k += blockDim.x) As[k] = A[k];
    __syncthreads();
    const int c = blockIdx.x;
    const int i = threadIdx.x >> 5, j = threadIdx.x & 31;
    const bool jv = j < N;
    const int t0 = ch.t0[c], len = ch.len[c], T = ch.T[c];
    const long long trow = ch.row0[c] - t0;
    // forward: the chain's own frames; backward: shifted by one (the emission of frame f multiplies beta_f)
    const int fa = dir > 0 ? t0 : t0 + 1;
    const int fb = dir > 0 ? t0 + len : std::min(t0 + len + 1, T);
    const bool dead = dir < 0 && t0 + len >= T;             // the trajectory's last chain needs no backward operator
    double m = (i == j) ? 1.0 : 0.0;
    double ll = 0.0, prod = 1.0;
    const double mu = (EM == EM_GAUSS && jv) ? em.mu[j] : 0.0, sg = (EM == EM_GAUSS && jv) ? em.sigma[j] : 1.0;
    if (!dead) {
        for (int t = fa; t < fb; ++t) {
            const long long row = trow + t;
            double p = 0.0;
            if (jv) {
                if (EM == EM_GAUSS) p = gauss_pdf(em.obs[row], mu, sg);
                else if (EM == EM_POBS) p = em.pobs[row * N + j];
                else p = em.Bt[(long long)em.sym[row] * N + j];
            }
            if (EM != EM_POBS && em.ignore_outliers) {
                if (!__any_sync(FULLM, p != 0.0)) p = jv ? 1.0 : 0.0;     // outputmodel.py:126-130
            }
            double x = 0.0;
            for (int k = 0; k < N; ++k) {
                const double mk = __shfl_sync(FULLM, m, k);
                if (jv) x = sr_acc<SR>(x, mk, As[k * N + j]);
            }
            x *= p;
            double s = x;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(FULLM, s, off);
            if (s > 0.0) {
                m = x / s;
                prod *= s;
                if (!(prod >= 0x1p-400 && prod <= 0x1p+400)) { ll += log(prod); prod = 1.0; }
            } else {
                m = 0.0;                                    // this unit vector has no weight left: the row drops out
                ll = -INFINITY;
                prod = 1.0;
            }
        }
    }
    if (jv && i < N) ops[((long long)c * N + i) * N + j] = m;
    if (j == 0 && i < N) lscale[(long long)c * N + i] = dead ? 0.0 : ll + log(prod);
}

// One block per run of contiguous chains (a trajectory, or its owned range on a time shard); thread j = state j.
// forward : he[c] = normalise(he[c-1] . M_c) for the chains after the run's first;
// backward: he[c] = normalise(B_c . he[c+1]) for the chains before the run's last.
template <int SR>
__global__ void k_scan_starts(Chains ch, int n_total, int N, int dir, const double* __restrict__ ops,
                              const double* __restrict__ lscale, double* __restrict__ he)
{
    __shared__ double s[32], wgt[32];
    const int c0 = blockIdx.x, j = threadIdx.x;
    const bool jv = j < N;
    // chain b continues chain a's trajectory (rows of different trajectories are contiguous too: a chain that starts at
    // frame 0 starts a new run)
    auto follows = [&](int a, int b) { return b < n_total && a >= 0 && ch.t0[b] != 0 && ch.row0[a] + ch.len[a] == ch.row0[b]; };
    if (dir > 0) {
        if (c0 > 0 && follows(c0 - 1, c0)) return;          // not the first chain of its run
        s[j] = jv ? he[(long long)c0 * N + j] : 0.0;
        __syncwarp();
        for (int c = c0 + 1; follows(c - 1, c) && follows(c, c + 1); ++c) {
            // weights of the operator's rows: s_i exp(L_i - max L)
            const double L = jv ? lscale[(long long)c * N + j] : -INFINITY;
            double Lmax = (jv && s[j] > 0.0) ? L : -INFINITY;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) Lmax = fmax(Lmax, __shfl_xor_sync(FULLM, Lmax, off));
            wgt[j] = (jv && s[j] > 0.0 && L > -INFINITY) ? s[j] * exp(L - Lmax) : 0.0;
            __syncwarp();
            double x = 0.0;
            if (jv)
                for (int i = 0; i < N; ++i) x = sr_acc<SR>(x, wgt[i], ops[((long long)c * N + i) * N + j]);
            double tot = x;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) tot += __shfl_xor_sync(FULLM, tot, off);
            __syncwarp();
            if (!(tot > 0.0)) return;                       // degenerate: leave the remaining hand-overs to the fix-up passes
            s[j] = x / tot;
            if (jv) he[(long long)c * N + j] = s[j];
            __syncwarp();
        }
    } else {
        if (follows(c0, c0 + 1)) return;                    // not the last chain of its run
        s[j] = jv ? he[(long long)c0 * N + j] : 0.0;
        __syncwarp();
        for (int c = c0 - 1; c > 0 && follows(c, c + 1) && follows(c - 1, c); --c) {
            double x = 0.0;
            if (jv)
                for (int k = 0; k < N; ++k) x = sr_acc<SR>(x, ops[((long long)c * N + j) * N + k], s[k]);
            const double L = jv ? lscale[(long long)c * N + j] : -INFINITY;
            double Lmax = (jv && x > 0.0) ? L : -INFINITY;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) Lmax = fmax(Lmax, __shfl_xor_sync(FULLM, Lmax, off));
            x = (jv && x > 0.0 && L > -INFINITY) ? x * exp(L - Lmax) : 0.0;
            double tot = x;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) tot += __shfl_xor_sync(FULLM, tot, off);
            __syncwarp();
            if (!(tot > 0.0)) {
                scan_zero_backward(ch, n_total, N, c, j, he);
                return;
            }
            s[j] = x / tot;
            if (jv) he[(long long)c * N + j] = s[j];
            __syncwarp();
        }
    }
}

// ---- 32 < N <= 128 ------------------------------------------------------------------------------------------------
// The same two kernels with NT = ceil(N / 32) columns per lane.  Operator: the 32 warps of a block (16 for SR_MAX) take the rows i = w,
// w + 32, ... of the chain's operator one after the other (every row is its own vector recursion through the chain's frames;
// the emission of a frame is re-evaluated per row: NT exponentials against N * NT multiply-adds); component k of the row
// vector lives in lane k & 31, slot k >> 5, and is broadcast by one shuffle.  A is read through the cache (80 KB at N = 100:
// every warp of the block walks the same rows of it).  N times the work of a vector pass, like the narrow kernel; this is
// the fallback for models that do not forget, not a fast path.
// Warps per block of k_chain_operator_wide: the max-product step needs a register more per column than the fused multiply-add,
// which spills at the 64 registers of a 1024-thread block (N > 64, Gaussian); half the warps give it 128.
template <int SR>
constexpr int op_wide_warps() { return SR == SR_SUM ? 32 : 16; }

template <int EM, int NT, int SR>
__global__ void __launch_bounds__(32 * op_wide_warps<SR>(), SR == SR_SUM ? 0 : 1) k_chain_operator_wide(Chains ch, Emission em, const double* __restrict__ A, int N,
                                                              int dir, double* __restrict__ ops, double* __restrict__ lscale)
{
    const int c = blockIdx.x;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t0 = ch.t0[c], len = ch.len[c], T = ch.T[c];
    const long long trow = ch.row0[c] - t0;
    const int fa = dir > 0 ? t0 : t0 + 1;
    const int fb = dir > 0 ? t0 + len : std::min(t0 + len + 1, T);
    const bool dead = dir < 0 && t0 + len >= T;
    bool jv[NT];
    double mu[NT], sg[NT];
#pragma unroll
    for (int q = 0; q < NT; ++q) {
        const int j = lane + 32 * q;
        jv[q] = j < N;
        mu[q] = (EM == EM_GAUSS && jv[q]) ? em.mu[j] : 0.0;
        sg[q] = (EM == EM_GAUSS && jv[q]) ? em.sigma[j] : 1.0;
    }
    for (int i = w; i < N; i += op_wide_warps<SR>()) {
        double m[NT];
#pragma unroll
        for (int q = 0; q < NT; ++q) m[q] = (lane + 32 * q == i) ? 1.0 : 0.0;
        double ll = 0.0, prod = 1.0;
        if (!dead) {
            for (int t = fa; t < fb; ++t) {
                const long long row = trow + t;
                double p[NT];
                bool nz = false;
#pragma unroll
                for (int q = 0; q < NT; ++q) {
                    const int j = lane + 32 * q;
                    p[q] = 0.0;
                    if (jv[q]) {
                        if (EM == EM_GAUSS) p[q] = gauss_pdf(em.obs[row], mu[q], sg[q]);
                        else if (EM == EM_POBS) p[q] = em.pobs[row * N + j];
                        else p[q] = em.Bt[(long long)em.sym[row] * N + j];
                    }
                    nz = nz || (p[q] != 0.0);
                }
                if (EM != EM_POBS && em.ignore_outliers) {
                    if (!__any_sync(FULLM, nz)) {                          // outputmodel.py:126-130
#pragma unroll
                        for (int q = 0; q < NT; ++q) p[q] = jv[q] ? 1.0 : 0.0;
                    }
                }
                double x[NT];
#pragma unroll
                for (int q = 0; q < NT; ++q) x[q] = 0.0;
                for (int k = 0; k < N; ++k) {
                    double src = m[0];
#pragma unroll
                    for (int q = 1; q < NT; ++q) src = ((k >> 5) == q) ? m[q] : src;     // k is uniform over the warp
                    const double mk = __shfl_sync(FULLM, src, k & 31);
                    const double* Ak = A + (long long)k * N + lane;
#pragma unroll
                    for (int q = 0; q < NT; ++q)
                        if (jv[q]) x[q] = sr_acc<SR>(x[q], mk, Ak[32 * q]);
                }
                double s = 0.0;
#pragma unroll
                for (int q = 0; q < NT; ++q) { x[q] *= p[q]; s += x[q]; }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(FULLM, s, off);
                if (s > 0.0) {
#pragma unroll
                    for (int q = 0; q < NT; ++q) m[q] = x[q] / s;
                    prod *= s;
                    if (!(prod >= 0x1p-400 && prod <= 0x1p+400)) { ll += log(prod); prod = 1.0; }
                } else {
#pragma unroll
                    for (int q = 0; q < NT; ++q) m[q] = 0.0;                // this unit vector has no weight left
                    ll = -INFINITY;
                    prod = 1.0;
                }
            }
        }
#pragma unroll
        for (int q = 0; q < NT; ++q)
            if (jv[q]) ops[((long long)c * N + i) * N + lane + 32 * q] = m[q];
        if (lane == 0) lscale[(long long)c * N + i] = dead ? 0.0 : ll + log(prod);
    }
}

template <int NT, bool MAXOP>
__device__ __forceinline__ double scan_block_reduce(double v, double* red)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double o = __shfl_xor_sync(FULLM, v, off);
        v = MAXOP ? fmax(v, o) : v + o;
    }
    __syncthreads();                                        // `red` may still be read from the previous reduction
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = red[0];
#pragma unroll
    for (int q = 1; q < NT; ++q) r = MAXOP ? fmax(r, red[q]) : r + red[q];
    return r;
}

// One block of 32 NT threads per run of contiguous chains; thread j = state j (see k_scan_starts).
template <int NT, int SR>
__global__ void k_scan_starts_wide(Chains ch, int n_total, int N, int dir, const double* __restrict__ ops,
                                   const double* __restrict__ lscale, double* __restrict__ he)
{
    __shared__ double s[32 * NT], wgt[32 * NT], red[NT];
    const int c0 = blockIdx.x, j = threadIdx.x;
    const bool jv = j < N;
    auto follows = [&](int a, int b) { return b < n_total && a >= 0 && ch.t0[b] != 0 && ch.row0[a] + ch.len[a] == ch.row0[b]; };
    if (dir > 0) {
        if (c0 > 0 && follows(c0 - 1, c0)) return;          // not the first chain of its run (uniform over the block)
        s[j] = jv ? he[(long long)c0 * N + j] : 0.0;
        __syncthreads();
        for (int c = c0 + 1; follows(c - 1, c) && follows(c, c + 1); ++c) {
            const double L = jv ? lscale[(long long)c * N + j] : -INFINITY;
            const double Lmax = scan_block_reduce<NT, true>((jv && s[j] > 0.0) ? L : -INFINITY, red);
            wgt[j] = (jv && s[j] > 0.0 && L > -INFINITY) ? s[j] * exp(L - Lmax) : 0.0;
            __syncthreads();
            double x = 0.0;
            if (jv)
                for (int i = 0; i < N; ++i) x = sr_acc<SR>(x, wgt[i], ops[((long long)c * N + i) * N + j]);
            const double tot = scan_block_reduce<NT, false>(x, red);       // (its barriers also fence the reads of wgt)
            if (!(tot > 0.0)) return;                       // degenerate: leave the remaining hand-overs to the fix-up passes
            s[j] = x / tot;
            if (jv) he[(long long)c * N + j] = s[j];
        }
    } else {
        if (follows(c0, c0 + 1)) return;                    // not the last chain of its run
        s[j] = jv ? he[(long long)c0 * N + j] : 0.0;
        __syncthreads();
        for (int c = c0 - 1; c > 0 && follows(c, c + 1) && follows(c - 1, c); --c) {
            double x = 0.0;
            if (jv)
                for (int k = 0; k < N; ++k) x = sr_acc<SR>(x, ops[((long long)c * N + j) * N + k], s[k]);
            const double L = jv ? lscale[(long long)c * N + j] : -INFINITY;
            const double Lmax = scan_block_reduce<NT, true>((jv && x > 0.0) ? L : -INFINITY, red);
            x = (jv && x > 0.0 && L > -INFINITY) ? x * exp(L - Lmax) : 0.0;
            const double tot = scan_block_reduce<NT, false>(x, red);       // (every thread has read s[] before its barriers)
            if (!(tot > 0.0)) {
                scan_zero_backward(ch, n_total, N, c, j, he);
                return;
            }
            s[j] = x / tot;
            if (jv) he[(long long)c * N + j] = s[j];
            __syncthreads();
        }
    }
}

template <int NT, int SR>
int launch_exact_scan_wide(const Chains& ch, int n_total, const Emission& em, int emkind, const double* dA, int N, int dir,
                           double* he, double* ops, double* lscale, cudaStream_t st)
{
    switch (emkind) {
        case EM_POBS: k_chain_operator_wide<EM_POBS, NT, SR><<<n_total, 32 * op_wide_warps<SR>(), 0, st>>>(ch, em, dA, N, dir, ops, lscale); break;
        case EM_GAUSS: k_chain_operator_wide<EM_GAUSS, NT, SR><<<n_total, 32 * op_wide_warps<SR>(), 0, st>>>(ch, em, dA, N, dir, ops, lscale); break;
        case EM_DISC: k_chain_operator_wide<EM_DISC, NT, SR><<<n_total, 32 * op_wide_warps<SR>(), 0, st>>>(ch, em, dA, N, dir, ops, lscale); break;
        default: return BHMM_ERR_INVALID;
    }
    k_scan_starts_wide<NT, SR><<<n_total, 32 * NT, 0, st>>>(ch, n_total, N, dir, ops, lscale, he);
    return BHMM_OK;
}

// ---- operators of a whole shard (time-sharded trajectories) --------------------------------------------------------
// One block per pair of one level of a tree reduction: X <- X . Y with X = operator of chain pairs[2b], Y = operator of chain
// pairs[2b + 1] (the chain right after X's range in time), both in the representation k_chain_operator writes (row i of the
// true operator = exp(L_i) m_i, m_i summing to one).  Warp w takes the rows i = w, w + 32, ...; component k of a row lives in
// lane k & 31, slot k >> 5 (NT = 1: lane per column, N <= 32).  A warp reads row i of X and writes it back itself, so the
// product is formed in place; Y is read through the cache.  Plain FP64 FMAs: this serves the fallback, not the fast path.
template <int NT, int SR>
__global__ void __launch_bounds__(1024) k_compose_operators(const int* __restrict__ pairs, int N, double* ops, double* lscale)
{
    const int dst = pairs[2 * blockIdx.x], src = pairs[2 * blockIdx.x + 1];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const double* Y = ops + (long long)src * N * N;
    double* X = ops + (long long)dst * N * N;
    bool jv[NT];
    double ly[NT];
#pragma unroll
    for (int q = 0; q < NT; ++q) {
        jv[q] = lane + 32 * q < N;
        ly[q] = jv[q] ? lscale[(long long)src * N + lane + 32 * q] : -INFINITY;
    }
    for (int i = w; i < N; i += 32) {
        double x[NT];
        double Lmax = -INFINITY;
#pragma unroll
        for (int q = 0; q < NT; ++q) {
            x[q] = jv[q] ? X[(long long)i * N + lane + 32 * q] : 0.0;
            if (x[q] > 0.0) Lmax = fmax(Lmax, ly[q]);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) Lmax = fmax(Lmax, __shfl_xor_sync(FULLM, Lmax, off));
        // weights of Y's rows: x_ik exp(L_k - max L)
#pragma unroll
        for (int q = 0; q < NT; ++q) x[q] = (x[q] > 0.0 && ly[q] > -INFINITY) ? x[q] * exp(ly[q] - Lmax) : 0.0;
        double r[NT];
#pragma unroll
        for (int q = 0; q < NT; ++q) r[q] = 0.0;
        for (int k = 0; k < N; ++k) {
            double s = x[0];
#pragma unroll
            for (int q = 1; q < NT; ++q) s = ((k >> 5) == q) ? x[q] : s;      // k is uniform over the warp
            const double wk = __shfl_sync(FULLM, s, k & 31);
            const double* Yk = Y + (long long)k * N + lane;
#pragma unroll
            for (int q = 0; q < NT; ++q)
                if (jv[q]) r[q] = sr_acc<SR>(r[q], wk, Yk[32 * q]);
        }
        double tot = 0.0;
#pragma unroll
        for (int q = 0; q < NT; ++q) tot += r[q];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) tot += __shfl_xor_sync(FULLM, tot, off);
        const double Lx = lscale[(long long)dst * N + i];
        const bool live = tot > 0.0 && Lx > -INFINITY;
#pragma unroll
        for (int q = 0; q < NT; ++q)
            if (jv[q]) X[(long long)i * N + lane + 32 * q] = live ? r[q] / tot : 0.0;
        if (lane == 0) lscale[(long long)dst * N + i] = live ? Lx + Lmax + log(tot) : -INFINITY;
    }
}

// out (K, N, N + 1) for one direction: row i = [operator row i | log-scale i] of the chain first[k], the identity with zero
// log-scales where the shard owns no frame of trajectory k (first[k] < 0).
__global__ void k_operator_out(const int* __restrict__ first, int N, const double* __restrict__ ops,
                               const double* __restrict__ lscale, double* __restrict__ out, long long kstride)
{
    const int k = blockIdx.x, c = first[k];
    double* o = out + (long long)k * kstride;
    for (int e = threadIdx.x; e < N * (N + 1); e += blockDim.x) {
        const int i = e / (N + 1), j = e - i * (N + 1);
        double v;
        if (c < 0) v = (j == N) ? 0.0 : (i == j ? 1.0 : 0.0);
        else v = (j == N) ? lscale[(long long)c * N + i] : ops[((long long)c * N + i) * N + j];
        o[e] = v;
    }
}

template <int NT, int SR>
void launch_chain_operator_wide(const Chains& ch, int n_total, const Emission& em, int emkind, const double* dA, int N,
                                int dir, double* ops, double* lscale, cudaStream_t st)
{
    switch (emkind) {
        case EM_POBS: k_chain_operator_wide<EM_POBS, NT, SR><<<n_total, 32 * op_wide_warps<SR>(), 0, st>>>(ch, em, dA, N, dir, ops, lscale); break;
        case EM_GAUSS: k_chain_operator_wide<EM_GAUSS, NT, SR><<<n_total, 32 * op_wide_warps<SR>(), 0, st>>>(ch, em, dA, N, dir, ops, lscale); break;
        default: k_chain_operator_wide<EM_DISC, NT, SR><<<n_total, 32 * op_wide_warps<SR>(), 0, st>>>(ch, em, dA, N, dir, ops, lscale); break;
    }
}

template <int NT, int SR>
void launch_compose_level(const int* pairs, int n, int N, double* ops, double* lscale, cudaStream_t st)
{
    k_compose_operators<NT, SR><<<n, 32 * std::min(N, 32), 0, st>>>(pairs, N, ops, lscale);
}

template <int SR>
void shard_operators_sr(const Chains& ch, int n_total, const Emission& em, int emkind, const double* dA, int N, int dir,
                        const int* d_pairs, const std::vector<int>& lev_n, const std::vector<long long>& lev_off, double* ops,
                        double* lscale, cudaStream_t st)
{
    if (N > 32) {
        switch ((N + 31) / 32) {
            case 2: launch_chain_operator_wide<2, SR>(ch, n_total, em, emkind, dA, N, dir, ops, lscale, st); break;
            case 3: launch_chain_operator_wide<3, SR>(ch, n_total, em, emkind, dA, N, dir, ops, lscale, st); break;
            default: launch_chain_operator_wide<4, SR>(ch, n_total, em, emkind, dA, N, dir, ops, lscale, st); break;
        }
    } else {
        const size_t smem = sizeof(double) * (size_t)N * N;
        switch (emkind) {
            case EM_POBS: k_chain_operator<EM_POBS, SR><<<n_total, 32 * N, smem, st>>>(ch, em, dA, N, dir, ops, lscale); break;
            case EM_GAUSS: k_chain_operator<EM_GAUSS, SR><<<n_total, 32 * N, smem, st>>>(ch, em, dA, N, dir, ops, lscale); break;
            default: k_chain_operator<EM_DISC, SR><<<n_total, 32 * N, smem, st>>>(ch, em, dA, N, dir, ops, lscale); break;
        }
    }
    for (size_t L = 0; L < lev_n.size(); ++L) {
        const int* pairs = d_pairs + 2 * lev_off[L];
        switch ((N + 31) / 32) {
            case 1: launch_compose_level<1, SR>(pairs, lev_n[L], N, ops, lscale, st); break;
            case 2: launch_compose_level<2, SR>(pairs, lev_n[L], N, ops, lscale, st); break;
            case 3: launch_compose_level<3, SR>(pairs, lev_n[L], N, ops, lscale, st); break;
            default: launch_compose_level<4, SR>(pairs, lev_n[L], N, ops, lscale, st); break;
        }
    }
}

template <int SR>
int exact_scan_sr(const Chains& ch, int n_total, const Emission& em, int emkind, const double* dA, int N, int dir, double* he,
                  double* ops, double* lscale, cudaStream_t st)
{
    if (N > 32) {
        switch ((N + 31) / 32) {
            case 2: return launch_exact_scan_wide<2, SR>(ch, n_total, em, emkind, dA, N, dir, he, ops, lscale, st);
            case 3: return launch_exact_scan_wide<3, SR>(ch, n_total, em, emkind, dA, N, dir, he, ops, lscale, st);
            default: return launch_exact_scan_wide<4, SR>(ch, n_total, em, emkind, dA, N, dir, he, ops, lscale, st);
        }
    }
    const int threads = 32 * N;
    const size_t smem = sizeof(double) * (size_t)N * N;
    switch (emkind) {
        case EM_POBS: k_chain_operator<EM_POBS, SR><<<n_total, threads, smem, st>>>(ch, em, dA, N, dir, ops, lscale); break;
        case EM_GAUSS: k_chain_operator<EM_GAUSS, SR><<<n_total, threads, smem, st>>>(ch, em, dA, N, dir, ops, lscale); break;
        case EM_DISC: k_chain_operator<EM_DISC, SR><<<n_total, threads, smem, st>>>(ch, em, dA, N, dir, ops, lscale); break;
        default: return BHMM_ERR_INVALID;
    }
    k_scan_starts<SR><<<n_total, 32, 0, st>>>(ch, n_total, N, dir, ops, lscale, he);
    return BHMM_OK;
}

}  // namespace

// Operators of the owned frames of every trajectory of a time shard (bhmm_b200_shard_operators_*,
// bhmm_b200_shard_viterbi_operators_*): the chains' operators in semiring sr, then level after level of the reduction
// (lev_n[L] pairs at d_pairs + 2 lev_off[L]), then one (N, N + 1) block per trajectory written to out (trajectory stride
// kstride doubles).
int launch_shard_operators(const Chains& all, int n_total, const Emission& em, int emkind, const double* dA, int N, int dir,
                           int sr, const int* d_pairs, const std::vector<int>& lev_n, const std::vector<long long>& lev_off,
                           const int* d_first, int K, double* ops, double* out, long long kstride, cudaStream_t st)
{
    if (!exact_scan_ok(N)) return BHMM_ERR_UNSUPPORTED;
    if (emkind != EM_POBS && emkind != EM_GAUSS && emkind != EM_DISC) return BHMM_ERR_INVALID;
    if (sr != SR_SUM && !(sr == SR_MAX && dir > 0)) return BHMM_ERR_INVALID;
    double* lscale = ops + (size_t)n_total * N * N;
    if (n_total > 0) {
        Chains ch = all;
        ch.list = nullptr; ch.n = n_total;
        if (sr == SR_SUM) shard_operators_sr<SR_SUM>(ch, n_total, em, emkind, dA, N, dir, d_pairs, lev_n, lev_off, ops, lscale, st);
        else shard_operators_sr<SR_MAX>(ch, n_total, em, emkind, dA, N, dir, d_pairs, lev_n, lev_off, ops, lscale, st);
    }
    k_operator_out<<<K, 256, 0, st>>>(d_first, N, ops, lscale, out, kstride);
    return BHMM_OK;
}

bool exact_scan_ok(int N) { return N >= 1 && N <= 128; }

size_t exact_scan_bytes(int n_chains, int N) { return sizeof(double) * (size_t)n_chains * N * (N + 1); }

// ops: device scratch of exact_scan_bytes(n_total, N).  On return he (= w.he_f or w.he_b) holds exact hand-over vectors for
// every chain whose run started from an exact end; run the chains with Chains.exact = 1 next.  sr = SR_MAX (Viterbi) runs
// forward only.
int launch_exact_scan(const Chains& all, int n_total, const Emission& em, int emkind, const double* dA, int N, int dir, int sr,
                      double* he, double* ops, cudaStream_t st)
{
    if (!exact_scan_ok(N)) return BHMM_ERR_UNSUPPORTED;
    if (sr != SR_SUM && !(sr == SR_MAX && dir > 0)) return BHMM_ERR_INVALID;
    if (n_total <= 0) return BHMM_OK;
    double* lscale = ops + (size_t)n_total * N * N;
    Chains ch = all;
    ch.list = nullptr; ch.n = n_total;
    return sr == SR_SUM ? exact_scan_sr<SR_SUM>(ch, n_total, em, emkind, dA, N, dir, he, ops, lscale, st)
                        : exact_scan_sr<SR_MAX>(ch, n_total, em, emkind, dA, N, dir, he, ops, lscale, st);
}
