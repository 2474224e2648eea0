// bhmm_b200/csrc/team_kernels.cu -- general-N chain kernels ("team" family).
//
// One TEAM of threads walks one chain sequentially; thread j of the team owns hidden state j.
//   N <= 32 : a block is one warp and carries cpb = 32/N teams (sub-warp packing),
//   N  > 32 : a block is one team of ceil32(N) threads.
// The transition matrix lives in shared memory, the per-frame vectors are exchanged through a
// double-buffered shared-memory slab (one __syncthreads per exchange).  Blocks are persistent:
// grid = min(#chain groups, SMs x resident blocks) and each block strides over the chain table.
//
// Replaces (reference file:line):
//   k_forward_team        _forward                      bhmm/hidden/impl_c/_hidden.c:16-66
//   k_backward_team       _backward                     _hidden.c:69-110
//   k_backward_stats_team _backward + state_probabilities (hidden/api.py:133-188) + state_counts (:191-211)
//                         + _compute_transition_counts (_hidden.c:148-183) + the data passes of
//                         GaussianOutputModel.estimate / _update_pout (gaussian.py:214-272, _discrete.c:1-32),
//                         with beta, gamma and xi kept on chip
//   k_viterbi_team        _compute_viterbi              _hidden.c:203-281 (bit-exact operation order)
// with the emission tile (_gaussian.c:45-70 / discrete.py:146-153 / outputmodel.py:119-131) fused in.
#include "common.cuh"
#include "kernels.h"

namespace {

struct TeamGeom {
    int team;        // team index inside the block
    int j;           // hidden state owned by this thread (valid iff owns && j < N)
    bool owns;       // thread belongs to a valid team
    unsigned mask;   // lanes of this team inside the warp (single-warp blocks only)
};

__device__ __forceinline__ TeamGeom team_geometry(int N, int cpb)
{
    TeamGeom g;
    const int tid = threadIdx.x;
    if (N <= 32) {
        g.team = tid / N;
        g.j = tid - g.team * N;
        g.owns = g.team < cpb;
        g.mask = g.owns ? (((N == 32) ? 0xffffffffu : ((1u << N) - 1u)) << (g.team * N)) : 0u;
    } else {
        g.team = 0;
        g.j = tid;
        g.owns = true;          // every thread follows team 0's control flow; j < N gates state ownership
        g.mask = 0u;
    }
    return g;
}

// true iff `pred` holds for at least one thread of the caller's team.  Uniform call sites only.
__device__ __forceinline__ bool team_any(bool pred, const TeamGeom& g)
{
    if (blockDim.x == 32) {
        const unsigned b = __ballot_sync(0xffffffffu, pred);
        return (b & g.mask) != 0u;
    }
    return __syncthreads_or(pred ? 1 : 0) != 0;
}

// ra = any(a), rb = any(b) over the caller's team, for predicates with b => a (one barrier in the common case)
__device__ __forceinline__ void team_any2(bool a, bool b, const TeamGeom& g, bool& ra, bool& rb)
{
    if (blockDim.x == 32) {
        const unsigned ba = __ballot_sync(0xffffffffu, a), bb = __ballot_sync(0xffffffffu, b);
        ra = (ba & g.mask) != 0u;
        rb = (bb & g.mask) != 0u;
        return;
    }
    // (__syncthreads_or returns a truth value, not the OR of the operands; b implies a at both call sites, so the
    // second barrier is only taken on the rare frames without any sizeable density)
    rb = __syncthreads_or(b ? 1 : 0) != 0;
    ra = rb ? true : (__syncthreads_or(a ? 1 : 0) != 0);
}

// A frame whose densities are ALL tiny (below 2^-500: an observation ~26 sigma away from every state) is lifted by
// 2^600 before it enters the recursion.  The kernels keep alpha / beta unnormalised for one step (the division by the
// previous frame's sum is folded into the next matvec), so two such frames in a row would otherwise multiply to an
// underflow, and a single one would push the exchanged vector into the denormal range, where products lose their
// digits; the reference normalises after every frame and is immune.  A uniform power of two changes nothing downstream
// (alpha, beta, gamma, xi are ratios); the forward log-likelihood subtracts it again.
#define TINY_P 0x1p-500
#define LIFT_P 0x1p+600
#define LIFT_LOG 415.88830833596718565          /* 600 ln 2 */

__device__ __forceinline__ int block_max(int v)
{
    if (blockDim.x == 32) return __reduce_max_sync(0xffffffffu, v);
    return v;   // multi-warp blocks carry a single team: the value is already uniform
}

// xor-butterfly sum over the 32 lanes: every lane ends with the bitwise identical total
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// Sums over a team's N shared-memory values with eight independent accumulators: a single running sum is a chain of N
// dependent FP64 operations (8 cycles each), which at N = 100 was most of a frame's time.
__device__ __forceinline__ double dot8(const double* __restrict__ x, int sx, const double* __restrict__ y, int sy, int N)
{
    double m[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int i = 0;
    for (; i + 7 < N; i += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) m[k] = fma(x[(i + k) * sx], y[(i + k) * sy], m[k]);
    }
    for (; i < N; ++i) m[0] = fma(x[i * sx], y[i * sy], m[0]);
    return ((m[0] + m[1]) + (m[2] + m[3])) + ((m[4] + m[5]) + (m[6] + m[7]));
}
__device__ __forceinline__ double sum8(const double* __restrict__ x, int sx, int N)
{
    double m[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int i = 0;
    for (; i + 7 < N; i += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) m[k] += x[(i + k) * sx];
    }
    for (; i < N; ++i) m[0] += x[i * sx];
    return ((m[0] + m[1]) + (m[2] + m[3])) + ((m[4] + m[5]) + (m[6] + m[7]));
}

// Raw emission input of (row, state j): the table entry, the observation, or the symbol's B entry.
template <int EM>
__device__ __forceinline__ double em_load(const Emission& em, long long row, int j, int N)
{
    if (EM == EM_POBS) return em.pobs[row * N + j];
    if (EM == EM_GAUSS) return em.obs[row];
    return em.Bt[(long long)em.sym[row] * N + j];
}

// L1 prefetch of the emission input `ahead` frames further along the trajectory (sequential walks with few warps per SM
// cannot hide the DRAM latency of a load issued one step ahead)
template <int EM>
__device__ __forceinline__ void em_prefetch(const Emission& em, long long row, int j, int N)
{
    const void* p;
    if (EM == EM_POBS) p = em.pobs + row * N + j;
    else if (EM == EM_GAUSS) p = em.obs + row;
    else p = em.sym + row;
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}

template <int EM>
__device__ __forceinline__ double em_value(double raw, double mu, double sigma)
{
    if (EM == EM_GAUSS) return gauss_pdf(raw, mu, sigma);
    return raw;
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
// WARP1: the block is one warp carrying one team (17 <= N <= 32): the thread's column of A lives in registers and the
// row sums are warp shuffles, which halves the shared-memory traffic that bounds the general code.
template <int EM, bool WARP1>
__global__ void k_forward_team(const FwdArgs a)
{
    extern __shared__ double sm[];
    const int N = a.N, cpb = a.cpb;
    double* A_s = sm;                       // N*N, A[i*N+j]
    double* xb = A_s + N * N;               // 2 * cpb * N exchange slab
    const TeamGeom g = team_geometry(N, cpb);
    const int j = g.j;
    const bool jv = g.owns && j < N;

    for (int k = threadIdx.x; k < N * N; k += blockDim.x) A_s[k] = a.A[k];
    double Acol[WARP1 ? 32 : 1];
    if (WARP1) {
#pragma unroll
        for (int i = 0; i < 32; ++i) Acol[WARP1 ? i : 0] = (i < N && jv) ? a.A[i * N + j] : 0.0;
    }
    const double pi_j = jv ? a.pi[j] : 0.0;
    double mu = 0.0, sigma = 1.0;
    if (EM == EM_GAUSS && jv) { mu = a.em.mu[j]; sigma = a.em.sigma[j]; }
    __syncthreads();

    for (int base = blockIdx.x * cpb; base < a.ch.n; base += gridDim.x * cpb) {
        const int idx = base + g.team;
        const bool have = g.owns && idx < a.ch.n;
        int c = -1, len = 0, t0 = 0, tstart = 0, mode = 0;   // mode 0: pi, 1: uniform warm-up, 2: exact vector
        long long trow = 0;
        if (have) {
            c = a.ch.list ? a.ch.list[idx] : idx;
            len = a.ch.len[c];
            t0 = a.ch.t0[c];
            trow = a.ch.row0[c] - t0;
            if (t0 == 0) { tstart = 0; mode = 0; }
            else if (chain_exact_start(a.ch, c)) { tstart = t0 - 1; mode = 2; }
            else { tstart = max(0, t0 - (a.ch.warmv ? a.ch.warmv[c] : a.ch.warm)); mode = (tstart == 0) ? 0 : 1; }
        }
        const int npre = have ? (t0 - tstart) : 0;
        const int maxpre = block_max(npre);
        const int total = maxpre + block_max(len);
        const int tend = t0 + len;

        double ll = 0.0, cprev = 1.0;
        double vec_j = 0.0;
        if (have && mode == 2 && jv) vec_j = chain_start_vec(a.ch, a.hand_end, c, c - 1, N)[j];

        // depth-1 software prefetch of the emission input
        auto fetch = [&](int s) -> double {
            int t = t0 - maxpre + s;
            if (!have || !jv) return 0.0;
            t = min(max(t, tstart + (mode == 2 ? 1 : 0)), tend - 1);
            return em_load<EM>(a.em, trow + t, j, N);
        };
        double raw_next = fetch(0);

        for (int s = 0; s < total; ++s) {
            const int t = t0 - maxpre + s;
            const bool on = have && t >= tstart && t < tend;
            const bool init = on && t == tstart;
            const double raw = raw_next;
            raw_next = fetch(s + 1);
            double p = 0.0;
            if (on && jv && !(init && mode == 2)) p = em_value<EM>(raw, mu, sigma);
            bool anynz, anybig;
            team_any2(p != 0.0, p >= TINY_P, g, anynz, anybig);
            if (EM != EM_POBS && a.em.ignore_outliers && !anynz) { p = 1.0; anybig = true; }   // outputmodel.py:126-130
            const bool lifted = anynz && !anybig;
            if (lifted) p *= LIFT_P;
            const double* xprev = xb + ((s + 1) & 1) * cpb * N + g.team * N;
            double* xcur = xb + (s & 1) * cpb * N + g.team * N;
            double av = 0.0;
            if (on && jv) {
                if (init) {
                    av = (mode == 0) ? pi_j * p : ((mode == 1) ? p : vec_j);
                } else {
                    double m = 0.0;
                    if (WARP1) {
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if (i < N) m = fma(xprev[i], Acol[WARP1 ? i : 0], m);
                    } else {
                        m = dot8(xprev, 1, A_s + j, N, N);
                    }
                    if (cprev != 0.0) m /= cprev;
                    av = m * p;
                }
            }
            if (g.owns && j < N) xcur[j] = av;
            __syncthreads();
            double csum = 0.0;
            if (WARP1) csum = warp_sum(av);
            else if (g.owns) csum = sum8(xcur, 1, N);
            if (on && jv) {
                const double outv = (csum != 0.0) ? av / csum : av;
                if (t >= t0) {
                    if (a.alpha) a.alpha[(trow + t) * N + j] = outv;
                    if (j == 0) ll += lifted ? log(csum) - LIFT_LOG : log(csum);
                    if (t == tend - 1) a.hand_end[(long long)c * N + j] = outv;
                } else if (t == t0 - 1) {
                    a.hand_used[(long long)c * N + j] = outv;
                }
            }
            cprev = csum;
        }
        if (have && j == 0) a.chain_ll[c] = ll;
        __syncthreads();   // slab reuse by the next chain group
    }
}

// ------------------------------------------------------------------------------------------------
// backward (literal: writes beta) and backward + sufficient statistics (fused E-step)
// ------------------------------------------------------------------------------------------------
// Walks frames f = fstart .. t0 downwards.  At frame f the team owns the UNNORMALISED backward
// vector b(f) (thread j holds b_j); exchange 1 publishes (w_j, b_j) with w_j = p_{f,j} b_j, which gives
// sb(f) = sum_j b_j, the normalised beta_f = b/sb, and b(f-1)_i = sum_j A_ij w_j / sb(f).
// STATS: exchange 2 publishes (g_i, alpha_{f-1,i}, b(f-1)_i) with g_i = alpha_{f-1,i} b(f-1)_i, whose sum
// S normalises both gamma_{f-1} = g/S and xi_{f-1} = alpha_{f-1,i} A_ij w_j / (sb S)  (_hidden.c:168-180),
// so gamma and xi are reduced on chip and never written unless a.gamma is given.
template <int EM, bool STATS, bool WARP1>
__global__ void k_backward_team(const BwdArgs a)
{
    extern __shared__ double sm[];
    const int N = a.N, cpb = a.cpb;
    double* At_s = sm;                          // N*N, At[j*N+i] = A[i][j]
    double* xb = At_s + N * N;                  // 2 * cpb * (3N) exchange slab.  literal: exchange 1 double-buffered
                                                // (one barrier per step); STATS: exchange 1 in the first half, exchange 2
                                                // in the second (two barriers per step make single buffers safe)
    double* Cacc = xb + 2 * cpb * 3 * N;        // STATS: cpb * N*N   (column j owned by thread j)
    const TeamGeom g = team_geometry(N, cpb);
    const int j = g.j;
    const bool jv = g.owns && j < N;

    for (int k = threadIdx.x; k < N * N; k += blockDim.x) {
        const int i = k / N, jj = k - i * N;
        At_s[jj * N + i] = a.A[k];
    }
    if (STATS) for (int k = threadIdx.x; k < cpb * N * N; k += blockDim.x) Cacc[k] = 0.0;
    double Arow[WARP1 ? 32 : 1];             // WARP1: A[j][i'] and the thread's column of the xi accumulator in registers
    double Ccol[(WARP1 && STATS) ? 32 : 1];
    if (WARP1) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            Arow[WARP1 ? i : 0] = (i < N && jv) ? a.A[j * N + i] : 0.0;
            if (STATS) Ccol[(WARP1 && STATS) ? i : 0] = 0.0;
        }
    }
    double mu = 0.0, sigma = 1.0;
    if (EM == EM_GAUSS && jv) { mu = a.em.mu[j]; sigma = a.em.sigma[j]; }
    double st_g0 = 0.0, st_g = 0.0, st_gd = 0.0, st_gdd = 0.0;
    __syncthreads();

    for (int base = blockIdx.x * cpb; base < a.ch.n; base += gridDim.x * cpb) {
        const int idx = base + g.team;
        const bool have = g.owns && idx < a.ch.n;
        int c = -1, len = 0, t0 = 0, T = 0, e = 0, fstart = 0, mode = 0;  // mode 0: ones (exact or warm), 2: exact vector
        bool virt = false;                                                 // chain ends its trajectory
        long long trow = 0;
        if (have) {
            c = a.ch.list ? a.ch.list[idx] : idx;
            len = a.ch.len[c];
            t0 = a.ch.t0[c];
            T = a.ch.T[c];
            trow = a.ch.row0[c] - t0;
            e = t0 + len;
            if (e >= T) { virt = true; fstart = STATS ? T : T - 1; }
            else if (chain_exact_start(a.ch, c)) { fstart = e; mode = 2; }
            else { fstart = min(T - 1, e + (a.ch.warmv ? a.ch.warmv[c] : a.ch.warm) - 1); }
        }
        // literal backward emits frame f at step f; STATS emits frame f-1 at step f.
        const int flast = STATS ? t0 + 1 : t0;
        const int npre = have ? (fstart - (e - 1)) : 0;           // steps before the chain's last frame is reached
        const int maxpre = block_max(npre);
        const int total = maxpre + block_max(have ? (e - flast) : 0);

        double b_own = 0.0;
        if (have && jv) b_own = (mode == 2) ? chain_start_vec(a.ch, a.hand_end, c, c + 1, N)[j] : 1.0;

        auto frame_of = [&](int s) -> int { return (e - 1) + maxpre - s; };
        auto fetch_em = [&](int s) -> double {
            int f = frame_of(s);
            if (!have || !jv) return 0.0;
            f = min(max(f, t0), T - 1);
            return em_load<EM>(a.em, trow + f, j, N);
        };
        auto fetch_alpha = [&](int s) -> double {
            int f = frame_of(s) - 1;
            if (!STATS || !have || !jv) return 0.0;
            f = min(max(f, t0), e - 1);
            return a.alpha[(trow + f) * N + j];
        };
        double raw_next = fetch_em(0), al_next = fetch_alpha(0);

        for (int s = 0; s < total; ++s) {
            const int f = frame_of(s);
            const bool on = have && f <= fstart && f >= flast;
            const bool isvirt = on && virt && STATS && f == T;      // virtual frame T: beta_{T-1} = 1/N
            const double raw = raw_next, al = al_next;
            raw_next = fetch_em(s + 1);
            al_next = fetch_alpha(s + 1);

            double p = 0.0;
            if (on && jv && !isvirt) p = em_value<EM>(raw, mu, sigma);
            {
                bool anynz, anybig;
                team_any2(p != 0.0, p >= TINY_P, g, anynz, anybig);
                if (EM != EM_POBS && a.em.ignore_outliers && !anynz) { p = 1.0; anybig = true; }
                if (anynz && !anybig) p *= LIFT_P;
            }
            // ---- exchange 1: (w_j, b_j) of frame f
            const int tm = WARP1 ? 0 : g.team;       // WARP1: the idle lanes (j >= N) read team 0's slab too
            double* x1 = xb + (STATS ? 0 : (s & 1)) * cpb * 3 * N + tm * 3 * N;
            const double w_own = p * b_own;
            if (jv) { x1[2 * j] = (on && !isvirt) ? w_own : 0.0; x1[2 * j + 1] = (on && !isvirt) ? b_own : 0.0; }
            __syncthreads();
            double sb = 0.0, bnew = 0.0;
            if (WARP1) {
                sb = warp_sum((jv && on && !isvirt) ? b_own : 0.0);
#pragma unroll
                for (int i = 0; i < 32; ++i)
                    if (i < N) bnew = fma(Arow[WARP1 ? i : 0], x1[2 * i], bnew);
                if (sb != 0.0) bnew /= sb;
                if (!jv) bnew = 0.0;
            } else if (g.owns) {
                sb = sum8(x1 + 1, 2, N);
                if (jv) {
                    bnew = dot8(At_s + j, N, x1, 2, N);                                         // sum_i' A[j][i'] w_i'
                    if (sb != 0.0) bnew /= sb;
                }
            }
            if (isvirt) { bnew = 1.0; sb = 1.0; }
            if (on && jv && !isvirt) {
                const double beta_f = (sb != 0.0) ? b_own / sb : b_own;
                if (!STATS) {
                    if (f < e) a.beta[(trow + f) * N + j] = beta_f;
                    if (f == t0 && t0 > 0) a.hand_end[(long long)c * N + j] = beta_f;
                }
                if (f == e) a.hand_used[(long long)c * N + j] = beta_f;
            }
            if (STATS) {
                // ---- exchange 2: (g_i, alpha_{f-1,i}, b(f-1)_i); emits frame f-1 when it lies in the chain
                const bool emit = on && (f - 1) < e;           // f-1 >= t0 holds because f >= flast = t0+1
                double* x2 = xb + cpb * 3 * N + tm * 3 * N;
                const double g_own = emit ? al * bnew : 0.0;
                if (jv) { x2[3 * j] = g_own; x2[3 * j + 1] = emit ? al : 0.0; x2[3 * j + 2] = emit ? bnew : 0.0; }
                __syncthreads();
                double S = 0.0, sbn = 0.0;
                if (WARP1) {                                 // every lane of the warp takes part in the shuffles
                    S = warp_sum(jv ? g_own : 0.0);
                    sbn = warp_sum((jv && emit) ? bnew : 0.0);
                }
                if (g.owns) {
                    if (!WARP1) {
                        S = sum8(x2, 3, N);
                        sbn = sum8(x2 + 2, 3, N);
                    }
                    if (emit && jv) {
                        const long long row = trow + (f - 1);
                        // transition f-1 -> f : C'[i][j] += alpha_{f-1,i} * w_j / (sb * S)
                        if (!isvirt) {
                            double wn = w_own;
                            if (sb != 0.0) wn /= sb;
                            wn /= S;
                            if (WARP1) {
#pragma unroll
                                for (int i = 0; i < 32; ++i)
                                    if (i < N) Ccol[(WARP1 && STATS) ? i : 0] = fma(x2[3 * i + 1], wn, Ccol[(WARP1 && STATS) ? i : 0]);
                            } else {
                                // column j of the team's xi accumulator: eight read-modify-writes in flight at a time
                                // (a rolled loop exposes the shared-memory round trip of every single one)
                                double* Cc = Cacc + g.team * N * N + j;
                                int i = 0;
                                for (; i + 7 < N; i += 8) {
                                    double cv[8], xv[8];
#pragma unroll
                                    for (int k = 0; k < 8; ++k) { cv[k] = Cc[(i + k) * N]; xv[k] = x2[3 * (i + k) + 1]; }
#pragma unroll
                                    for (int k = 0; k < 8; ++k) Cc[(i + k) * N] = fma(xv[k], wn, cv[k]);
                                }
                                for (; i < N; ++i) Cc[i * N] = fma(x2[3 * i + 1], wn, Cc[i * N]);
                            }
                        }
                        const double gam = g_own / S;
                        st_g += gam;
                        if (f - 1 == 0) st_g0 += gam;
                        if (EM == EM_GAUSS) {
                            const double d = a.em.obs[row] - mu;
                            st_gd = fma(gam, d, st_gd);
                            st_gdd = fma(gam, d * d, st_gdd);
                        }
                        if (EM == EM_DISC && a.Bnum) atomicAdd(a.Bnum + (long long)j * a.em.M + a.em.sym[row], gam);
                        if (a.gamma) a.gamma[row * N + j] = gam;
                        if (f - 1 == t0 && t0 > 0) a.hand_end[(long long)c * N + j] = (sbn != 0.0) ? bnew / sbn : bnew;
                    }
                }
            }
            if (on) b_own = bnew;     // teams that have not started yet keep their initial vector
        }
        __syncthreads();
    }

    if (STATS) {
        // per-block partial statistics: [C' (N*N) | gamma0 (N) | sum gamma (N) | sum gamma d (N) | sum gamma d^2 (N)]
        const int nstat = N * N + 4 * N;
        double* out = a.partials + (long long)blockIdx.x * nstat;
        if (WARP1 && jv) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
                if (i < N) Cacc[i * N + j] = Ccol[(WARP1 && STATS) ? i : 0];
        }
        __syncthreads();
        for (int k = threadIdx.x; k < N * N; k += blockDim.x) {
            double v = 0.0;
            for (int tm = 0; tm < cpb; ++tm) v += Cacc[tm * N * N + k];
            out[k] = v;
        }
        double* red = xb;                         // reuse slab: cpb * 4 * N  <= 2*cpb*3N
        __syncthreads();
        if (jv) {
            double* r = red + g.team * 4 * N;
            r[j] = st_g0; r[N + j] = st_g; r[2 * N + j] = st_gd; r[3 * N + j] = st_gdd;
        }
        __syncthreads();
        for (int k = threadIdx.x; k < 4 * N; k += blockDim.x) {
            double v = 0.0;
            for (int tm = 0; tm < cpb; ++tm) v += red[tm * 4 * N + k];
            out[N * N + k] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Viterbi (one team per trajectory, sequential in t, bit-exact operation order)
// ------------------------------------------------------------------------------------------------
// _hidden.c:229-265: h_i = v_i*A[i][j]; first maximum with strict '>'; vnext_j = (p_j*v_best)*A[best][j];
// sum over j in increasing order; every entry divided by the sum.  __dmul_rn/__dadd_rn/__ddiv_rn keep the
// compiler from contracting products into FMAs, which would change roundings and, in near ties, paths.
template <int EM, typename PtrT>
__global__ void k_viterbi_team(const VitArgs a)
{
    // CHASE (N <= 256): the kernel writes the map F[t][s'] = state at t given state s' at t+1 (i.e. the back-pointers
    // shifted by one frame, and the final argmax in the last row); the path is then resolved in parallel by the
    // segment-wise map composition of sample_kernels.cu (k_chase_*).  Otherwise thread 0 backtraces in place.
    constexpr bool CHASE = (sizeof(PtrT) == 1);
    extern __shared__ double sm[];
    const int N = a.N, cpb = a.cpb;
    double* A_s = sm;                         // N*N
    double* ub = A_s + N * N;                 // cpb * N  unnormalised row
    double* vb = ub + cpb * N;                // cpb * N  normalised row
    const TeamGeom g = team_geometry(N, cpb);
    const int j = g.j;
    const bool jv = g.owns && j < N;
    for (int k = threadIdx.x; k < N * N; k += blockDim.x) A_s[k] = a.A[k];
    double mu = 0.0, sigma = 1.0;
    if (EM == EM_GAUSS && jv) { mu = a.em.mu[j]; sigma = a.em.sigma[j]; }
    const double pi_j = jv ? a.pi[j] : 0.0;
    PtrT* bp = reinterpret_cast<PtrT*>(a.backptr);
    __syncthreads();
    const bool onewarp = (blockDim.x == 32);
    auto team_sync = [&]() { if (onewarp) __syncwarp(); else __syncthreads(); };

    for (int base = blockIdx.x * cpb; base < a.K; base += gridDim.x * cpb) {
        const int k = base + g.team;
        const bool have = g.owns && k < a.K;
        long long row0 = 0;
        int T = 0;
        if (have) { row0 = a.offsets[k]; T = (int)(a.offsets[k + 1] - row0); }
        const int Tmax = block_max(T);
        double* urow = ub + (g.owns ? g.team : 0) * N;
        double* vrow = vb + (g.owns ? g.team : 0) * N;
        double raw_next = (have && jv && T > 0) ? em_load<EM>(a.em, row0, j, N) : 0.0;
        for (int t = 0; t < Tmax; ++t) {
            const bool on = have && t < T;
            const double raw = raw_next;
            if (have && jv && t + 1 < T) raw_next = em_load<EM>(a.em, row0 + t + 1, j, N);
            if (have && jv && t + 64 < T && (EM == EM_POBS || (t & 3) == 0)) em_prefetch<EM>(a.em, row0 + t + 64, j, N);
            double p = 0.0;
            if (on && jv) p = em_value<EM>(raw, mu, sigma);
            if (EM != EM_POBS && a.em.ignore_outliers) {
                const bool anynz = team_any(p != 0.0, g);
                if (!anynz) p = 1.0;
            }
            double vn = 0.0;
            if (on && jv) {
                if (t == 0) {
                    vn = __dmul_rn(p, pi_j);
                } else {
                    int best = 0;
                    double m = __dmul_rn(vrow[0], A_s[j]);
                    for (int i = 1; i < N; ++i) {
                        const double h = __dmul_rn(vrow[i], A_s[i * N + j]);
                        if (h > m) { m = h; best = i; }
                    }
                    if (CHASE) bp[(row0 + t - 1) * N + j] = (PtrT)best;
                    else bp[(row0 + t) * N + j] = (PtrT)best;
                    vn = __dmul_rn(__dmul_rn(p, vrow[best]), A_s[best * N + j]);
                }
                urow[j] = vn;
            }
            team_sync();
            if (on && jv) {
                double ssum = 0.0;
                for (int i = 0; i < N; ++i) ssum = __dadd_rn(ssum, urow[i]);
                vrow[j] = __ddiv_rn(vn, ssum);      // finished teams keep their last row
            }
            team_sync();
        }
        // path[T-1] = first maximum of the last row (_hidden.c:268)
        if (have && jv && T > 0) {
            int best = 0;
            double m = vrow[0];
            for (int i = 1; i < N; ++i) if (vrow[i] > m) { m = vrow[i]; best = i; }
            if (CHASE) {
                bp[(row0 + T - 1) * N + j] = (PtrT)best;
            } else if (j == 0) {
                // the back-pointer rows were written by this block: a block-level fence suffices
                __threadfence_block();
                int* path = a.path + row0;
                path[T - 1] = best;
                for (int t = T - 2; t >= 0; --t) {
                    best = (int)bp[(row0 + t + 1) * N + best];
                    path[t] = best;
                }
            }
        }
        __syncthreads();
    }
}

template <typename K>
int set_smem(K kernel, size_t bytes)
{
    if (bytes > 48 * 1024) {
        if (bytes > 227 * 1024) return BHMM_ERR_UNSUPPORTED;
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
            return BHMM_ERR_CUDA;
    }
    return BHMM_OK;
}

int sm_count()
{
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

int persistent_grid(int groups, int threads, size_t smem)
{
    int per_sm = 32;
    if (threads > 32) per_sm = max(1, min(32, 2048 / threads));
    if (smem > 0) per_sm = max(1, min(per_sm, (int)((220 * 1024) / (smem + 1024))));
    const long long cap = (long long)sm_count() * per_sm;
    return (int)max(1LL, min((long long)groups, cap));
}

}  // namespace

static void team_shape_raw(int N, int* threads, int* cpb)
{
    if (N <= 32) { *threads = 32; *cpb = 32 / N; }
    else { *threads = ((N + 31) / 32) * 32; *cpb = 1; }
}

// what the planners see: chains per row of partial statistics (a block here, a warp in the opt-in panel family)
void team_shape(int N, int* threads, int* cpb)
{
    if (panel_enabled(N)) { panel_shape(N, threads, cpb); return; }
    team_shape_raw(N, threads, cpb);
}

template <int EM>
static int launch_forward_em(const FwdArgs& a, cudaStream_t st)
{
    int threads, cpb;
    team_shape_raw(a.N, &threads, &cpb);
    FwdArgs b = a;
    b.cpb = cpb;
    const size_t smem = sizeof(double) * ((size_t)a.N * a.N + 2 * (size_t)cpb * a.N);
    int rc = set_smem(k_forward_team<EM, false>, smem);
    if (rc) return rc;
    const int groups = (a.ch.n + cpb - 1) / cpb;
    if (groups <= 0) return BHMM_OK;
    if (threads == 32 && cpb == 1) k_forward_team<EM, true><<<persistent_grid(groups, threads, smem), threads, smem, st>>>(b);
    else k_forward_team<EM, false><<<persistent_grid(groups, threads, smem), threads, smem, st>>>(b);
    return BHMM_OK;
}

int launch_forward_team(const FwdArgs& a, int em, cudaStream_t st)
{
    if (a.N < 1 || a.N > 1024) return BHMM_ERR_UNSUPPORTED;
    if (panel_enabled(a.N) && panel_forward_ok(a, em)) return launch_forward_panel(a, em, st);
    switch (em) {
        case EM_POBS: return launch_forward_em<EM_POBS>(a, st);
        case EM_GAUSS: return launch_forward_em<EM_GAUSS>(a, st);
        case EM_DISC: return launch_forward_em<EM_DISC>(a, st);
    }
    return BHMM_ERR_INVALID;
}

int backward_stats_grid(int N, int n_chains)
{
    if (panel_enabled(N)) return panel_stats_rows(N, n_chains);
    int threads, cpb;
    team_shape_raw(N, &threads, &cpb);
    const size_t smem = sizeof(double) * ((size_t)N * N + 6 * (size_t)cpb * N + (size_t)cpb * N * N);
    return persistent_grid((n_chains + cpb - 1) / cpb, threads, smem);
}

template <int EM, bool STATS>
static int launch_backward_em(const BwdArgs& a, cudaStream_t st)
{
    int threads, cpb;
    team_shape_raw(a.N, &threads, &cpb);
    BwdArgs b = a;
    b.cpb = cpb;
    size_t smem = sizeof(double) * ((size_t)a.N * a.N + 6 * (size_t)cpb * a.N);
    if (STATS) smem += sizeof(double) * (size_t)cpb * a.N * a.N;
    int rc = set_smem(k_backward_team<EM, STATS, false>, smem);
    if (rc) return rc;
    const int groups = (a.ch.n + cpb - 1) / cpb;
    if (groups <= 0) return BHMM_OK;
    const int grid = STATS ? a.grid : persistent_grid(groups, threads, smem);
#ifndef TEAM_WARP1_STATS
#define TEAM_WARP1_STATS 0   // measured slower for the fused statistics kernel at N=32 (33 vs 25 ms); kept for forward and literal backward
#endif
    if (threads == 32 && cpb == 1 && (!STATS || TEAM_WARP1_STATS)) k_backward_team<EM, STATS, true><<<grid, threads, smem, st>>>(b);
    else k_backward_team<EM, STATS, false><<<grid, threads, smem, st>>>(b);
    return BHMM_OK;
}

int launch_backward_team(const BwdArgs& a, int em, bool stats, cudaStream_t st)
{
    if (a.N < 1 || a.N > 1024) return BHMM_ERR_UNSUPPORTED;
    // (a launch the panel kernel cannot take -- an unaligned caller buffer -- runs on the team kernel with a.grid blocks)
    if (stats && panel_enabled(a.N) && panel_backward_ok(a, em)) return launch_backward_stats_panel(a, em, st);
    if (stats) {
        switch (em) {
            case EM_POBS: return launch_backward_em<EM_POBS, true>(a, st);
            case EM_GAUSS: return launch_backward_em<EM_GAUSS, true>(a, st);
            case EM_DISC: return launch_backward_em<EM_DISC, true>(a, st);
        }
    } else {
        switch (em) {
            case EM_POBS: return launch_backward_em<EM_POBS, false>(a, st);
            case EM_GAUSS: return launch_backward_em<EM_GAUSS, false>(a, st);
            case EM_DISC: return launch_backward_em<EM_DISC, false>(a, st);
        }
    }
    return BHMM_ERR_INVALID;
}

template <int EM>
static int launch_viterbi_em(const VitArgs& a, cudaStream_t st)
{
    int threads, cpb;
    team_shape_raw(a.N, &threads, &cpb);
    VitArgs b = a;
    b.cpb = cpb;
    const size_t smem = sizeof(double) * ((size_t)a.N * a.N + 2 * (size_t)cpb * a.N);
    const int groups = (a.K + cpb - 1) / cpb;
    if (groups <= 0) return BHMM_OK;
    int rc;
    if (a.N <= 256) {
        rc = set_smem(k_viterbi_team<EM, unsigned char>, smem);
        if (rc) return rc;
        k_viterbi_team<EM, unsigned char><<<persistent_grid(groups, threads, smem), threads, smem, st>>>(b);
    } else {
        rc = set_smem(k_viterbi_team<EM, unsigned short>, smem);
        if (rc) return rc;
        k_viterbi_team<EM, unsigned short><<<persistent_grid(groups, threads, smem), threads, smem, st>>>(b);
    }
    return BHMM_OK;
}

int launch_viterbi_team(const VitArgs& a, int em, cudaStream_t st)
{
    if (a.N < 1 || a.N > 1024) return BHMM_ERR_UNSUPPORTED;
    if (panel_viterbi_ok(a.N)) return launch_viterbi_panel(a, em, st);
    switch (em) {
        case EM_POBS: return launch_viterbi_em<EM_POBS>(a, st);
        case EM_GAUSS: return launch_viterbi_em<EM_GAUSS>(a, st);
        case EM_DISC: return launch_viterbi_em<EM_DISC>(a, st);
    }
    return BHMM_ERR_INVALID;
}
