// bhmm_b200/csrc/lane_kernels.cuh -- small-N fast path ("lane" family): ONE THREAD PER CHAIN.
//
// For N <= 16 hidden states a whole chain fits in one thread's registers: alpha / beta vectors are register
// arrays indexed at compile time, the transition matrix and the emission constants are a __grid_constant__
// kernel parameter, so every A[i][j] is a constant-bank operand of the FP64 FMA and the N x N matvec is N*N
// back-to-back DFMAs with no loads, no shuffles and no barriers.  A warp carries 32 independent chains; the work
// that is scalar per chain (normalisation, reciprocal, log-likelihood) costs one instruction for 32 chains
// instead of one per 3 chains as in the team family (ncu, profiles/r1_v0_*: the team kernels are issue bound).
//
// Memory: the forward variables never leave the GPU in the fused E-step, so they are stored in a layout chosen
// for coalescing, not the reference's (T,N): alpha_il[group][frame][pair][lane] as double2, where group = chain/32,
// lane = chain%32, pair = state/2.  A warp's store of one state pair of one frame is 512 contiguous bytes.
// Observations are read straight from the caller's concatenated array: each lane streams its own chain
// (8 B per frame, 4 frames per 32 B sector, prefetched 8 frames ahead); L1 keeps the sector between uses.
//
// Emission: p_j = nrm_j * exp(-0.5 ((o - mu_j) * isg_j)^2) with exp() evaluated by fast_exp (Cody-Waite reduction
// by ln 2 + degree-11 near-minimax polynomial, < 1 ulp, tools/gen_exp_poly.py); the log-likelihood is the sum of
// log c_t, accumulated as a running mantissa product with integer exponent bookkeeping (one DMUL + integer ops per
// frame instead of a log()).  Results agree with the reference to ~1e-13 relative (tests: 1e-10).
//
// Statistics: xi needs an N x N accumulator per chain, too many registers for N = 10.  Since only the SUM over
// chains is wanted, the G lanes of a lane-group share the work: lane q accumulates rows [q*NH, (q+1)*NH) for all
// G chains of its group, receiving the other chains' w vector and its rows of u, gamma (and the observation) by
// warp shuffles.  gamma and xi are never written to memory unless a gamma buffer is requested.
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int LANE_THREADS = 64;
constexpr unsigned FULL = 0xffffffffu;

// build-time tunables (python bhmm_b200/build.py --name=v_x -DLANE_...=... builds a variant library next to the default
// one; tools/lane_sweep.py with BHMM_B200_LIB=<variant> times it on the GPU box)
#ifndef LANE_MINB_F
#define LANE_MINB_F 4        // minimum resident blocks per SM asked of the compiler, forward kernel
#endif
#ifndef LANE_MINB_B
#define LANE_MINB_B 4        // ... backward + statistics kernel
#endif
#ifndef LANE_FOLD_NRM
#define LANE_FOLD_NRM 1      // Gaussian normalisation constant folded into the exponent's argument (one FMA less per state)
#endif
#ifndef LANE_CONST_SMEM
#define LANE_CONST_SMEM 1    // 1: all model constants (A, mu, isg, nrm) are read from shared memory into vector registers
#endif                       //    (LDS broadcast) instead of the uniform datapath (LDCU / R2UR), whose 63 registers thrash
                             // 2: emission constants from shared memory, transition matrix through the uniform datapath
#ifndef LANE_KEEP_F
#define LANE_KEEP_F 40       // forward kernel: this many entries of A stay in registers for the whole kernel, the rest comes
#endif                       // from shared memory every step (30 .. 60 measure the same at N = 10)
#ifndef LANE_EXP_TABLE
#define LANE_EXP_TABLE 1     // exp() of the Gaussian emission: 0 = degree-11 polynomial on |r| <= ln2/2; 1 = 32-entry table of
#endif                       // 2^(j/32) in shared memory + degree-5 polynomial on |r| <= ln2/64 (6 FP64 instructions less
                             // per state; fetching the entry with warp shuffles instead was measured slower)
#ifndef LANE_EXP_REPL
#define LANE_EXP_REPL 0      // 1: the exp table is stored 16 times, lane l reads copy l & 15: every look-up is conflict free
#endif                       //    (2 wavefronts per LDS.64) whatever the 32 indices are; 0: one copy, the lanes' indices collide
constexpr int kExpCopies = LANE_EXP_REPL ? 16 : 1;
#ifndef LANE_AT_B
#define LANE_AT_B 0          // 1: the backward kernel reads a TRANSPOSED copy of A, so that the N entries one column step of
#endif                       //    b = A w needs are contiguous (whole LDS.128 pairs consumed at once)
#ifndef LANE_UNROLL_F
#define LANE_UNROLL_F 1      // unroll factor of the run loops over the chain fast path (forward / backward kernel)
#endif
#ifndef LANE_UNROLL_B
#define LANE_UNROLL_B 1
#endif
constexpr int kUnrollF = LANE_UNROLL_F, kUnrollB = LANE_UNROLL_B;
#ifndef LANE_ALPHA_PREFETCH
#define LANE_ALPHA_PREFETCH 1        // backward kernel: L1 prefetch of the next step's forward variables for N <= MAXN
#endif                               // (N = 3: -21 %, N = 8: -10 % kernel time; N = 10: no gain, a step is long enough)
#ifndef LANE_ALPHA_PREFETCH_MAXN
#define LANE_ALPHA_PREFETCH_MAXN 8
#endif
#ifndef LANE_SAMPLE_AHEAD
#define LANE_SAMPLE_AHEAD 2          // sampler: frames ahead of the L1 prefetch of the forward variables
#endif
#ifndef LANE_PF
#define LANE_PF 1            // depth of the register ring of prefetched observations: with the L1 prefetch of the next cache
                             // line one step ahead is enough (4 -> 1: -1.4 % at N = 10, fewer registers and moves)
#endif
#ifndef LANE_OBS_PREFETCH
#define LANE_OBS_PREFETCH 1  // prefetch the next cache line of the lane's observations into L1 (the register ring's
#endif                       // rotation waits for the newest load, so its effective distance is one step)
#ifndef LANE_XCH_MIN_G
#define LANE_XCH_MIN_G 4     // lane groups of at least this size exchange their rows of u and gamma through shared memory
#endif
#ifndef LANE_G_MID
#define LANE_G_MID 4         // lanes sharing the xi accumulator rows for 9 <= N <= 12
#endif

__device__ __forceinline__ void prefetch_l1(const void* p)
{
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}

// pairwise (tree) sum of a register array: depth log2(N) instead of N-1 dependent DADDs
template <int N>
__device__ __forceinline__ double tree_sum(const double (&v)[N])
{
    double t[N];
#pragma unroll
    for (int j = 0; j < N; ++j) t[j] = v[j];
#pragma unroll
    for (int w = 1; w < N; w <<= 1) {
#pragma unroll
        for (int j = 0; j + w < N; j += 2 * w) t[j] += t[j + w];
    }
    return t[0];
}

// exp() constants live in constant memory so that each one is a constant-bank operand of its DFMA (as 64-bit
// literals they cost two UMOVs per use).  [0..9] = c11..c2 of the degree-11 polynomial (tools/gen_exp_poly.py),
// [10] = log2(e), [11] = ln2 high part, [12] = ln2 low part (fdlibm split).
__constant__ double EXPK[13] = {
    0x1.af632a0f7e2cep-26, 0x1.28b4101c77212p-22, 0x1.71ddf56d8deb5p-19, 0x1.a01991a10d9aep-16,
    0x1.a01a01b1461c5p-13, 0x1.6c16c1880029fp-10, 0x1.111111110f21ep-7,  0x1.555555554f0bap-5,
    0x1.555555555555ap-3,  0x1.0000000000011p-1,
    1.4426950408889634074, 6.93147180369123816490e-01, 1.90821492927058770002e-10};

// Table variant: exp(x) = 2^k 2^(j/32) exp(r), 32 k + j = rint(32 x / ln 2), |r| <= ln2/64.  EXPK2 = c5..c2 of the
// degree-5 Chebyshev-node interpolant of exp on that interval (relative error 1.4e-16), 32/ln2, ln2/32.  The reduction
// is a single FMA: the rounding of ln2/32 costs |x| 8e-17 relative, below the rounding of x itself.
__constant__ double EXPK2[6] = {0x1.11115c0cff61ap-7, 0x1.5555d88e3ae37p-5, 0x1.5555555547d22p-3, 0x1.ffffffffd0b4bp-2,
                                0x1.71547652b82fep+5, 0x1.62e42fefa39efp-6};
__constant__ double EXPT[32] = {
    0x1.0000000000000p+0, 0x1.059b0d3158574p+0, 0x1.0b5586cf9890fp+0, 0x1.11301d0125b51p+0,
    0x1.172b83c7d517bp+0, 0x1.1d4873168b9aap+0, 0x1.2387a6e756238p+0, 0x1.29e9df51fdee1p+0,
    0x1.306fe0a31b715p+0, 0x1.371a7373aa9cbp+0, 0x1.3dea64c123422p+0, 0x1.44e086061892dp+0,
    0x1.4bfdad5362a27p+0, 0x1.5342b569d4f82p+0, 0x1.5ab07dd485429p+0, 0x1.6247eb03a5585p+0,
    0x1.6a09e667f3bcdp+0, 0x1.71f75e8ec5f74p+0, 0x1.7a11473eb0187p+0, 0x1.82589994cce13p+0,
    0x1.8ace5422aa0dbp+0, 0x1.93737b0cdc5e5p+0, 0x1.9c49182a3f090p+0, 0x1.a5503b23e255dp+0,
    0x1.ae89f995ad3adp+0, 0x1.b7f76f2fb5e47p+0, 0x1.c199bdd85529cp+0, 0x1.cb720dcef9069p+0,
    0x1.d5818dcfba487p+0, 0x1.dfc97337b9b5fp+0, 0x1.ea4afa2a490dap+0, 0x1.f50765b6e4540p+0};

__device__ __noinline__ double slow_exp(double x) { return exp(x); }

// Gaussian emission of one frame for all N states, evaluated "vertically": every stage of the exp() (range
// reduction by ln 2, Horner steps, exponent insertion) is issued for all states before the next stage, so the N
// dependent chains interleave and hide the FP64 latency.  exp(x) = 2^n exp(r), n = rint(x/ln2), |r| <= ln2/2,
// degree-11 near-minimax polynomial (< 1 ulp).  The main path is branch free; states whose argument lies below
// -708 (result denormal or zero) or is NaN are redone with the library exp() in a rarely taken tail.
template <int N, int TB, typename CV>
__device__ __forceinline__ void emission_gauss(const CV& P, double o, int ignore_outliers, double (&p)[N])
{
    const double MAGIC = 6755399441055744.0;                 // 1.5 * 2^52
    double x[N], t[N], r[N];
    // x = log(nrm) - ((o - mu) * isg/sqrt2)^2 in one FMA: the normalisation constant rides in the exponent's
    // argument (same half-ulp rounding of x as without it) instead of costing a multiplication at the end
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const double d = (o - P.mu[j]) * P.isg[j];
#if LANE_FOLD_NRM
        x[j] = fma(-d, d, P.nrm[j]);
#else
        x[j] = -(d * d);
#endif
    }
    if constexpr (TB == 0) {
#pragma unroll
        for (int j = 0; j < N; ++j) t[j] = fma(x[j], EXPK[10], MAGIC);
#pragma unroll
        for (int j = 0; j < N; ++j) {
            const double n = t[j] - MAGIC;
            r[j] = fma(n, -EXPK[11], x[j]);
            r[j] = fma(n, -EXPK[12], r[j]);
        }
#pragma unroll
        for (int j = 0; j < N; ++j) p[j] = fma(EXPK[0], r[j], EXPK[1]);
#pragma unroll
        for (int k = 2; k < 10; ++k) {
#pragma unroll
            for (int j = 0; j < N; ++j) p[j] = fma(p[j], r[j], EXPK[k]);
        }
#pragma unroll
        for (int j = 0; j < N; ++j) p[j] = fma(p[j], r[j], 1.0);
#pragma unroll
        for (int j = 0; j < N; ++j) p[j] = fma(p[j], r[j], 1.0);
#pragma unroll
        for (int j = 0; j < N; ++j) {
            const int ni = __double2loint(t[j]);
            p[j] = __longlong_as_double(__double_as_longlong(p[j]) + ((long long)ni << 52));
#if !LANE_FOLD_NRM
            p[j] *= P.nrml[j];          // (comparison build only)
#endif
        }
    } else {
#pragma unroll
        for (int j = 0; j < N; ++j) t[j] = fma(x[j], EXPK2[4], MAGIC);
#pragma unroll
        for (int j = 0; j < N; ++j) r[j] = fma(t[j] - MAGIC, -EXPK2[5], x[j]);
        // 2^k 2^(j/32) as one double: the table's high words are stored minus (j << 15), so adding kk << 15
        // (kk = 32 k + j) leaves hi(2^(j/32)) + (k << 20)
        double tb[N];
#pragma unroll
        for (int j = 0; j < N; ++j) {
            const int kk = __double2loint(t[j]);
            const double e = LANE_EXP_REPL ? P.tab[((kk & 31) << 4) + (threadIdx.x & 15)] : P.tab[kk & 31];
            tb[j] = __hiloint2double(__double2hiint(e) + (kk << 15), __double2loint(e));
        }
#pragma unroll
        for (int j = 0; j < N; ++j) p[j] = fma(EXPK2[0], r[j], EXPK2[1]);
#pragma unroll
        for (int k = 2; k < 4; ++k) {
#pragma unroll
            for (int j = 0; j < N; ++j) p[j] = fma(p[j], r[j], EXPK2[k]);
        }
#pragma unroll
        for (int j = 0; j < N; ++j) p[j] = fma(p[j], r[j], 1.0);
#pragma unroll
        for (int j = 0; j < N; ++j) p[j] = fma(p[j], r[j], 1.0);
#pragma unroll
        for (int j = 0; j < N; ++j) {
            p[j] *= tb[j];
#if !LANE_FOLD_NRM
            p[j] *= P.nrml[j];          // (comparison build only)
#endif
        }
    }
    // tail test on the high words with integer instructions: x < -708 (result denormal or zero), x > 708 or x not
    // finite  <=>  max_j (unsigned) hi(x_j) > hi(-708.0)  or  max_j (signed) hi(x_j) > hi(708.0)
    {
        unsigned umax = (unsigned)__double2hiint(x[0]);
        int smax = __double2hiint(x[0]);
#pragma unroll
        for (int j = 1; j < N; ++j) {
            umax = max(umax, (unsigned)__double2hiint(x[j]));
            smax = max(smax, __double2hiint(x[j]));
        }
        if (umax > 0xC0862000u || smax > 0x40862000) {
            // Far states are common (any state more than 37.6 sigma away from the observation lands here), so the
            // usual case is cheap: x <= -746 underflows to exactly zero.  Only the thin band whose result is
            // denormal, overflow and non-finite arguments go through the library exp(), out of line.
            // The reference multiplies exp(-d^2) by the normalisation constant (_gaussian.c:18-20): its density is exactly zero
            // as soon as exp(-d^2) underflows (-d^2 < -745.13...), whatever the constant -- and an all-zero row is what fires
            // the outlier rule (outputmodel.py:119-131).  With the constant folded into the argument a narrow state (constant
            // > 1) would keep a denormal density in the band in between and the frame would not count as an outlier, so the
            // zero is decided from the un-normalised argument here, off the fast path.  (The band is reachable only through
            // this block while log(constant) < 37, i.e. sigma > 3e-17; smaller sigmas run on the team kernels.)
#pragma unroll
            for (int j = 0; j < N; ++j) {
                const unsigned hx = (unsigned)__double2hiint(x[j]);
#if LANE_FOLD_NRM
                if (x[j] - P.nrm[j] < -745.1332191019412) {
                    p[j] = 0.0;
                } else
#endif
                if (hx >= 0xC0875000u && hx <= 0xFFF00000u) {
                    p[j] = 0.0;
                } else if ((hx & 0x7fffffffu) > 0x40862000u) {
                    p[j] = slow_exp(x[j]);
#if !LANE_FOLD_NRM
                    p[j] *= P.nrml[j];
#endif
                }
            }
        }
    }
    int nzbits = 0;
#pragma unroll
    for (int j = 0; j < N; ++j) nzbits |= __double2hiint(p[j]) | __double2loint(p[j]);
    const bool anynz = (nzbits & 0x7fffffff) != 0 || nzbits != 0;
    if (ignore_outliers && !anynz) {
#pragma unroll
        for (int j = 0; j < N; ++j) p[j] = 1.0;            // outputmodel.py:126-130
    }
}

template <int N>
__device__ __forceinline__ void emission_disc(const LaneArgs& a, int sym, double (&p)[N])
{
    const double* src = a.Bt + (long long)sym * N;
    bool anynz = false;
#pragma unroll
    for (int j = 0; j < N; ++j) { p[j] = __ldg(src + j); anynz |= (p[j] != 0.0); }
    if (a.ignore_outliers && !anynz) {
#pragma unroll
        for (int j = 0; j < N; ++j) p[j] = 1.0;
    }
}

// log-likelihood accumulator: sum of log(c) kept as (integer exponent sum, mantissa product in [1,2)) plus a slow
// path for zero / denormal / non-finite scaling factors (log(0) = -inf like the reference, _hidden.c:34,62).
struct LogAcc {
    double prod = 1.0;
    long long esum = 0;
    double slow = 0.0;
    __device__ __forceinline__ void add(double c)
    {
        const int ec = (int)((__double_as_longlong(c) >> 52) & 0x7ff);
        if (ec == 0 || ec == 0x7ff || c < 0.0) { slow += log(c); return; }
        prod *= c;
        const long long b = __double_as_longlong(prod);
        esum += (long long)((b >> 52) & 0x7ff) - 1023;
        prod = __longlong_as_double((b & 0x800fffffffffffffLL) | 0x3ff0000000000000LL);
    }
    __device__ __forceinline__ double value() const { return (double)esum * 0.693147180559945309417 + log(prod) + slow; }
};

// Power-of-two renormalisation.  alpha and beta only have to stay inside the double range (gamma and xi are ratios), so
// they are rescaled by an exact power of two, and only when the largest component has drifted out of the band
// [1, 2^LANE_LAZY] (then it is put back to the middle; about one step in four has a lane that needs it).  The band
// lies ABOVE one: a lazily scaled vector is never smaller than the reference's sum-normalised one, so nothing underflows
// here that does not underflow there, and with LANE_LAZY = 480 the products alpha_i b_i of two such vectors and one
// step's growth (at most N x the largest emission density) stay far below 2^1024.  top_exponent() is the biased
// exponent of the largest component (integer max over the high words: off the FP64 pipe); when it is not a normal,
// comfortably large number (tiny, zero, negative, not finite) the caller normalises by the sum like the reference
// does (_hidden.c:57-63).
#ifndef LANE_LAZY
#define LANE_LAZY 480
#endif
template <int N>
__device__ __forceinline__ int top_exponent(const double (&v)[N])
{
    // ternary tree (the integer max takes three operands): depth 3 for N = 10 instead of a chain of 5
    int h[N];
#pragma unroll
    for (int j = 0; j < N; ++j) h[j] = __double2hiint(v[j]);
#pragma unroll
    for (int w = 1; w < N; w *= 3) {
#pragma unroll
        for (int j = 0; j < N; j += 3 * w) {
            if (j + w < N) h[j] = max(h[j], h[j + w]);
            if (j + 2 * w < N) h[j] = max(h[j], h[j + 2 * w]);
        }
    }
    return h[0] >> 20;
}
__device__ __forceinline__ bool regular_exponent(int e) { return e >= 64 && e < 2040; }
// v *= 2^-shift unless e lies in the band; returns the shift applied
template <int N>
__device__ __forceinline__ int rescale_pow2(double (&v)[N], int e)
{
    if ((unsigned)(e - 1023) <= (unsigned)LANE_LAZY) return 0;
    const int shift = max(e - (1023 + LANE_LAZY / 2), -1022);
    const double f = __hiloint2double((1023 - shift) << 20, 0);
#pragma unroll
    for (int j = 0; j < N; ++j) v[j] *= f;
    return shift;
}

__device__ __forceinline__ long long il_base(int c, int Lmax, int NP2)
{
    // index (in double2 units) of alpha_il[chain c][frame 0][pair 0]
    return ((long long)(c >> 5) * Lmax * NP2 << 5) + (c & 31);
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
// Every lane of a warp walks its own chain in lock step (frame index relative to the chain start is the same in all
// lanes, so the interleaved stores coalesce).  Each step is dispatched on a warp-uniform vote to one of three code
// paths: CHAIN (every lane is inside its chain: straight-line code, no predicates), WARM (every lane is warming up:
// no stores, no likelihood) and GENERAL (mixed lanes, first frames, hand-over frames).  The two fast paths are single
// basic blocks, which is what lets the compiler interleave the N exp() chains with the matvec.
template <int V> struct BoolTag2 { static constexpr int value = V; };

// Where the kernels read the model constants from: the kernel parameter itself (uniform datapath) or a copy of it in
// shared memory (plain LDS into vector registers).  Same member names either way.
template <int N>
struct ConstView {
    const double* A;
    const double* pi;
    const double* mu;
    const double* isg;
    const double* nrm;
    const double* nrml;
    const double* tab;      // 2^(j/32), j = 0..31, in shared memory (high words pre-shifted, see emission_gauss)
    const double* At;       // LANE_AT_B: A transposed
};
template <int N>
constexpr int lane_const_doubles() { return (int)(sizeof(LaneParams<N>) / sizeof(double)) + 32 * kExpCopies + (LANE_AT_B ? N * N : 0); }
template <int N>
__device__ __forceinline__ ConstView<N> make_const_view(const LaneParams<N>& P, double* smem)
{
    // layout of LaneParams is [A | pi | mu | isg | nrm | nrml], all doubles
    constexpr int TOT = sizeof(LaneParams<N>) / sizeof(double);
    const double* src = reinterpret_cast<const double*>(&P);
    for (int k = threadIdx.x; k < TOT; k += blockDim.x) smem[k] = src[k];
    for (int k = threadIdx.x; k < 32 * kExpCopies; k += blockDim.x) {
        const int j = k / kExpCopies;
        const double e = EXPT[j];
        smem[TOT + k] = __hiloint2double(__double2hiint(e) - (j << 15), __double2loint(e));
    }
    if (LANE_AT_B) {
        for (int k = threadIdx.x; k < N * N; k += blockDim.x) smem[TOT + 32 * kExpCopies + k] = src[(k % N) * N + k / N];
    }
    __syncthreads();
    ConstView<N> v;
    v.tab = smem + TOT;
    v.At = smem + TOT + 32 * kExpCopies;

#if LANE_CONST_SMEM == 2
    v.A = P.A;
#else
    v.A = smem;
#endif
    v.pi = smem + N * N; v.mu = v.pi + N; v.isg = v.mu + N; v.nrm = v.isg + N; v.nrml = v.nrm + N;
    return v;
}
enum { PATH_GENERAL = 0, PATH_CHAIN = 1, PATH_WARM = 2 };

template <int N, int EM, bool ROWMAJOR>
__global__ void __launch_bounds__(LANE_THREADS, LANE_MINB_F)
k_forward_lane(const __grid_constant__ LaneParams<N> Pk, const LaneArgs a)
{
    constexpr int NP2 = (N + 1) / 2;
    constexpr int PF = LANE_PF;
#if LANE_CONST_SMEM
    __shared__ double cs[lane_const_doubles<N>()];
    const ConstView<N> P = make_const_view<N>(Pk, cs);
#else
    const LaneParams<N>& P = Pk;
#endif
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const bool have = idx < a.ch.n;
    int c = 0, len = 0, t0 = 0, tstart = 0, mode = 0;        // mode 0: pi, 1: uniform warm-up, 2: exact vector
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
    const int maxpre = __reduce_max_sync(FULL, have ? (t0 - tstart) : 0);
    const int total = maxpre + __reduce_max_sync(FULL, len);
    const int tend = t0 + len;

    double al[N];
#pragma unroll
    for (int j = 0; j < N; ++j) al[j] = 0.0;
    if (have && mode == 2) {
        const double* hv = chain_start_vec(a.ch, a.hand_end, c, c - 1, N);
#pragma unroll
        for (int j = 0; j < N; ++j) al[j] = hv[j];
    }
    long long esum = 0;             // sum of the power-of-two shifts applied to the chain's own frames
    double slow = 0.0, log_start = 0.0, log_end = 0.0;
    double2* il = reinterpret_cast<double2*>(a.alpha_il) + il_base(c, a.Lmax, NP2);

    auto fetch = [&](int s) -> double {
        int t = t0 - maxpre + s;
        if (!have) return 0.0;
        t = min(max(t, tstart), tend - 1);
#ifdef LANE_DEBUG_NOFETCH
        return 0.37 + 1e-3 * (t & 1023);     // (timing experiment: no observation loads)
#endif
#if LANE_OBS_PREFETCH
        if (EM == EM_GAUSS) prefetch_l1(a.obs + trow + min(t + 16, tend - 1));
        else prefetch_l1(a.sym + trow + min(t + 32, tend - 1));
#endif
        if (EM == EM_GAUSS) return __ldg(a.obs + trow + t);
        return __longlong_as_double((long long)__ldg(a.sym + trow + t));
    };
    // observations are fetched PF frames ahead into a rotating register ring
    double ring[PF];
#pragma unroll
    for (int k = 0; k < PF; ++k) ring[k] = fetch(k);
    auto emission = [&](double rawv, double (&pv)[N]) {
        if (EM == EM_GAUSS) emission_gauss<N, LANE_EXP_TABLE>(P, rawv, a.ignore_outliers, pv);
        else emission_disc<N>(a, (int)__double_as_longlong(rawv), pv);
    };

    // part of the transition matrix is register resident (the forward kernel has the head-room)
    constexpr int KEEP = (LANE_KEEP_F < N * N) ? LANE_KEEP_F : N * N;
    double Areg[KEEP > 0 ? KEEP : 1];
#pragma unroll
    for (int k = 0; k < KEEP; ++k) Areg[k] = P.A[k];
    auto Aat = [&](int k) -> double { return (k < KEEP) ? Areg[k] : P.A[k]; };

    // v = (al A) o p
    auto propagate = [&](double (&v)[N], const double (&p)[N]) {
#pragma unroll
        for (int j = 0; j < N; ++j) v[j] = al[0] * Aat(j);
#pragma unroll
        for (int i = 1; i < N; ++i) {
#pragma unroll
            for (int j = 0; j < N; ++j) v[j] = fma(al[i], Aat(i * N + j), v[j]);
        }
#pragma unroll
        for (int j = 0; j < N; ++j) v[j] *= p[j];
    };

    // one frame of the recursion; PATH is a compile-time constant so that the fast paths carry no predicates
    auto step = [&](auto path_tag, int t, double raw, bool on) {
        constexpr int PATH = decltype(path_tag)::value;
        if (!on) return;
        double p[N];
        const bool init = (PATH == PATH_GENERAL) && (t == tstart);
        double v[N];
        if (init && mode == 2) {
#pragma unroll
            for (int j = 0; j < N; ++j) v[j] = al[j];
        } else {
            emission(raw, p);
            if (init) {
#pragma unroll
                for (int j = 0; j < N; ++j) v[j] = (mode == 0) ? P.pi[j] * p[j] : p[j];
            } else {
                propagate(v, p);
            }
        }
        // Renormalise.  Any positive scaling is equivalent for everything downstream (gamma and xi are ratios), so
        // the fast path scales by an exact power of two and the log-likelihood is kept as
        //   sum_t log c_t = log sigma_end - log sigma_start + ln2 * sum shift_t (+ slow-path terms),
        // sigma = sum_j alpha_j at the frame before the chain and at its last frame (telescoping product).
        const bool inchain = (PATH == PATH_CHAIN) || (PATH == PATH_GENERAL && t >= t0);
        const int e = top_exponent<N>(v);
        if (regular_exponent(e)) {
            const int shift = rescale_pow2<N>(v, e);
#pragma unroll
            for (int j = 0; j < N; ++j) al[j] = v[j];
            if (inchain) esum += shift;
        } else {
            const double csum = tree_sum<N>(v);
            const double rc = (csum != 0.0) ? 1.0 / csum : 1.0;
#pragma unroll
            for (int j = 0; j < N; ++j) al[j] = v[j] * rc;
            if (inchain) slow += log(csum);
        }
        if (inchain) {
            if (ROWMAJOR) {
                double* dst = a.alpha_rm + (trow + t) * N;
#pragma unroll
                for (int j = 0; j < N; ++j) dst[j] = al[j];
            } else {
                double2* dst = il + ((long long)(t - t0) * NP2 << 5);
#ifdef LANE_DEBUG_NOSTORE
                if (al[0] == 1.2345e-200)      // (timing experiment: the stores are never executed)
#endif
#pragma unroll
                for (int jp = 0; jp < NP2; ++jp)
                    __stcs(dst + (jp << 5), make_double2(al[2 * jp], (2 * jp + 1 < N) ? al[2 * jp + 1] : 0.0));
            }
        }
        if (PATH == PATH_GENERAL) {
            if (t == tend - 1 || t == t0 - 1) {          // hand-over frames: the sum-normalised vector is recorded
                const double sig = tree_sum<N>(al);
                const double rs = (sig != 0.0) ? 1.0 / sig : 1.0;
                double* dst = (t == tend - 1) ? a.hand_end : a.hand_used;
                if (t == tend - 1) log_end = log(sig);
                else log_start = (sig != 0.0) ? log(sig) : 0.0;    // an all-zero start keeps the chain's -inf
#pragma unroll
                for (int j = 0; j < N; ++j) dst[(long long)c * N + j] = al[j] * rs;
            }
        }
    };

    // The steps of a warp come in runs: between two special frames of any of its lanes (first frame, hand-over
    // frames, last frame) every lane keeps its class, so the class vote is taken once per run and the run itself is
    // a tight loop over one of the fast paths.
    auto next_raw = [&](int s) -> double {
        const double raw = ring[0];
#pragma unroll
        for (int k = 0; k + 1 < PF; ++k) ring[k] = ring[k + 1];
        ring[PF - 1] = fetch(s + PF);
        return raw;
    };
    int s = 0;
    while (s < total) {
        const int t = t0 - maxpre + s;
        // lane class: 0 idle, 1 plain frame inside the chain, 2 plain warm-up frame, 3 first / hand-over frame
        const bool on = have && t >= tstart && t < tend;
        const int cls = !on ? 0 : ((t == tstart || t == tend - 1 || t == t0 - 1) ? 3 : (t >= t0 ? 1 : 2));
        const unsigned m1 = __ballot_sync(FULL, cls == 1), m2 = __ballot_sync(FULL, cls == 2),
                       m3 = __ballot_sync(FULL, cls == 3);
        if (m3 || (m1 && m2) || !(m1 | m2)) {
            step(BoolTag2<PATH_GENERAL>(), t, next_raw(s), on);
            ++s;
            continue;
        }
        // plain steps this lane has left before its next special frame (idle lanes: before they start)
        const int rem = (cls == 1) ? tend - 2 - t : (cls == 2) ? t0 - 2 - t : (have && t < tstart) ? tstart - 1 - t : 0x7fffffff;
        const int run = 1 + __reduce_min_sync(FULL, rem);
        if (m1) {
#pragma unroll kUnrollF
            for (int k = 0; k < run; ++k, ++s) step(BoolTag2<PATH_CHAIN>(), t0 - maxpre + s, next_raw(s), on);
        } else {
            for (int k = 0; k < run; ++k, ++s) step(BoolTag2<PATH_WARM>(), t0 - maxpre + s, next_raw(s), on);
        }
    }
    // a chain whose last frame was renormalised by the slow path ends with sigma = 1: log_end = 0 is then exact
    if (have) a.chain_ll[c] = (log_end - log_start) + (double)esum * 0.693147180559945309417 + slow;
}

// ------------------------------------------------------------------------------------------------
// backward + sufficient statistics
// ------------------------------------------------------------------------------------------------
// value of arr[qsel*NH + ii] for a run-time qsel in [0,G): a chain of compile-time-indexed selects
template <int N, int G, int NH>
__device__ __forceinline__ double pick_row(const double (&arr)[N], int qsel, int ii)
{
    double v = arr[ii];
#pragma unroll
    for (int qq = 1; qq < G; ++qq)
        if (qq * NH + ii < N) v = (qsel == qq) ? arr[qq * NH + ii] : v;
    return v;
}

template <int N, int EM, int G>
__global__ void __launch_bounds__(LANE_THREADS, LANE_MINB_B)
k_backward_stats_lane(const __grid_constant__ LaneParams<N> Pk, const LaneArgs a)
{
    constexpr int NP2 = (N + 1) / 2;
    constexpr int NH = (N + G - 1) / G;
    constexpr int PF = LANE_PF;
    constexpr int NSTAT = N * N + 4 * N;
    __shared__ double red[(LANE_THREADS / 32) * NSTAT];
#if LANE_CONST_SMEM
    __shared__ double cs[lane_const_doubles<N>()];
    const ConstView<N> P = make_const_view<N>(Pk, cs);
#else
    const LaneParams<N>& P = Pk;
#endif

    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int q = lane & (G - 1);
    const bool have = idx < a.ch.n;
    int c = 0, len = 0, t0 = 0, T = 0, e = 0, fs = 0, mode = 0;   // mode 0: beta = 1/N at fs, 2: exact vector at fs = e
    long long trow = 0;
    if (have) {
        c = a.ch.list ? a.ch.list[idx] : idx;
        len = a.ch.len[c];
        t0 = a.ch.t0[c];
        T = a.ch.T[c];
        trow = a.ch.row0[c] - t0;
        e = t0 + len;
        if (e >= T) fs = T - 1;
        else if (chain_exact_start(a.ch, c)) { fs = e; mode = 2; }
        else fs = min(T - 1, e + (a.ch.warmv ? a.ch.warmv[c] : a.ch.warm) - 1);
    }
    const int maxpre = __reduce_max_sync(FULL, have ? (fs - (e - 1)) : 0);
    const int total = maxpre + __reduce_max_sync(FULL, len);

    double Cq[NH][N];
    double sg[NH], sgd[NH], sgdd[NH], muq[NH];
#pragma unroll
    for (int ii = 0; ii < NH; ++ii) {
        sg[ii] = sgd[ii] = sgdd[ii] = 0.0;
        muq[ii] = P.mu[min(q * NH + ii, N - 1)];
#pragma unroll
        for (int j = 0; j < N; ++j) Cq[ii][j] = 0.0;
    }
    double bt[N];                   // beta of frame f+1 (power-of-two scaled)
#pragma unroll
    for (int j = 0; j < N; ++j) bt[j] = 0.0;
    const double2* il = reinterpret_cast<const double2*>(a.alpha_il) + il_base(c, a.Lmax, NP2);

    auto frame_of = [&](int s) -> int { return (e - 1) + maxpre - s; };
    auto fetch = [&](int s) -> double {
        int f = frame_of(s);
        if (!have) return 0.0;
        f = min(max(f, t0), T - 1);
#if LANE_OBS_PREFETCH
        if (EM == EM_GAUSS) prefetch_l1(a.obs + trow + max(f - 16, t0));
        else prefetch_l1(a.sym + trow + max(f - 32, t0));
#endif
        if (EM == EM_GAUSS) return __ldg(a.obs + trow + f);
        return __longlong_as_double((long long)__ldg(a.sym + trow + f));
    };
    double ring[PF];
#pragma unroll
    for (int k = 0; k < PF; ++k) ring[k] = fetch(k);
    auto emission = [&](double rawv, double (&pv)[N]) {
        if (EM == EM_GAUSS) emission_gauss<N, LANE_EXP_TABLE>(P, rawv, a.ignore_outliers, pv);
        else emission_disc<N>(a, (int)__double_as_longlong(rawv), pv);
    };
    double raw_next = 0.0;          // emission input of frame f+1

    // statistics of one frame: lane q owns rows q*NH .. q*NH+NH-1 for every chain of its lane group.  The rows of u and
    // gamma that the partner lanes need depend on the partner's q: picking them out of registers costs a chain of selects
    // per value, so for G >= LANE_XCH_MIN_G they travel through shared memory instead (every lane stores its vectors
    // blocked by owner, 16-byte units, and reads block q of its partners: dynamic addressing is free there); w and the
    // observation, which every partner needs whole, stay on warp shuffles.
    constexpr bool XCH = (G >= LANE_XCH_MIN_G);
    constexpr int XU = NH;                       // 16-byte units per block: (u_0..u_NH-1, gamma_0..gamma_NH-1)
    __shared__ double2 xch[XCH ? (LANE_THREADS / 32) * G * XU * 32 : 1];
    double2* const xw = xch + (threadIdx.x >> 5) * (G * XU * 32);
    auto accumulate = [&](const double (&w)[N], const double (&u)[N], const double (&gam)[N], double o_f) {
        if (XCH) {
#pragma unroll
            for (int blk = 0; blk < G; ++blk) {
                double L[2 * NH];
#pragma unroll
                for (int ii = 0; ii < NH; ++ii) {
                    L[ii] = (blk * NH + ii < N) ? u[(blk * NH + ii < N) ? blk * NH + ii : 0] : 0.0;
                    L[NH + ii] = (blk * NH + ii < N) ? gam[(blk * NH + ii < N) ? blk * NH + ii : 0] : 0.0;
                }
#pragma unroll
                for (int k = 0; k < XU; ++k) xw[(blk * XU + k) * 32 + lane] = make_double2(L[2 * k], L[2 * k + 1]);
            }
            __syncwarp();
        }
#pragma unroll
        for (int d = 0; d < G; ++d) {
            double ur[NH], gr[NH];
            double od;
            if (XCH) {
                double L[2 * NH];
#pragma unroll
                for (int k = 0; k < XU; ++k) {
                    const double2 v = xw[(q * XU + k) * 32 + (lane ^ d)];
                    L[2 * k] = v.x;
                    L[2 * k + 1] = v.y;
                }
#pragma unroll
                for (int ii = 0; ii < NH; ++ii) { ur[ii] = L[ii]; gr[ii] = L[NH + ii]; }
                od = (d == 0) ? o_f : __shfl_xor_sync(FULL, o_f, d);
            } else if (d == 0) {
#pragma unroll
                for (int ii = 0; ii < NH; ++ii) {
                    ur[ii] = pick_row<N, G, NH>(u, q, ii);
                    gr[ii] = pick_row<N, G, NH>(gam, q, ii);
                }
                od = o_f;
            } else {
                // the partner lane^d owns rows (q^d)*NH..: send it those rows of my u and gamma, receive mine
#pragma unroll
                for (int ii = 0; ii < NH; ++ii) {
                    ur[ii] = __shfl_xor_sync(FULL, pick_row<N, G, NH>(u, q ^ d, ii), d);
                    gr[ii] = __shfl_xor_sync(FULL, pick_row<N, G, NH>(gam, q ^ d, ii), d);
                }
                od = __shfl_xor_sync(FULL, o_f, d);
            }
#pragma unroll
            for (int j = 0; j < N; ++j) {
                const double wj = (d == 0) ? w[j] : __shfl_xor_sync(FULL, w[j], d);
#pragma unroll
                for (int ii = 0; ii < NH; ++ii) Cq[ii][j] = fma(ur[ii], wj, Cq[ii][j]);
            }
#pragma unroll
            for (int ii = 0; ii < NH; ++ii) {
                sg[ii] += gr[ii];
                if (EM == EM_GAUSS) {
                    const double dd = od - muq[ii];
                    sgd[ii] = fma(gr[ii], dd, sgd[ii]);
                    sgdd[ii] = fma(gr[ii], dd * dd, sgdd[ii]);
                }
            }
        }
        if (XCH) __syncwarp();
    };

    // w = p o bt, b = A w
    auto back_propagate = [&](double (&b)[N], double (&w)[N], const double (&p)[N]) {
#pragma unroll
        for (int j = 0; j < N; ++j) w[j] = p[j] * bt[j];
#pragma unroll
        for (int i = 0; i < N; ++i) b[i] = (LANE_AT_B ? P.At[i] : P.A[i * N]) * w[0];
#pragma unroll
        for (int j = 1; j < N; ++j) {
#pragma unroll
            for (int i = 0; i < N; ++i) b[i] = fma(LANE_AT_B ? P.At[j * N + i] : P.A[i * N + j], w[j], b[i]);
        }
    };

    // one frame f: given beta_{f+1} (bt) and the emission input of f+1, form b = A (p_{f+1} o beta_{f+1}), emit the
    // statistics of frame f when it belongs to the chain, leave beta_f in bt
    auto step = [&](auto path_tag, int f, double raw, bool on) {
        constexpr int PATH = decltype(path_tag)::value;
        // CHAIN: straight-line code for all 32 lanes.  A lane whose chain has already ended (shorter chains of the
        // same warp) keeps computing on the clamped inputs and is masked where its contribution is formed (rS = 0),
        // which is cheaper than predicating the step and zeroing its w, u, gamma for the exchange.
        const bool act = (PATH == PATH_CHAIN) || on;
        const bool init = (PATH == PATH_GENERAL) && on && f == fs;
        const bool emit = (PATH == PATH_CHAIN) || (PATH == PATH_GENERAL && on && f < e);
        double w[N], u[N], gam[N];
        double o_f = 0.0;
        double p[N];
        if (PATH == PATH_GENERAL) {
#pragma unroll
            for (int j = 0; j < N; ++j) { w[j] = 0.0; u[j] = 0.0; gam[j] = 0.0; }
        }
        if (act) {
            // forward variables of frame f: issued first, consumed after the matvec
            double2 a2[NP2];
            if (emit) {
                const double2* src = il + ((long long)(on ? f - t0 : 0) * NP2 << 5);
#pragma unroll
                for (int jp = 0; jp < NP2; ++jp) a2[jp] = __ldcs(src + (jp << 5));
#if LANE_ALPHA_PREFETCH
                // the forward variables of the NEXT step (frame f-1) into L1: the loads above are consumed only half a
                // step after they are issued, and for few states a step is too short to cover the DRAM latency
                if (N <= LANE_ALPHA_PREFETCH_MAXN && on && f > t0) {
#pragma unroll
                    for (int jp = 0; jp < NP2; ++jp) prefetch_l1(src - (NP2 << 5) + (jp << 5));
                }
#endif
            }
            double b[N];
            if (init) {
                if (mode == 2) {
                    const double* hv = chain_start_vec(a.ch, a.hand_end, c, c + 1, N);
#pragma unroll
                    for (int j = 0; j < N; ++j) b[j] = hv[j];
                } else {
#pragma unroll
                    for (int j = 0; j < N; ++j) b[j] = 1.0;
                }
            } else {
                emission(raw_next, p);
                back_propagate(b, w, p);
            }
            const int eb = top_exponent<N>(b);
            if (emit) {
                // gamma_f = alpha_f o b / S ; xi_f = (alpha_f / S) (x) w   with S = sum_i alpha_f,i b_i
                double al[N], gi[N];
#pragma unroll
                for (int jp = 0; jp < NP2; ++jp) {
                    al[2 * jp] = a2[jp].x;
                    if (2 * jp + 1 < N) al[2 * jp + 1] = a2[jp].y;
                }
#pragma unroll
                for (int i = 0; i < N; ++i) gi[i] = al[i] * b[i];
                const double S = tree_sum<N>(gi);
                const double rS = (PATH == PATH_CHAIN && !on) ? 0.0 : 1.0 / S;
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    u[i] = al[i] * rS;
                    gam[i] = gi[i] * rS;
                }
                if (EM == EM_GAUSS) o_f = raw;
                if (PATH == PATH_GENERAL && f == 0) {
#pragma unroll
                    for (int i = 0; i < N; ++i) a.g0buf[(long long)c * N + i] = gam[i];
                }
                if (a.gamma && on) {
                    double* dst = a.gamma + (trow + f) * N;
#pragma unroll
                    for (int i = 0; i < N; ++i) dst[i] = gam[i];
                }
                if (EM == EM_DISC && a.Bnum && on) {
                    const int sy = (int)__double_as_longlong(raw);
#pragma unroll
                    for (int i = 0; i < N; ++i) atomicAdd(a.Bnum + (long long)i * a.M + sy, gam[i]);
                }
            }
            // beta only needs to stay in range: exact power-of-two scaling, and only when it has drifted; the
            // sum-normalised vector of the reference (_hidden.c:104-107) is formed only where it is handed over
            if (regular_exponent(eb)) {
                rescale_pow2<N>(b, eb);
#pragma unroll
                for (int i = 0; i < N; ++i) bt[i] = b[i];
            } else {
                const double sb = tree_sum<N>(b);
                const double rsb = (sb != 0.0) ? 1.0 / sb : 1.0;
#pragma unroll
                for (int i = 0; i < N; ++i) bt[i] = b[i] * rsb;
            }
            if (PATH == PATH_GENERAL && (f == e || (f == t0 && t0 > 0))) {
                const double sb = tree_sum<N>(bt);
                const double rsb = (sb != 0.0) ? 1.0 / sb : 1.0;
                double* dst = (f == e) ? a.hand_used : a.hand_end;
#pragma unroll
                for (int i = 0; i < N; ++i) dst[(long long)c * N + i] = bt[i] * rsb;
            }
            raw_next = raw;
        }
        if (PATH != PATH_WARM) accumulate(w, u, gam, o_f);
    };

    // runs of plain steps between the special frames of the warp's lanes, as in the forward kernel
    auto next_raw = [&](int s) -> double {
        const double raw = ring[0];                 // emission input of frame f
#pragma unroll
        for (int k = 0; k + 1 < PF; ++k) ring[k] = ring[k + 1];
        ring[PF - 1] = fetch(s + PF);
        return raw;
    };
    int s = 0;
    while (s < total) {
        const int f = frame_of(s);
        // lane class: 0 idle, 1 plain frame inside the chain, 2 plain warm-up frame, 3 first / hand-over / frame 0
        const bool on = have && f <= fs && f >= t0;
        const int cls = !on ? 0 : ((f == fs || f == e || f == t0 || f == 0) ? 3 : (f < e ? 1 : 2));
        const unsigned m1 = __ballot_sync(FULL, cls == 1), m2 = __ballot_sync(FULL, cls == 2),
                       m3 = __ballot_sync(FULL, cls == 3);
        if (m3 || (m1 && m2) || !(m1 | m2)) {
            step(BoolTag2<PATH_GENERAL>(), f, next_raw(s), on);
            ++s;
            continue;
        }
        const int rem = (cls == 1) ? f - t0 - 1 : (cls == 2) ? f - e - 1 : (have && f > fs) ? f - fs - 1 : 0x7fffffff;
        const int run = 1 + __reduce_min_sync(FULL, rem);
        if (m1) {
#pragma unroll kUnrollB
            for (int k = 0; k < run; ++k, ++s) step(BoolTag2<PATH_CHAIN>(), frame_of(s), next_raw(s), on);
        } else {
            for (int k = 0; k < run; ++k, ++s) step(BoolTag2<PATH_WARM>(), frame_of(s), next_raw(s), on);
        }
    }

    // ---- reduce over the lanes that own the same rows (lane bits >= log2 G), then over the block's warps
#pragma unroll
    for (int off = G; off < 32; off <<= 1) {
#pragma unroll
        for (int ii = 0; ii < NH; ++ii) {
            sg[ii] += __shfl_xor_sync(FULL, sg[ii], off);
            sgd[ii] += __shfl_xor_sync(FULL, sgd[ii], off);
            sgdd[ii] += __shfl_xor_sync(FULL, sgdd[ii], off);
#pragma unroll
            for (int j = 0; j < N; ++j) Cq[ii][j] += __shfl_xor_sync(FULL, Cq[ii][j], off);
        }
    }
    double* myred = red + (threadIdx.x >> 5) * NSTAT;
    if (lane < G) {
#pragma unroll
        for (int ii = 0; ii < NH; ++ii) {
            const int i = q * NH + ii;
            if (i < N) {
#pragma unroll
                for (int j = 0; j < N; ++j) myred[i * N + j] = Cq[ii][j];
                myred[N * N + i] = 0.0;                       // gamma0 travels through g0buf
                myred[N * N + N + i] = sg[ii];
                myred[N * N + 2 * N + i] = sgd[ii];
                myred[N * N + 3 * N + i] = sgdd[ii];
            }
        }
    }
    __syncthreads();
    double* out = a.partials + (long long)blockIdx.x * NSTAT;
    for (int k = threadIdx.x; k < NSTAT; k += blockDim.x) {
        double v = 0.0;
#pragma unroll
        for (int wp = 0; wp < LANE_THREADS / 32; ++wp) v += red[wp * NSTAT + k];
        out[k] = v;
    }
}

// ------------------------------------------------------------------------------------------------
// forward-filter / backward-sample on the interleaved forward variables
// ------------------------------------------------------------------------------------------------
// Given its uniform, the draw at frame t is a function F_t(s_{t+1}) of the next state only (sample_kernels.cu).  A chain
// does not know the state that enters it from the next chain, so pass 1 (SAMPLE_MAP) walks the chain backwards carrying
// ALL N hypothetical entering states (4 bits each in one 64-bit word).  The hypotheses coalesce after a few frames
// (F_t depends only weakly on the next state); from there on a single path is followed, written and counted.  The
// chains of a trajectory are then linked (k_chase_link), and pass 2 (SAMPLE_FIX) re-walks only the few frames before
// the coalescence with the now-known entering state.  Same draws as the serial reference for the same uniforms.
__device__ __forceinline__ void lane_philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0,
                                                  uint32_t k1)
{
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}

// identical to philox_uniform() of sample_kernels.cu: uniform in [0,1) keyed by seed, counter (ctr, row)
__device__ __forceinline__ double lane_philox_uniform(unsigned long long seed, unsigned long long ctr, long long row)
{
    uint32_t c0 = (uint32_t)row, c1 = (uint32_t)((unsigned long long)row >> 32);
    uint32_t c2 = (uint32_t)ctr, c3 = (uint32_t)(ctr >> 32);
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        lane_philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    const unsigned long long bits = ((unsigned long long)c0 << 32) | c1;
    return (double)(bits >> 11) * (1.0 / 9007199254740992.0);
}

// state drawn at a frame with forward variables al, uniform r, given next state v (ignored at a trajectory's last frame)
template <int N, bool EXACT>
__device__ __forceinline__ int lane_draw(const double (&al)[N], const double* __restrict__ A_s, int v, double r,
                                         bool last, bool& bad)
{
    double pv[N];
#pragma unroll
    for (int i = 0; i < N; ++i) pv[i] = last ? al[i] : __dmul_rn(al[i], A_s[i * N + v]);
    if (EXACT) {
        // the reference's arithmetic: sequential sum, division of every term, running sum (_hidden.c:283-319)
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) s = __dadd_rn(s, pv[i]);
        double acc = 0.0;
        int pick = -1;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            acc = __dadd_rn(acc, __ddiv_rn(pv[i], s));
            if (pick < 0 && acc >= r) pick = i;
        }
        if (pick < 0) { pick = N - 1; bad = true; }
        return pick;
    }
    // production: first i with sum_{k<=i} pv_k >= r * sum_k pv_k (no divisions)
    double s = pv[0];
#pragma unroll
    for (int i = 1; i < N; ++i) s += pv[i];
    const double thr = r * s;
    double acc = 0.0;
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        acc += pv[i];
        cnt += (acc < thr) ? 1 : 0;
    }
    if (!(s > 0.0)) bad = true;
    return min(cnt, N - 1);
}

template <int N, int EM, bool EXACT, bool FIXPASS>
__global__ void __launch_bounds__(LANE_THREADS)
k_sample_lane(const __grid_constant__ LaneParams<N> Pk, const LaneArgs a)
{
    constexpr int NP2 = (N + 1) / 2;
    constexpr int NI = N * N + 2 * N;                 // int counters per thread: C (N*N), n0 (N), frames per state (N)
    extern __shared__ unsigned char smraw[];
    double* A_s = reinterpret_cast<double*>(smraw);                       // N*N
    double* mom = A_s + N * N;                                            // [2N][LANE_THREADS] sum o, sum o^2
    int* cnts = reinterpret_cast<int*>(mom + 2 * N * LANE_THREADS);       // [NI][LANE_THREADS]
    for (int k = threadIdx.x; k < N * N; k += blockDim.x) A_s[k] = Pk.A[k];
    for (int k = threadIdx.x; k < 2 * N * LANE_THREADS; k += blockDim.x) mom[k] = 0.0;
    for (int k = threadIdx.x; k < NI * LANE_THREADS; k += blockDim.x) cnts[k] = 0;
    __syncthreads();

    const int tid = threadIdx.x;
    const int idx = blockIdx.x * blockDim.x + tid;
    const bool have = idx < a.ch.n;
    int c = 0, len = 0, t0 = 0, T = 0, e = 0;
    long long trow = 0;
    if (have) {
        c = idx;
        len = a.ch.len[c];
        t0 = a.ch.t0[c];
        T = a.ch.T[c];
        trow = a.ch.row0[c] - t0;
        e = t0 + len;
    }
    const double2* il = reinterpret_cast<const double2*>(a.alpha_il) + il_base(c, a.Lmax, NP2);
    bool bad = false;

    auto load_alpha = [&](int f, double (&al)[N]) {
        const double2* src = il + ((long long)(f - t0) * NP2 << 5);
#pragma unroll
        for (int jp = 0; jp < NP2; ++jp) {
            const double2 v2 = __ldcs(src + (jp << 5));
            al[2 * jp] = v2.x;
            if (2 * jp + 1 < N) al[2 * jp + 1] = v2.y;
        }
    };
    // Every step needs its forward variables at once (the draw depends on them), so they are prefetched into L1 two
    // steps ahead, together with the next cache line of the observations and of the supplied uniforms: without it a
    // step costs the full DRAM latency (3400 cycles per frame at the C3 shape).
    auto prefetch_step = [&](int f) {
        const int fa = f - LANE_SAMPLE_AHEAD;
        if (fa >= t0) {
            const double2* src = il + ((long long)(fa - t0) * NP2 << 5);
#pragma unroll
            for (int jp = 0; jp < NP2; ++jp) prefetch_l1(src + (jp << 5));
        }
        const int fo = max(f - 16, t0);
        if (EM == EM_GAUSS) prefetch_l1(a.obs + trow + fo);
        if (a.u_row) prefetch_l1(a.u_row + trow + fo);
    };
    auto uniform = [&](int f) -> double {
        return a.u_row ? __ldg(a.u_row + trow + f) : lane_philox_uniform(a.seed, a.sweep, trow + f);
    };
    auto count_frame = [&](int f, int st) {           // per-state frame count and observation moments
        cnts[(N * N + N + st) * LANE_THREADS + tid] += 1;
        if (f == 0) cnts[(N * N + st) * LANE_THREADS + tid] += 1;
        if (EM == EM_GAUSS) {
            const double o = __ldg(a.obs + trow + f);
            mom[st * LANE_THREADS + tid] += o;
            mom[(N + st) * LANE_THREADS + tid] += o * o;
        }
        if (a.path) a.path[trow + f] = st;
    };
    auto count_transition = [&](int st, int nxt) { cnts[(st * N + nxt) * LANE_THREADS + tid] += 1; };

    // uniform trip count per warp keeps the interleaved loads coalesced
    const int maxlen = __reduce_max_sync(FULL, len);
    if (!FIXPASS) {
        unsigned long long hyp = 0ULL;                // nibble s' = current state given entering state s'
#pragma unroll
        for (int sp = 0; sp < N; ++sp) hyp |= (unsigned long long)sp << (4 * sp);
        const unsigned long long ones = 0x1111111111111111ULL & ((N == 16) ? ~0ULL : ((1ULL << (4 * N)) - 1ULL));
        bool coalesced = false;
        int coal = t0 - 1, prev = 0;
        for (int k = 0; k < maxlen; ++k) {
            const int f = e - 1 - k;
            if (!have || f < t0) continue;
            double al[N];
            load_alpha(f, al);
            prefetch_step(f);
            const double r = uniform(f);
            const bool last = (f == T - 1);
            if (!coalesced) {
                unsigned long long nsp = 0ULL;        // nibble v = state drawn when the next state is v
#pragma unroll
                for (int v = 0; v < N; ++v) nsp |= (unsigned long long)lane_draw<N, EXACT>(al, A_s, v, r, last, bad) << (4 * v);
                unsigned long long nh = 0ULL;
#pragma unroll
                for (int sp = 0; sp < N; ++sp) {
                    const int cur = (int)((hyp >> (4 * sp)) & 15ULL);
                    nh |= ((nsp >> (4 * cur)) & 15ULL) << (4 * sp);
                }
                hyp = nh;
                if (hyp == (hyp & 15ULL) * ones) {
                    coalesced = true;
                    coal = f;
                    prev = (int)(hyp & 15ULL);
                    count_frame(f, prev);
                }
            } else {
                const int st = lane_draw<N, EXACT>(al, A_s, prev, r, last, bad);
                count_frame(f, st);
                count_transition(st, prev);
                prev = st;
            }
        }
        if (have) {
#pragma unroll
            for (int sp = 0; sp < N; ++sp)
                a.smap[(long long)c * N + sp] = (unsigned char)(coalesced ? prev : (int)((hyp >> (4 * sp)) & 15ULL));
            a.coal[c] = coal;
        }
    } else {
        // frames after the coalescence point: re-walk with the known entering state
        const int coal = have ? a.coal[c] : 0;
        int prev = (have && e < T) ? a.enter[c] : 0;
        for (int k = 0; k < maxlen; ++k) {
            const int f = e - 1 - k;
            if (!have || f < t0 || f < coal) continue;
            double al[N];
            load_alpha(f, al);
            prefetch_step(f);
            const double r = uniform(f);
            const bool last = (f == T - 1);
            const int st = lane_draw<N, EXACT>(al, A_s, prev, r, last, bad);
            if (f > coal) count_frame(f, st);
            if (!last) count_transition(st, prev);
            prev = st;
        }
    }
    if (bad) atomicExch(a.err, BHMM_ERR_SAMPLE);

    // ---- block reduction of the private counters (fixed order), then one atomic per counter and block
    __syncthreads();
    unsigned long long* gcnt = reinterpret_cast<unsigned long long*>(a.counts);
    for (int k = tid; k < NI; k += blockDim.x) {
        long long s = 0;
        for (int t = 0; t < LANE_THREADS; ++t) s += cnts[k * LANE_THREADS + t];
        if (s) atomicAdd(gcnt + k, (unsigned long long)s);
    }
    if (EM == EM_GAUSS && a.partials) {
        double* out = a.partials + ((long long)(FIXPASS ? gridDim.x : 0) + blockIdx.x) * 2 * N;
        for (int k = tid; k < 2 * N; k += blockDim.x) {
            double s = 0.0;
            for (int t = 0; t < LANE_THREADS; ++t) s += mom[k * LANE_THREADS + t];
            out[k] = s;
        }
    }
}

template <int N>
void fill_params(LaneParams<N>& P, const double* A, const double* pi, const double* mu, const double* sigma)
{
    for (int k = 0; k < N * N; ++k) P.A[k] = A ? A[k] : 0.0;
    for (int j = 0; j < N; ++j) {
        P.pi[j] = pi ? pi[j] : 0.0;
        P.mu[j] = mu ? mu[j] : 0.0;
        const double s = sigma ? sigma[j] : 1.0;
        P.isg[j] = 1.0 / (s * sqrt(2.0));                                  // d = (o - mu) * isg, x = -d*d
        P.nrm[j] = log(1.0 / (sqrt(2.0 * 3.14159265358979323846) * s));    // log of C of _gaussian.c:18
        P.nrml[j] = 1.0 / (sqrt(2.0 * 3.14159265358979323846) * s);
    }
}

template <int N>
constexpr int group_of()
{
    return N <= 5 ? 1 : (N <= 8 ? 2 : (N <= 12 ? LANE_G_MID : 8));
}

template <int N>
int launch_lane_n(const LaneArgs& a, const LaneHostParams& hp, int em, int what, cudaStream_t st)
{
    LaneParams<N> P;
    fill_params<N>(P, hp.A, hp.pi, hp.mu, hp.sigma);
    const int blocks = (a.ch.n + LANE_THREADS - 1) / LANE_THREADS;
    if (blocks <= 0 && what != LANE_QUERY_BLOCKS) return BHMM_OK;
    constexpr int G = group_of<N>();
    if (what == LANE_QUERY_BLOCKS) {
        // (returned through the int result: resident blocks per SM, limited by the backward + statistics kernel)
        int nf = 0, nb = 0;
        if (em == EM_GAUSS) {
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nf, k_forward_lane<N, EM_GAUSS, false>, LANE_THREADS, 0);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_backward_stats_lane<N, EM_GAUSS, G>, LANE_THREADS, 0);
        } else {
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nf, k_forward_lane<N, EM_DISC, false>, LANE_THREADS, 0);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_backward_stats_lane<N, EM_DISC, G>, LANE_THREADS, 0);
        }
        return -max(1, min(nf, nb));     // negative: not an error code
    }
    if (what == LANE_FORWARD) {
        if (em == EM_GAUSS) k_forward_lane<N, EM_GAUSS, false><<<blocks, LANE_THREADS, 0, st>>>(P, a);
        else k_forward_lane<N, EM_DISC, false><<<blocks, LANE_THREADS, 0, st>>>(P, a);
    } else if (what == LANE_FORWARD_ROWMAJOR) {
        if (em == EM_GAUSS) k_forward_lane<N, EM_GAUSS, true><<<blocks, LANE_THREADS, 0, st>>>(P, a);
        else k_forward_lane<N, EM_DISC, true><<<blocks, LANE_THREADS, 0, st>>>(P, a);
    } else if (what == LANE_BACKWARD_STATS) {
        if (em == EM_GAUSS) k_backward_stats_lane<N, EM_GAUSS, G><<<blocks, LANE_THREADS, 0, st>>>(P, a);
        else k_backward_stats_lane<N, EM_DISC, G><<<blocks, LANE_THREADS, 0, st>>>(P, a);
    } else {
        const size_t smem = sizeof(double) * ((size_t)N * N + 2 * N * LANE_THREADS) + sizeof(int) * (size_t)(N * N + 2 * N) * LANE_THREADS;
        const bool exact = a.u_row != nullptr;
        const bool fix = (what == LANE_SAMPLE_FIX);
#define LAUNCH_SAMPLE(EMK, EX, FX)                                                                              \
    do {                                                                                                      \
        if (smem > 48 * 1024 &&                                                                               \
            cudaFuncSetAttribute(k_sample_lane<N, EMK, EX, FX>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                 (int)smem) != cudaSuccess)                                                   \
            return BHMM_ERR_CUDA;                                                                             \
        k_sample_lane<N, EMK, EX, FX><<<blocks, LANE_THREADS, smem, st>>>(P, a);                              \
    } while (0)
        if (em == EM_GAUSS) {
            if (exact) { if (fix) LAUNCH_SAMPLE(EM_GAUSS, true, true); else LAUNCH_SAMPLE(EM_GAUSS, true, false); }
            else { if (fix) LAUNCH_SAMPLE(EM_GAUSS, false, true); else LAUNCH_SAMPLE(EM_GAUSS, false, false); }
        } else {
            if (exact) { if (fix) LAUNCH_SAMPLE(EM_DISC, true, true); else LAUNCH_SAMPLE(EM_DISC, true, false); }
            else { if (fix) LAUNCH_SAMPLE(EM_DISC, false, true); else LAUNCH_SAMPLE(EM_DISC, false, false); }
        }
#undef LAUNCH_SAMPLE
    }
    return BHMM_OK;
}

}  // namespace

// one translation unit per group of N (compiled in parallel): lane_inst_*.cu
#define LANE_INSTANTIATE(NN) \
    int launch_lane_##NN(const LaneArgs& a, const LaneHostParams& hp, int em, int what, cudaStream_t st) \
    { return launch_lane_n<NN>(a, hp, em, what, st); }
