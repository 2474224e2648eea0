// bhmm_b200/csrc/panel_kernels.cu -- N = 32 chain kernels on the FP64 tensor pipe ("panel" family, DESIGN.md section 5.5).
//
// STATUS: the default for 17 <= N <= 104 since round 2 (first B200 runs: parity against the oracle for N = 21, 32, 37, 64, 100,
// compute-sanitizer memcheck + racecheck clean); BHMM_B200_PANEL=0 (read once per process) falls back to the team kernels,
// =2 runs N = 32 on the 4-warp wide kernels.  tests/test_panel_cuda.py is the parity test; the fragment/index algebra below
// is also checked on the CPU by tests/test_panel_layout_cpu.py and tests/emu.
//
// One WARP walks 8 chains at once.  The 8 x 32 panel of the chains' vectors times the 32 x 32 transition matrix is
// 32 mma.sync.m8n8k4.f64 (DMMA) per frame, with the matrix resident in registers as B fragments.  Lane (g, q),
// g = lane / 4, q = lane % 4, belongs to chain g of the warp and owns the 8 states
//     state(k) = 8 (k / 2) + 2 q + (k % 2),   k = 0..7,
// which is exactly what the accumulator fragments of the four n-tiles hand it (row g, columns 8 nt + 2 q + {0, 1}).
// The k-steps of the product are ordered so that k-step ks contracts the states {state(ks) : q = 0..3}: the A operand
// of k-step ks is then the lane's own element k = ks of the previous frame's result -- the recursion needs no shuffle
// and no shared memory (prototype and measurements: tools/micro/dmma_panel.cu).  A "team" in the sense of
// team_kernels.cu is here a quad of lanes; sums over the states of a chain are two xor-shuffles.
//
// Unlike the team kernels the panel kernels normalise every frame like the reference does (_hidden.c:40-64, :92-108),
// so no frame is ever lifted; divisions by a chain's sum are one reciprocal and 8 multiplications (one rounding more
// than the reference's true divisions: 1e-16 relative, the parity bar is 1e-10).
//
// Replaces (reference file:line), fused exactly like team_kernels.cu:
//   k_forward_panel32         _forward  bhmm/hidden/impl_c/_hidden.c:16-66   (+ emission: _gaussian.c:45-70 /
//                             discrete.py:146-153 / outputmodel.py:119-131)
//   k_backward_stats_panel32  _backward _hidden.c:69-110 + state_probabilities hidden/api.py:133-188 + state_counts
//                             :191-211 + _compute_transition_counts _hidden.c:148-183 + the data passes of
//                             GaussianOutputModel.estimate gaussian.py:214-272 / _update_pout _discrete.c:1-32
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int PN = 32;            // hidden states
constexpr int PW = 4;             // warps per block
constexpr int PCH = 8;            // chains per warp
constexpr int PSTRIDE = 36;       // doubles per chain row of the transposition buffers: (4 q + g) mod 16 distinct per
                                  // half warp, so the operand loads of the xi product are bank-conflict free
constexpr unsigned FULL = 0xffffffffu;

// dynamic shared memory of a kernel; the CPU emulation (tests/emu) hands out its own buffer
#ifdef PANEL_HOST_EMU
#define PANEL_DYN_SMEM(name) double* name = reinterpret_cast<double*>(emu::dyn_smem())
#else
#define PANEL_DYN_SMEM(name) extern __shared__ double name[]
#endif

// PANEL_HOST_EMU: the kernels' source compiled for the CPU by tests/emu (every CUDA thread a fiber, collectives emulated)
__device__ __forceinline__ void dmma(double& d0, double& d1, double a, double b)
{
#ifdef PANEL_HOST_EMU
    emu_dmma(d0, d1, a, b);
#else
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
#endif
}

__device__ __forceinline__ void prefetch_l1(const void* p)
{
#ifdef PANEL_HOST_EMU
    (void)*reinterpret_cast<const volatile char*>(p);       // the emulation reads the byte: a stray address faults
#else
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
#endif
}

// sum over the four lanes of a quad; every lane ends with the bitwise identical total
__device__ __forceinline__ double quad_sum(double v)
{
    v += __shfl_xor_sync(FULL, v, 1);
    v += __shfl_xor_sync(FULL, v, 2);
    return v;
}

__device__ __forceinline__ int state_of(int k, int q) { return 8 * (k >> 1) + 2 * q + (k & 1); }

// 8 doubles of a 32-state row, the lane's states: four 16-byte accesses
__device__ __forceinline__ void load8(const double* __restrict__ row, int q, double (&v)[8])
{
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
        const double2 x = *reinterpret_cast<const double2*>(row + 8 * nt + 2 * q);
        v[2 * nt] = x.x;
        v[2 * nt + 1] = x.y;
    }
}
__device__ __forceinline__ void store8(double* __restrict__ row, int q, const double (&v)[8])
{
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) *reinterpret_cast<double2*>(row + 8 * nt + 2 * q) = make_double2(v[2 * nt], v[2 * nt + 1]);
}

// ---- exp() of 8 arguments, evaluated stage by stage so that the 8 dependent chains interleave (same scheme and
// constants as lane_kernels.cuh:emission_gauss, TB == 0 path): exp(x) = 2^n exp(r), n = rint(x / ln 2), |r| <= ln2 / 2,
// degree-11 polynomial (< 1 ulp); arguments below -708 or not finite take the library exp() in a rare tail.
__constant__ double PEXPK[13] = {
    0x1.af632a0f7e2cep-26, 0x1.28b4101c77212p-22, 0x1.71ddf56d8deb5p-19, 0x1.a01991a10d9aep-16,
    0x1.a01a01b1461c5p-13, 0x1.6c16c1880029fp-10, 0x1.111111110f21ep-7,  0x1.555555554f0bap-5,
    0x1.555555555555ap-3,  0x1.0000000000011p-1,
    1.4426950408889634074, 6.93147180369123816490e-01, 1.90821492927058770002e-10};

__device__ __noinline__ double panel_slow_exp(double x) { return exp(x); }

__device__ __forceinline__ void exp8(const double (&x)[8], double (&p)[8])
{
#ifdef PANEL_LIBM_EXP
#pragma unroll
    for (int k = 0; k < 8; ++k) p[k] = exp(x[k]);
#else
    const double MAGIC = 6755399441055744.0;                 // 1.5 * 2^52
    double t[8], r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) t[k] = fma(x[k], PEXPK[10], MAGIC);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const double n = t[k] - MAGIC;
        r[k] = fma(n, -PEXPK[11], x[k]);
        r[k] = fma(n, -PEXPK[12], r[k]);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) p[k] = fma(PEXPK[0], r[k], PEXPK[1]);
#pragma unroll
    for (int c = 2; c < 10; ++c) {
#pragma unroll
        for (int k = 0; k < 8; ++k) p[k] = fma(p[k], r[k], PEXPK[c]);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) p[k] = fma(p[k], r[k], 1.0);
#pragma unroll
    for (int k = 0; k < 8; ++k) p[k] = fma(p[k], r[k], 1.0);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int ni = __double2loint(t[k]);
        p[k] = __longlong_as_double(__double_as_longlong(p[k]) + ((long long)ni << 52));
    }
    unsigned umax = (unsigned)__double2hiint(x[0]);
    int smax = __double2hiint(x[0]);
#pragma unroll
    for (int k = 1; k < 8; ++k) {
        umax = max(umax, (unsigned)__double2hiint(x[k]));
        smax = max(smax, __double2hiint(x[k]));
    }
    if (umax > 0xC0862000u || smax > 0x40862000) {           // some x < -708, > 708 or not finite
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const unsigned hx = (unsigned)__double2hiint(x[k]);
            if (hx >= 0xC0875000u && hx <= 0xFFF00000u) p[k] = 0.0;              // x <= -746 (or -inf): exactly zero
            else if ((hx & 0x7fffffffu) > 0x40862000u) p[k] = panel_slow_exp(x[k]);
        }
    }
#endif
}

// Raw emission input of one frame for one lane: the observation (Gaussian), or the lane's 8 table entries.
template <int EM>
struct Raw {
    double v[EM == EM_GAUSS ? 1 : 8];
    int sym;
};

template <int EM>
__device__ __forceinline__ void raw_load(const Emission& em, long long row, int q, Raw<EM>& r)
{
    r.sym = 0;
    if (EM == EM_GAUSS) {
        r.v[0] = em.obs[row];
    } else if (EM == EM_POBS) {
        double t[8];
        load8(em.pobs + row * PN, q, t);
#pragma unroll
        for (int k = 0; k < 8; ++k) r.v[EM == EM_GAUSS ? 0 : k] = t[k];
    } else {
        r.sym = em.sym[row];
        double t[8];
        load8(em.Bt + (long long)r.sym * PN, q, t);
#pragma unroll
        for (int k = 0; k < 8; ++k) r.v[EM == EM_GAUSS ? 0 : k] = t[k];
    }
}

template <int EM>
__device__ __forceinline__ void raw_prefetch(const Emission& em, long long row, int q)
{
    const void* p;
    if (EM == EM_POBS) p = em.pobs + row * PN + 8 * q;        // the quad touches the row's two 128-byte lines
    else if (EM == EM_GAUSS) p = em.obs + row;
    else p = em.sym + row;
    prefetch_l1(p);
}

// p[k] = density of the lane's state k at this frame.  Gaussian: nrm exp(-((o - mu) isg)^2) with isg = 1 / (sqrt 2 sigma),
// nrm = 1 / (sqrt(2 pi) sigma) (_gaussian.c:18-20 up to the rounding of the reciprocal), constants from `kc` =
// [mu (32) | isg (32) | log nrm (32)] in shared memory.
template <int EM>
__device__ __forceinline__ void emission8(const Raw<EM>& r, const double* __restrict__ kc, int q, double (&p)[8])
{
    if (EM == EM_GAUSS) {
        double mu[8], isg[8], lnrm[8], x[8];
        load8(kc, q, mu);
        load8(kc + PN, q, isg);
        load8(kc + 2 * PN, q, lnrm);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const double d = (r.v[0] - mu[k]) * isg[k];
            x[k] = fma(-d, d, lnrm[k]);
        }
        exp8(x, p);
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) p[k] = r.v[EM == EM_GAUSS ? 0 : k];
    }
}

// outputmodel.py:126-130: a frame whose densities are all zero becomes all one
template <int EM>
__device__ __forceinline__ void outlier_rule(const Emission& em, unsigned qmask, double (&p)[8])
{
    if (EM == EM_POBS || !em.ignore_outliers) return;
    bool nz = false;
#pragma unroll
    for (int k = 0; k < 8; ++k) nz = nz || (p[k] != 0.0);
    const unsigned b = __ballot_sync(FULL, nz);
    if ((b & qmask) == 0u) {
#pragma unroll
        for (int k = 0; k < 8; ++k) p[k] = 1.0;
    }
}

__device__ __forceinline__ void fill_gauss_constants(const Emission& em, double* kc)
{
    for (int j = threadIdx.x; j < PN; j += blockDim.x) {
        const double sg = em.sigma[j];
        kc[j] = em.mu[j];
        kc[PN + j] = 1.0 / (sqrt(2.0) * sg);
        kc[2 * PN + j] = log(1.0 / (sqrt(2.0 * 3.14159265358979323846) * sg));
    }
}

// Running sum of log c_t as a product that is folded into the sum only when it leaves [2^-400, 2^400]: one
// multiplication per frame instead of one log().
struct LogAcc {
    double ll = 0.0, prod = 1.0;
    __device__ __forceinline__ void add(double c)
    {
        prod *= c;
        if (!(prod >= 0x1p-400 && prod <= 0x1p+400)) { ll += log(prod); prod = 1.0; }
    }
    __device__ __forceinline__ double value() const { return ll + log(prod); }
};

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <int EM>
__global__ void __launch_bounds__(PW * 32) k_forward_panel32(const FwdArgs a)
{
    __shared__ __align__(16) double kc[3 * PN];
    const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
    const int gw = blockIdx.x * PW + (threadIdx.x >> 5), nw = gridDim.x * PW;
    const unsigned qmask = 0xFu << (4 * g);
    if (EM == EM_GAUSS) fill_gauss_constants(a.em, kc);
    // B fragments of alpha' = alpha A: k-step ks contracts state_of(ks, q), n-tile nt produces column 8 nt + g
    double Bf[8][4];
#pragma unroll
    for (int ks = 0; ks < 8; ++ks)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) Bf[ks][nt] = a.A[state_of(ks, q) * PN + 8 * nt + g];
    __syncthreads();

    for (int base = gw * PCH; base < a.ch.n; base += nw * PCH) {
        const int idx = base + g;
        const bool have = idx < a.ch.n;
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
        const int maxpre = __reduce_max_sync(FULL, npre);
        const int total = maxpre + __reduce_max_sync(FULL, len);
        const int tend = t0 + len;

        double av[8];                                      // normalised alpha of the previous frame, the lane's states
#pragma unroll
        for (int k = 0; k < 8; ++k) av[k] = 0.0;
        if (have && mode == 2) load8(chain_start_vec(a.ch, a.hand_end, c, c - 1, PN), q, av);
        LogAcc acc;

        auto fetch = [&](int s, Raw<EM>& r) {
            int t = t0 - maxpre + s;
            t = min(max(t, tstart + (mode == 2 ? 1 : 0)), tend - 1);
            if (have) raw_load<EM>(a.em, trow + t, q, r);
            else {
                r.sym = 0;
#pragma unroll
                for (int k = 0; k < (EM == EM_GAUSS ? 1 : 8); ++k) r.v[k] = 0.0;
            }
        };
        Raw<EM> raw_next;
        fetch(0, raw_next);

        for (int s = 0; s < total; ++s) {
            const int t = t0 - maxpre + s;
            const bool on = have && t >= tstart && t < tend;
            const bool init = on && t == tstart;
            const Raw<EM> raw = raw_next;
            fetch(s + 1, raw_next);
            if (have && max(t, tstart) + 48 < tend) raw_prefetch<EM>(a.em, trow + max(t, tstart) + 48, q);

            double p[8];
            emission8<EM>(raw, kc, q, p);
            outlier_rule<EM>(a.em, qmask, p);

            double d[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) d[k] = 0.0;
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) dmma(d[2 * nt], d[2 * nt + 1], av[ks], Bf[ks][nt]);

            double v[8];
            if (init) {
                if (mode == 0) {
                    double pi8[8];
                    load8(a.pi, q, pi8);
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[k] = pi8[k] * p[k];
                } else if (mode == 1) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[k] = p[k];
                } else {
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[k] = av[k];
                }
            } else {
#pragma unroll
                for (int k = 0; k < 8; ++k) v[k] = on ? d[k] * p[k] : 0.0;
            }
            const double part = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
            const double csum = quad_sum(part);
            if (on) {
                const double rc = (csum != 0.0) ? 1.0 / csum : 1.0;      // _hidden.c:31-34, :58-61: divide iff c != 0
#pragma unroll
                for (int k = 0; k < 8; ++k) av[k] = v[k] * rc;
                if (t >= t0) {
                    if (a.alpha) store8(a.alpha + (trow + t) * PN, q, av);
                    acc.add(csum);
                    if (t == tend - 1) store8(a.hand_end + (long long)c * PN, q, av);
                } else if (t == t0 - 1) {
                    store8(a.hand_used + (long long)c * PN, q, av);
                }
            }
        }
        if (have && q == 0) a.chain_ll[c] = acc.value();
    }
}

// ------------------------------------------------------------------------------------------------
// backward + sufficient statistics (fused E-step)
// ------------------------------------------------------------------------------------------------
// Frames f = fstart .. t0+1 downwards; at frame f the lane holds the NORMALISED beta_f of its chain (bn, sum 1).
//   w_j = p_{f,j} bn_j;   d_i = sum_j A_ij w_j  (32 DMMA, B fragments of A^T);   beta_{f-1} = d / sum d
//   gamma_{f-1,i} = alpha_{f-1,i} d_i / S,  S = sum_i alpha_{f-1,i} d_i
//   xi_{f-1}[i][j] = alpha_{f-1,i} A_ij w_j / S   (_hidden.c:168-180: S is the sum of the unnormalised xi)
// The A-independent part X[i][j] += sum over the warp's 8 chains of u_i w_j, u = alpha_{f-1} / S, is a second 32 x 32 x 8
// product: 4 x 4 output tiles, two k-steps over the chains, operands transposed through shared memory (each lane needs
// element [chain 4 kk + q][state 8 t + g] of U and of W).  launch_finalize_stats multiplies by A.
template <int EM>
__global__ void __launch_bounds__(PW * 32) k_backward_stats_panel32(const BwdArgs a)
{
    __shared__ __align__(16) double kc[3 * PN];
    __shared__ __align__(16) double tb[PW][2][PCH * PSTRIDE];      // per warp: U, W
    const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3, wib = threadIdx.x >> 5;
    const int gw = blockIdx.x * PW + wib, nw = gridDim.x * PW;
    const unsigned qmask = 0xFu << (4 * g);
    double* Us = tb[wib][0];
    double* Ws = tb[wib][1];
    if (EM == EM_GAUSS) fill_gauss_constants(a.em, kc);
    // B fragments of d = A w: contraction index j = state_of(ks, q), output column i = 8 nt + g
    double Bt[8][4];
#pragma unroll
    for (int ks = 0; ks < 8; ++ks)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) Bt[ks][nt] = a.A[(8 * nt + g) * PN + state_of(ks, q)];
    double X[4][4][2];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) { X[mt][nt][0] = 0.0; X[mt][nt][1] = 0.0; }
    double st_g[8], st_gd[8], st_gdd[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { st_g[k] = 0.0; st_gd[k] = 0.0; st_gdd[k] = 0.0; }
    // this warp's row of partial statistics: [X (N*N) | gamma0 (N) | sum gamma (N) | sum gamma d (N) | sum gamma d^2 (N)]
    const int nstat = PN * PN + 4 * PN;
    double* out = a.partials + (long long)gw * nstat;
    out[PN * PN + lane] = 0.0;                             // gamma0 is accumulated with atomics by this warp's lanes
    __syncthreads();

    for (int base = gw * PCH; base < a.ch.n; base += nw * PCH) {
        const int idx = base + g;
        const bool have = idx < a.ch.n;
        int c = -1, len = 0, t0 = 0, T = 0, e = 0, fstart = 0, mode = 0;   // mode 0: uniform (exact or warm-up), 2: exact vector
        bool virt = false;                                                  // the chain ends its trajectory
        long long trow = 0;
        if (have) {
            c = a.ch.list ? a.ch.list[idx] : idx;
            len = a.ch.len[c];
            t0 = a.ch.t0[c];
            T = a.ch.T[c];
            trow = a.ch.row0[c] - t0;
            e = t0 + len;
            if (e >= T) { virt = true; fstart = T; }
            else if (chain_exact_start(a.ch, c)) { fstart = e; mode = 2; }
            else { fstart = min(T - 1, e + (a.ch.warmv ? a.ch.warmv[c] : a.ch.warm) - 1); }
        }
        const int flast = t0 + 1;                           // step f emits frame f-1
        const int npre = have ? (fstart - (e - 1)) : 0;
        const int maxpre = __reduce_max_sync(FULL, npre);
        const int total = maxpre + __reduce_max_sync(FULL, have ? (e - flast) : 0);

        double bn[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) bn[k] = 1.0 / PN;      // beta_{T-1} = 1/N (_hidden.c:76-77), also the warm-up start
        if (have && mode == 2) load8(chain_start_vec(a.ch, a.hand_end, c, c + 1, PN), q, bn);

        auto frame_of = [&](int s) -> int { return (e - 1) + maxpre - s; };
        auto fetch = [&](int s, Raw<EM>& r) {
            const int f = min(max(frame_of(s), t0), T - 1);
            if (have) raw_load<EM>(a.em, trow + f, q, r);
            else {
                r.sym = 0;
#pragma unroll
                for (int k = 0; k < (EM == EM_GAUSS ? 1 : 8); ++k) r.v[k] = 0.0;
            }
        };
        auto fetch_alpha = [&](int s, double (&al)[8]) {
            const int f = min(max(frame_of(s) - 1, t0), e - 1);
            if (have) load8(a.alpha + (trow + f) * PN, q, al);
            else {
#pragma unroll
                for (int k = 0; k < 8; ++k) al[k] = 0.0;
            }
        };
        Raw<EM> raw_next;
        double al_next[8];
        fetch(0, raw_next);
        fetch_alpha(0, al_next);

        for (int s = 0; s < total; ++s) {
            const int f = frame_of(s);
            const bool on = have && f <= fstart && f >= flast;
            const bool isvirt = on && virt && f == T;       // virtual frame T: beta_{T-1} proportional to one
            const Raw<EM> raw = raw_next;
            double al[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) al[k] = al_next[k];
            fetch(s + 1, raw_next);                         // frame f-1: also the observation / symbol of the emitted frame
            fetch_alpha(s + 1, al_next);
            if (have && f - 48 > t0) {
                raw_prefetch<EM>(a.em, trow + min(f, T - 1) - 48, q);
                if (f - 48 < e) prefetch_l1(a.alpha + (trow + f - 48) * PN + 8 * q);
            }

            double p[8];
            emission8<EM>(raw, kc, q, p);
            outlier_rule<EM>(a.em, qmask, p);

            double w[8], d[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) { w[k] = (on && !isvirt) ? p[k] * bn[k] : 0.0; d[k] = 0.0; }
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) dmma(d[2 * nt], d[2 * nt + 1], w[ks], Bt[ks][nt]);
            if (isvirt) {
#pragma unroll
                for (int k = 0; k < 8; ++k) d[k] = 1.0;
            }
            if (on && !isvirt && f == e) store8(a.hand_used + (long long)c * PN, q, bn);

            const bool emit = on && (f - 1) < e;            // f-1 >= t0 holds because f >= flast
            const bool xi = emit && !isvirt;
            double gq[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) gq[k] = emit ? al[k] * d[k] : 0.0;
            const double S = quad_sum(((gq[0] + gq[1]) + (gq[2] + gq[3])) + ((gq[4] + gq[5]) + (gq[6] + gq[7])));
            const double sbn = quad_sum(((d[0] + d[1]) + (d[2] + d[3])) + ((d[4] + d[5]) + (d[6] + d[7])));
            const double rS = 1.0 / S;

            // ---- publish u = alpha_{f-1} / S and w for the xi product (zeros from chains that do not emit)
            const bool any_xi = __any_sync(FULL, xi);
            if (any_xi) {
                double u[8], wz[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) { u[k] = xi ? al[k] * rS : 0.0; wz[k] = xi ? w[k] : 0.0; }
                store8(Us + g * PSTRIDE, q, u);
                store8(Ws + g * PSTRIDE, q, wz);
            }
            __syncwarp();

            if (emit) {
                const long long row = trow + (f - 1);
                double gam[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) { gam[k] = gq[k] * rS; st_g[k] += gam[k]; }
                if (f - 1 == 0) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) atomicAdd(out + PN * PN + state_of(k, q), gam[k]);
                }
                if (EM == EM_GAUSS) {
                    double mu[8];
                    load8(kc, q, mu);
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const double dd = raw_next.v[0] - mu[k];
                        st_gd[k] = fma(gam[k], dd, st_gd[k]);
                        st_gdd[k] = fma(gam[k], dd * dd, st_gdd[k]);
                    }
                }
                if (EM == EM_DISC && a.Bnum) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) atomicAdd(a.Bnum + (long long)state_of(k, q) * a.em.M + raw_next.sym, gam[k]);
                }
                if (a.gamma) store8(a.gamma + row * PN, q, gam);
                if (f - 1 == t0 && t0 > 0) {
                    const double r2 = (sbn != 0.0) ? 1.0 / sbn : 1.0;
                    double hb[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) hb[k] = d[k] * r2;
                    store8(a.hand_end + (long long)c * PN, q, hb);
                }
            }
            if (on) {
                const double r2 = (sbn != 0.0) ? 1.0 / sbn : 1.0;          // _hidden.c:104-107: divide iff the sum != 0
#pragma unroll
                for (int k = 0; k < 8; ++k) bn[k] = d[k] * r2;
            }

            // ---- X += U^T W over the warp's chains
            if (any_xi) {
                double ua[2][4], wb[2][4];
#pragma unroll
                for (int kk = 0; kk < 2; ++kk)
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        ua[kk][t] = Us[(4 * kk + q) * PSTRIDE + 8 * t + g];
                        wb[kk][t] = Ws[(4 * kk + q) * PSTRIDE + 8 * t + g];
                    }
#pragma unroll
                for (int kk = 0; kk < 2; ++kk)
#pragma unroll
                    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
                        for (int nt = 0; nt < 4; ++nt) dmma(X[mt][nt][0], X[mt][nt][1], ua[kk][mt], wb[kk][nt]);
            }
            __syncwarp();                                   // the buffers are rewritten by the next step
        }
    }

    // ---- this warp's partial statistics
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
            *reinterpret_cast<double2*>(out + (8 * mt + g) * PN + 8 * nt + 2 * q) = make_double2(X[mt][nt][0], X[mt][nt][1]);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        // lanes with equal q own the same states: sum over g = lane bits 2..4
#pragma unroll
        for (int off = 4; off < 32; off <<= 1) {
            st_g[k] += __shfl_xor_sync(FULL, st_g[k], off);
            st_gd[k] += __shfl_xor_sync(FULL, st_gd[k], off);
            st_gdd[k] += __shfl_xor_sync(FULL, st_gdd[k], off);
        }
    }
    if (g == 0) {
        store8(out + PN * PN + PN, q, st_g);
        store8(out + PN * PN + 2 * PN, q, st_gd);
        store8(out + PN * PN + 3 * PN, q, st_gdd);
    }
}

// ================================================================================================
// "Wide" panel kernels: 32 < N <= 104 (C4: N = 100).  A block of NT warps walks 8 chains; NP = 8 NT padded states.
// Warp w owns state tile w: lane (g, q) holds, for chain g, the states 8 w + 2 q and 8 w + 2 q + 1, and the warp keeps
// the matching 8-column slice of the transition matrix as KS = 2 NT B fragments in registers.  The A operands (the
// previous frame's vector of chain g, all NP states) come from shared memory, where the warps exchange their slices
// once per frame: ONE block barrier per forward frame, two per backward frame.  The vector is normalised when it is
// loaded (a = x / c, c the chain's sum read from the same exchange), i.e. the recursion runs on normalised vectors like
// the reference's (_hidden.c:40-64) and nothing is deferred or lifted.  The outlier rule needs "are all densities of this
// frame zero", a fact only known after the exchange: every frame publishes its vector twice -- with the densities and
// with all densities set to one -- plus the per-tile "any density non-zero" flag, and the consumer picks the source.
// ================================================================================================
template <int NT>
struct WideGeom {
    static constexpr int NP = 8 * NT;
    static constexpr int KS = 2 * NT;
    static constexpr int NPS = NP + ((4 - NP % 16 + 16) % 16);   // row stride = 4 mod 16 doubles: conflict-free operand loads
    // one block per SM: 64 K registers / (32 threads x warps), where the hardware allocates registers to a block in units of
    // FOUR warps -- 13 warps cost 16 (first B200 run of the family: __maxnreg__(152) with 416 threads failed to launch,
    // "too many resources requested"; ptxas itself stops at 128 when it is only given __launch_bounds__(416))
    static constexpr int WALLOC = (NT + 3) / 4 * 4;
    static constexpr int MAXREG = ((65536 / (32 * WALLOC)) / 8 * 8) > 255 ? 255 : ((65536 / (32 * WALLOC)) / 8 * 8);
};
#ifdef PANEL_HOST_EMU
#define WIDE_KERNEL_ATTR(NT)
#else
#define WIDE_KERNEL_ATTR(NT) __maxnreg__(WideGeom<NT>::MAXREG)
#endif

// Emission pipeline of the wide kernels (2 states per lane and frame).  Gaussian: the observation is fetched one frame
// ahead and the two densities are evaluated in the frame.  Table / discrete: the two densities themselves are fetched one
// frame ahead, and for the discrete model the symbol that addresses them one frame before that, so neither dependent load
// sits on a frame's critical path.
__device__ __forceinline__ void wide_gauss2(double o, const double (&mu)[2], const double (&isg)[2], const double (&lnrm)[2],
                                            bool ok0, bool ok1, double (&p)[2])
{
    const double d0 = (o - mu[0]) * isg[0], d1 = (o - mu[1]) * isg[1];
    p[0] = ok0 ? exp(fma(-d0, d0, lnrm[0])) : 0.0;
    p[1] = ok1 ? exp(fma(-d1, d1, lnrm[1])) : 0.0;
}

template <int EM>
__device__ __forceinline__ void wide_table2(const Emission& em, long long row, int sym, int N, int s0, bool ok0, bool ok1,
                                            double (&p)[2])
{
    const double* src = (EM == EM_POBS) ? em.pobs + row * N : em.Bt + (long long)sym * N;
    p[0] = ok0 ? src[s0] : 0.0;
    p[1] = ok1 ? src[s0 + 1] : 0.0;
}

template <int EM, int NT>
__global__ void WIDE_KERNEL_ATTR(NT) k_forward_wide(const FwdArgs a)
{
    constexpr int KS = WideGeom<NT>::KS, NPS = WideGeom<NT>::NPS;
    __shared__ __align__(16) double Sx[2][PCH * NPS];     // the frame's vector with the densities ...
    __shared__ __align__(16) double Sd[2][PCH * NPS];     // ... and with all densities set to one (outlier rule)
    __shared__ double red[2][3][NT][PCH];                 // per tile and chain: sum of Sx, sum of Sd, any density != 0
    const int N = a.N;
    const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3, w = threadIdx.x >> 5;
    const unsigned qmask = 0xFu << (4 * g);
    const int s0 = 8 * w + 2 * q;
    const bool ok0 = s0 < N, ok1 = s0 + 1 < N;
    double Bf[KS];
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
        const int k = 4 * ks + q, col = 8 * w + g;
        Bf[ks] = (k < N && col < N) ? a.A[k * N + col] : 0.0;
    }
    double mu[2] = {0.0, 0.0}, isg[2] = {1.0, 1.0}, lnrm[2] = {0.0, 0.0};
    if (EM == EM_GAUSS) {
#pragma unroll
        for (int r = 0; r < 2; ++r)
            if (s0 + r < N) {
                const double sg = a.em.sigma[s0 + r];
                mu[r] = a.em.mu[s0 + r];
                isg[r] = 1.0 / (sqrt(2.0) * sg);
                lnrm[r] = log(1.0 / (sqrt(2.0 * 3.14159265358979323846) * sg));
            }
    }

    for (int base = blockIdx.x * PCH; base < a.ch.n; base += gridDim.x * PCH) {
        const int idx = base + g;
        const bool have = idx < a.ch.n;
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
        const int maxpre = __reduce_max_sync(FULL, npre);
        const int total = maxpre + __reduce_max_sync(FULL, len);
        const int tend = t0 + len;
        for (int k = threadIdx.x; k < 2 * PCH * NPS; k += blockDim.x) { (&Sx[0][0])[k] = 0.0; (&Sd[0][0])[k] = 0.0; }
        for (int k = threadIdx.x; k < 2 * 3 * NT * PCH; k += blockDim.x) (&red[0][0][0][0])[k] = 0.0;
        __syncthreads();

        double vec[2] = {0.0, 0.0};
        if (have && mode == 2) {
            const double* hv = chain_start_vec(a.ch, a.hand_end, c, c - 1, N);
            if (ok0) vec[0] = hv[s0];
            if (ok1) vec[1] = hv[s0 + 1];
        }
        double v[2] = {0.0, 0.0}, dd[2] = {0.0, 0.0};       // the lane's values of the frame in flight: with densities / with ones
        LogAcc acc;
        auto frame_row = [&](int s) -> long long {
            int t = t0 - maxpre + s;
            t = min(max(t, tstart + (mode == 2 ? 1 : 0)), tend - 1);
            return trow + t;
        };
        double o_next = 0.0, pn[2] = {0.0, 0.0};
        int symA = 0;                                       // discrete: symbol of the frame after the one whose densities are in pn
        if (have) {
            if (EM == EM_GAUSS) o_next = a.em.obs[frame_row(0)];
            if (EM == EM_DISC) {
                wide_table2<EM>(a.em, 0, a.em.sym[frame_row(0)], N, s0, ok0, ok1, pn);
                symA = a.em.sym[frame_row(1)];
            }
            if (EM == EM_POBS) wide_table2<EM>(a.em, frame_row(0), 0, N, s0, ok0, ok1, pn);
        }

        for (int s = 0; s <= total; ++s) {
            const int cur = s & 1, prev = cur ^ 1;
            // ---- finish frame s-1: the chain's sums are complete, normalise, store
            double rc = 1.0;
            bool use_d = false;
            if (s > 0) {
                const int tp = t0 - maxpre + s - 1;
                const bool onp = have && tp >= tstart && tp < tend;
                // every quad sums the NT tile partials of its chain: lane q takes tiles q, q+4, ... (the same order in
                // every warp, so all warps derive the bitwise identical chain sum)
                double cs = 0.0, cd = 0.0, nz = 0.0;
#pragma unroll
                for (int w2 = 0; w2 < NT; w2 += 4)
                    if (w2 + q < NT) { cs += red[prev][0][w2 + q][g]; cd += red[prev][1][w2 + q][g]; nz += red[prev][2][w2 + q][g]; }
                cs = quad_sum(cs);
                cd = quad_sum(cd);
                nz = quad_sum(nz);
                if (EM != EM_POBS && a.em.ignore_outliers && onp && nz == 0.0) { use_d = true; cs = cd; }   // outputmodel.py:126-130
                rc = (cs != 0.0) ? 1.0 / cs : 1.0;          // _hidden.c:31-34, :58-61: divide iff c != 0
                if (onp) {
                    const double out0 = (use_d ? dd[0] : v[0]) * rc, out1 = (use_d ? dd[1] : v[1]) * rc;
                    if (tp >= t0) {
                        if (a.alpha) {
                            if (ok0) a.alpha[(trow + tp) * N + s0] = out0;
                            if (ok1) a.alpha[(trow + tp) * N + s0 + 1] = out1;
                        }
                        if (w == 0 && q == 0) acc.add(cs);
                        if (tp == tend - 1) {
                            if (ok0) a.hand_end[(long long)c * N + s0] = out0;
                            if (ok1) a.hand_end[(long long)c * N + s0 + 1] = out1;
                        }
                    } else if (tp == t0 - 1) {
                        if (ok0) a.hand_used[(long long)c * N + s0] = out0;
                        if (ok1) a.hand_used[(long long)c * N + s0 + 1] = out1;
                    }
                }
            }
            if (s == total) break;

            // ---- frame s
            const int t = t0 - maxpre + s;
            const bool on = have && t >= tstart && t < tend;
            const bool init = on && t == tstart;
            double p[2] = {0.0, 0.0};
            if (have) {
                if (EM == EM_GAUSS) {
                    const double o = o_next;
                    o_next = a.em.obs[frame_row(s + 1)];
                    wide_gauss2(o, mu, isg, lnrm, ok0, ok1, p);
                } else {
                    p[0] = pn[0]; p[1] = pn[1];
                    if (EM == EM_DISC) {
                        wide_table2<EM>(a.em, 0, symA, N, s0, ok0, ok1, pn);
                        symA = a.em.sym[frame_row(s + 2)];
                    } else {
                        wide_table2<EM>(a.em, frame_row(s + 1), 0, N, s0, ok0, ok1, pn);
                    }
                }
            }
            const double* src = (use_d ? Sd[prev] : Sx[prev]) + g * NPS;
            double e0 = 0.0, e1 = 0.0, f0 = 0.0, f1 = 0.0;  // two accumulator pairs halve the dependent DMMA chain
#pragma unroll
            for (int ks = 0; ks < KS; ks += 2) {
                dmma(e0, e1, src[4 * ks + q] * rc, Bf[ks]);
                dmma(f0, f1, src[4 * ks + 4 + q] * rc, Bf[ks + 1]);
            }
            bool nzflag = (p[0] != 0.0) || (p[1] != 0.0);
            if (init) {
                if (mode == 0) { dd[0] = ok0 ? a.pi[s0] : 0.0; dd[1] = ok1 ? a.pi[s0 + 1] : 0.0; }
                else if (mode == 1) { dd[0] = ok0 ? 1.0 : 0.0; dd[1] = ok1 ? 1.0 : 0.0; }
                else { dd[0] = vec[0]; dd[1] = vec[1]; }
                if (mode == 2) { v[0] = vec[0]; v[1] = vec[1]; nzflag = true; }
                else { v[0] = dd[0] * p[0]; v[1] = dd[1] * p[1]; }
            } else if (on) {
                dd[0] = e0 + f0; dd[1] = e1 + f1;
                v[0] = dd[0] * p[0]; v[1] = dd[1] * p[1];
            } else {
                dd[0] = dd[1] = v[0] = v[1] = 0.0;
                nzflag = false;
            }
            const double pv = quad_sum(v[0] + v[1]), pd = quad_sum(dd[0] + dd[1]);
            const bool nzq = (__ballot_sync(FULL, nzflag) & qmask) != 0u;
            *reinterpret_cast<double2*>(&Sx[cur][g * NPS + s0]) = make_double2(v[0], v[1]);
            *reinterpret_cast<double2*>(&Sd[cur][g * NPS + s0]) = make_double2(dd[0], dd[1]);
            if (q == 0) { red[cur][0][w][g] = pv; red[cur][1][w][g] = pd; red[cur][2][w][g] = nzq ? 1.0 : 0.0; }
            __syncthreads();
        }
        if (have && w == 0 && q == 0) a.chain_ll[c] = acc.value();
        __syncthreads();                                    // the buffers are cleared for the next chain group
    }
}

// Backward + statistics, wide.  Step for frame f (downwards), chain g, lane's states s0, s0+1:
//   publish w = p_f bn (and bn itself for the outlier rule)                       -- barrier 1
//   xi product of the PREVIOUS step: X[:, tile w] += U^T W over the 8 chains (U, W of that step still in shared memory)
//   d_i = sum_j A_ij w_j for the warp's tile; partial sums of alpha_{f-1} d and of d          -- barrier 2
//   S, sum d complete: u = alpha_{f-1} / S published, gamma and moments, bn = d / sum d
template <int EM, int NT>
__global__ void WIDE_KERNEL_ATTR(NT) k_backward_stats_wide(const BwdArgs a)
{
    constexpr int KS = WideGeom<NT>::KS, NPS = WideGeom<NT>::NPS;
    __shared__ __align__(16) double Sw[2][PCH * NPS];
    __shared__ __align__(16) double Sb[2][PCH * NPS];
    __shared__ __align__(16) double Su[PCH * NPS];
    __shared__ double red[2][NT][PCH];                     // partial S, partial sum of d
    __shared__ double redn[NT][PCH];                       // any density != 0
    const int N = a.N;
    const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3, w = threadIdx.x >> 5;
    const unsigned qmask = 0xFu << (4 * g);
    const int s0 = 8 * w + 2 * q;
    const bool ok0 = s0 < N, ok1 = s0 + 1 < N;
    double Bt[KS];                                          // d = A w: contraction index j = 4 ks + q, output i = 8 w + g
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
        const int j = 4 * ks + q, i = 8 * w + g;
        Bt[ks] = (i < N && j < N) ? a.A[i * N + j] : 0.0;
    }
    double X[NT][2];
#pragma unroll
    for (int mt = 0; mt < NT; ++mt) { X[mt][0] = 0.0; X[mt][1] = 0.0; }
    double mu[2] = {0.0, 0.0}, isg[2] = {1.0, 1.0}, lnrm[2] = {0.0, 0.0};
    if (EM == EM_GAUSS) {
#pragma unroll
        for (int r = 0; r < 2; ++r)
            if (s0 + r < N) {
                const double sg = a.em.sigma[s0 + r];
                mu[r] = a.em.mu[s0 + r];
                isg[r] = 1.0 / (sqrt(2.0) * sg);
                lnrm[r] = log(1.0 / (sqrt(2.0 * 3.14159265358979323846) * sg));
            }
    }
    double st_g[2] = {0.0, 0.0}, st_gd[2] = {0.0, 0.0}, st_gdd[2] = {0.0, 0.0};
    const long long nstat = (long long)N * N + 4 * N;
    double* out = a.partials + (long long)blockIdx.x * nstat;
    for (int j = threadIdx.x; j < N; j += blockDim.x) out[(long long)N * N + j] = 0.0;   // gamma0: atomics below
    __syncthreads();

    auto xi_product = [&](int buf) {
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
            const double wb = Sw[buf][(4 * kk + q) * NPS + 8 * w + g];
#pragma unroll
            for (int mt = 0; mt < NT; ++mt) dmma(X[mt][0], X[mt][1], Su[(4 * kk + q) * NPS + 8 * mt + g], wb);
        }
    };

    for (int base = blockIdx.x * PCH; base < a.ch.n; base += gridDim.x * PCH) {
        const int idx = base + g;
        const bool have = idx < a.ch.n;
        int c = -1, len = 0, t0 = 0, T = 0, e = 0, fstart = 0, mode = 0;
        bool virt = false;
        long long trow = 0;
        if (have) {
            c = a.ch.list ? a.ch.list[idx] : idx;
            len = a.ch.len[c];
            t0 = a.ch.t0[c];
            T = a.ch.T[c];
            trow = a.ch.row0[c] - t0;
            e = t0 + len;
            if (e >= T) { virt = true; fstart = T; }
            else if (chain_exact_start(a.ch, c)) { fstart = e; mode = 2; }
            else { fstart = min(T - 1, e + (a.ch.warmv ? a.ch.warmv[c] : a.ch.warm) - 1); }
        }
        const int flast = t0 + 1;
        const int npre = have ? (fstart - (e - 1)) : 0;
        const int maxpre = __reduce_max_sync(FULL, npre);
        const int total = maxpre + __reduce_max_sync(FULL, have ? (e - flast) : 0);
        for (int k = threadIdx.x; k < 2 * PCH * NPS; k += blockDim.x) { (&Sw[0][0])[k] = 0.0; (&Sb[0][0])[k] = 0.0; }
        for (int k = threadIdx.x; k < PCH * NPS; k += blockDim.x) Su[k] = 0.0;
        __syncthreads();

        double bn[2] = {ok0 ? 1.0 / N : 0.0, ok1 ? 1.0 / N : 0.0};   // beta_{T-1} = 1/N (_hidden.c:76-77); warm-up start
        if (have && mode == 2) {
            const double* hv = chain_start_vec(a.ch, a.hand_end, c, c + 1, N);
            if (ok0) bn[0] = hv[s0];
            if (ok1) bn[1] = hv[s0 + 1];
        }
        auto frame_of = [&](int s) -> int { return (e - 1) + maxpre - s; };
        auto em_row = [&](int s) -> long long { return trow + min(max(frame_of(s), t0), T - 1); };
        auto al_row = [&](int s) -> long long { return trow + min(max(frame_of(s) - 1, t0), e - 1); };
        double o_next = 0.0, al_next[2] = {0.0, 0.0}, pn[2] = {0.0, 0.0};
        int symA = 0;                                       // discrete: symbol of the step after the one whose densities are in pn
        if (have) {
            if (EM == EM_GAUSS) o_next = a.em.obs[em_row(0)];
            if (EM == EM_DISC) {
                wide_table2<EM>(a.em, 0, a.em.sym[em_row(0)], N, s0, ok0, ok1, pn);
                symA = a.em.sym[em_row(1)];
            }
            if (EM == EM_POBS) wide_table2<EM>(a.em, em_row(0), 0, N, s0, ok0, ok1, pn);
            if (ok0) al_next[0] = a.alpha[al_row(0) * N + s0];
            if (ok1) al_next[1] = a.alpha[al_row(0) * N + s0 + 1];
        }
        bool pending_xi = false;                            // the previous step published a non-zero U

        for (int s = 0; s < total; ++s) {
            const int cur = s & 1;
            const int f = frame_of(s);
            const bool on = have && f <= fstart && f >= flast;
            const bool isvirt = on && virt && f == T;
            const double al0 = al_next[0], al1 = al_next[1];
            double p[2] = {0.0, 0.0};
            int sym_emit = 0;                               // symbol of frame f-1, the frame this step emits
            if (have) {
                if (ok0) al_next[0] = a.alpha[al_row(s + 1) * N + s0];
                if (ok1) al_next[1] = a.alpha[al_row(s + 1) * N + s0 + 1];
                if (EM == EM_GAUSS) {
                    const double o = o_next;
                    o_next = a.em.obs[em_row(s + 1)];       // frame f-1: also the emitted frame's observation
                    wide_gauss2(o, mu, isg, lnrm, ok0, ok1, p);
                } else {
                    p[0] = pn[0]; p[1] = pn[1];
                    if (EM == EM_DISC) {
                        sym_emit = symA;
                        wide_table2<EM>(a.em, 0, symA, N, s0, ok0, ok1, pn);
                        symA = a.em.sym[em_row(s + 2)];
                    } else {
                        wide_table2<EM>(a.em, em_row(s + 1), 0, N, s0, ok0, ok1, pn);
                    }
                }
            }
            const bool act = on && !isvirt;
            double wv[2] = {act ? p[0] * bn[0] : 0.0, act ? p[1] * bn[1] : 0.0};
            const double bv[2] = {act ? bn[0] : 0.0, act ? bn[1] : 0.0};
            const bool nzq = (__ballot_sync(FULL, (p[0] != 0.0) || (p[1] != 0.0)) & qmask) != 0u;
            *reinterpret_cast<double2*>(&Sw[cur][g * NPS + s0]) = make_double2(wv[0], wv[1]);
            *reinterpret_cast<double2*>(&Sb[cur][g * NPS + s0]) = make_double2(bv[0], bv[1]);
            if (q == 0) redn[w][g] = nzq ? 1.0 : 0.0;
            __syncthreads();                                // ---- barrier 1

            if (pending_xi) xi_product(cur ^ 1);

            double nz = 0.0;
#pragma unroll
            for (int w2 = 0; w2 < NT; w2 += 4)
                if (w2 + q < NT) nz += redn[w2 + q][g];
            nz = quad_sum(nz);
            const bool use_b = (EM != EM_POBS) && a.em.ignore_outliers && act && nz == 0.0;   // outputmodel.py:126-130
            const double* src = (use_b ? Sb[cur] : Sw[cur]) + g * NPS;
            double e0 = 0.0, e1 = 0.0, f0 = 0.0, f1 = 0.0;
#pragma unroll
            for (int ks = 0; ks < KS; ks += 2) {
                dmma(e0, e1, src[4 * ks + q], Bt[ks]);
                dmma(f0, f1, src[4 * ks + 4 + q], Bt[ks + 1]);
            }
            double d[2] = {e0 + f0, e1 + f1};
            if (isvirt) { d[0] = ok0 ? 1.0 : 0.0; d[1] = ok1 ? 1.0 : 0.0; }
            if (use_b) {                                    // the xi product of the next step reads W from Sw
                wv[0] = bv[0]; wv[1] = bv[1];
                *reinterpret_cast<double2*>(&Sw[cur][g * NPS + s0]) = make_double2(wv[0], wv[1]);
            }
            if (act && f == e) {
                if (ok0) a.hand_used[(long long)c * N + s0] = bn[0];
                if (ok1) a.hand_used[(long long)c * N + s0 + 1] = bn[1];
            }
            const bool emit = on && (f - 1) < e;
            const bool xi = emit && !isvirt;
            const double gq0 = emit ? al0 * d[0] : 0.0, gq1 = emit ? al1 * d[1] : 0.0;
            const double pS = quad_sum(gq0 + gq1), pb = quad_sum(d[0] + d[1]);
            if (q == 0) { red[0][w][g] = pS; red[1][w][g] = pb; }
            __syncthreads();                                // ---- barrier 2

            double S = 0.0, sbn = 0.0;
#pragma unroll
            for (int w2 = 0; w2 < NT; w2 += 4)
                if (w2 + q < NT) { S += red[0][w2 + q][g]; sbn += red[1][w2 + q][g]; }
            S = quad_sum(S);
            sbn = quad_sum(sbn);
            const double rS = 1.0 / S;
            *reinterpret_cast<double2*>(&Su[g * NPS + s0]) = make_double2(xi ? al0 * rS : 0.0, xi ? al1 * rS : 0.0);
            pending_xi = __any_sync(FULL, xi);
            if (emit) {
                const long long orow = trow + (f - 1);
                const double gam[2] = {gq0 * rS, gq1 * rS};
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    if (s0 + r >= N) continue;
                    st_g[r] += gam[r];
                    if (f - 1 == 0) atomicAdd(out + (long long)N * N + s0 + r, gam[r]);
                    if (EM == EM_GAUSS) {
                        const double dv = o_next - mu[r];
                        st_gd[r] = fma(gam[r], dv, st_gd[r]);
                        st_gdd[r] = fma(gam[r], dv * dv, st_gdd[r]);
                    }
                    if (EM == EM_DISC && a.Bnum) atomicAdd(a.Bnum + (long long)(s0 + r) * a.em.M + sym_emit, gam[r]);
                    if (a.gamma) a.gamma[orow * N + s0 + r] = gam[r];
                }
                if (f - 1 == t0 && t0 > 0) {
                    const double r2 = (sbn != 0.0) ? 1.0 / sbn : 1.0;
                    if (ok0) a.hand_end[(long long)c * N + s0] = d[0] * r2;
                    if (ok1) a.hand_end[(long long)c * N + s0 + 1] = d[1] * r2;
                }
            }
            if (on) {
                const double r2 = (sbn != 0.0) ? 1.0 / sbn : 1.0;          // _hidden.c:104-107
                bn[0] = d[0] * r2;
                bn[1] = d[1] * r2;
            }
        }
        __syncthreads();
        if (pending_xi) xi_product((total - 1) & 1);
        __syncthreads();                                    // the buffers are cleared for the next chain group
    }

    // ---- the block's row of partial statistics: [X (N*N) | gamma0 (N) | sum gamma | sum gamma d | sum gamma d^2]
#pragma unroll
    for (int mt = 0; mt < NT; ++mt) {
        const int i = 8 * mt + g;
        if (i < N) {
            if (ok0) out[(long long)i * N + s0] = X[mt][0];
            if (ok1) out[(long long)i * N + s0 + 1] = X[mt][1];
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
#pragma unroll
        for (int off = 4; off < 32; off <<= 1) {
            st_g[r] += __shfl_xor_sync(FULL, st_g[r], off);
            st_gd[r] += __shfl_xor_sync(FULL, st_gd[r], off);
            st_gdd[r] += __shfl_xor_sync(FULL, st_gdd[r], off);
        }
        if (g == 0 && s0 + r < N) {
            out[(long long)N * N + N + s0 + r] = st_g[r];
            out[(long long)N * N + 2 * N + s0 + r] = st_gd[r];
            out[(long long)N * N + 3 * N + s0 + r] = st_gdd[r];
        }
    }
}

// ================================================================================================
// "wide2" kernels: the wide kernels with TWO chain sets (16 chains) per block and one set of barriers for both.
//
// First B200 profile of the wide kernels at N = 100 (profiles/r2_wide13_ncu.md): the FP64 tensor pipe is busy a third of the
// time; a frame is DMMA phase (all 13 warps queue on the pipe) followed by a latency phase (chain sums through shared memory,
// shuffles, a division, the emission) in which the pipe idles, separated by block barriers at which 13 warps on 4 schedulers
// wait for the scheduler that carries 4 of them.  Here every warp walks two independent groups of 8 chains with the SAME B
// fragments: the latency phase and the barriers are paid once per two frames of work.  Also: the previous frame's vector is
// no longer rescaled operand by operand (26 DMUL per lane and frame on the pipe the DMMAs need) -- the product runs on the
// raw vector and the result is scaled once; four accumulator pairs instead of two shorten the dependent DMMA chains; the
// outlier machinery (second copy of the vector, two extra reductions) is compiled out when the rule is off (OUTL = false:
// discrete models by default, caller tables always); the backward kernel reads its B fragments from shared memory when
// they do not fit the register file next to the xi accumulators (BSM, NT = 13: no spills).
// ================================================================================================
constexpr int WS = 2;                                       // chain sets per block (forward; the backward kernel takes it as a template parameter)

template <int NT, bool OUTL>
constexpr size_t wide2_forward_smem()
{
    return sizeof(double) * ((size_t)WS * 2 * PCH * WideGeom<NT>::NPS * (OUTL ? 2 : 1) + (size_t)WS * 2 * (OUTL ? 3 : 1) * NT * PCH);
}

template <int EM, int NT, bool OUTL>
__global__ void WIDE_KERNEL_ATTR(NT) k_forward_wide2(const FwdArgs a)
{
    constexpr int KS = WideGeom<NT>::KS, NPS = WideGeom<NT>::NPS, NR = OUTL ? 3 : 1, ROW = PCH * NPS;
    PANEL_DYN_SMEM(wsm);
    double* const Sx = wsm;                                 // [WS][2][ROW]   the frame's vector with the densities ...
    double* const Sd = Sx + WS * 2 * ROW;                   // [WS][2][ROW]   ... and with all densities set to one (OUTL only)
    double* const red = Sd + (OUTL ? WS * 2 * ROW : 0);     // [WS][2][NR][NT][PCH] per tile and chain: sum of Sx (, sum of Sd, any density != 0)
    const int N = a.N;
    const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3, w = threadIdx.x >> 5;
    const unsigned qmask = 0xFu << (4 * g);
    const int s0 = 8 * w + 2 * q;
    const bool ok0 = s0 < N, ok1 = s0 + 1 < N;
    // state pairs are 16-byte aligned in (rows, N) arrays when N is even and the arrays are
    const bool pair_ok = ((N & 1) == 0) && (((reinterpret_cast<uintptr_t>(a.alpha) | reinterpret_cast<uintptr_t>(a.hand_end) |
                                              reinterpret_cast<uintptr_t>(a.hand_used)) & 15u) == 0);
    double Bf[KS];
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
        const int k = 4 * ks + q, col = 8 * w + g;
        Bf[ks] = (k < N && col < N) ? a.A[k * N + col] : 0.0;
    }
    double mu[2] = {0.0, 0.0}, isg[2] = {1.0, 1.0}, lnrm[2] = {0.0, 0.0};
    if (EM == EM_GAUSS) {
#pragma unroll
        for (int r = 0; r < 2; ++r)
            if (s0 + r < N) {
                const double sg = a.em.sigma[s0 + r];
                mu[r] = a.em.mu[s0 + r];
                isg[r] = 1.0 / (sqrt(2.0) * sg);
                lnrm[r] = log(1.0 / (sqrt(2.0 * 3.14159265358979323846) * sg));
            }
    }
    auto store2 = [&](double* dst, double x0, double x1) {   // dst -> element s0 of a (rows, N) row
        if (pair_ok && ok1) *reinterpret_cast<double2*>(dst) = make_double2(x0, x1);
        else { if (ok0) dst[0] = x0; if (ok1) dst[1] = x1; }
    };

    for (int base = blockIdx.x * (WS * PCH); base < a.ch.n; base += gridDim.x * (WS * PCH)) {
        bool have[WS];
        int c[WS], t0[WS], tstart[WS], mode[WS], tend[WS], maxpre[WS];
        long long trow[WS];
        int total = 0;
#pragma unroll
        for (int z = 0; z < WS; ++z) {
            const int idx = base + z * PCH + g;
            have[z] = idx < a.ch.n;
            c[z] = -1; t0[z] = 0; tstart[z] = 0; mode[z] = 0; trow[z] = 0;   // mode 0: pi, 1: uniform warm-up, 2: exact vector
            int len = 0;
            if (have[z]) {
                c[z] = a.ch.list ? a.ch.list[idx] : idx;
                len = a.ch.len[c[z]];
                t0[z] = a.ch.t0[c[z]];
                trow[z] = a.ch.row0[c[z]] - t0[z];
                if (t0[z] == 0) { tstart[z] = 0; mode[z] = 0; }
                else if (chain_exact_start(a.ch, c[z])) { tstart[z] = t0[z] - 1; mode[z] = 2; }
                else { tstart[z] = max(0, t0[z] - (a.ch.warmv ? a.ch.warmv[c[z]] : a.ch.warm)); mode[z] = (tstart[z] == 0) ? 0 : 1; }
            }
            tend[z] = t0[z] + len;
            maxpre[z] = __reduce_max_sync(FULL, have[z] ? (t0[z] - tstart[z]) : 0);
            total = max(total, maxpre[z] + __reduce_max_sync(FULL, len));
        }
        for (int k = threadIdx.x; k < WS * 2 * ROW; k += blockDim.x) { Sx[k] = 0.0; if (OUTL) Sd[k] = 0.0; }
        for (int k = threadIdx.x; k < WS * 2 * NR * NT * PCH; k += blockDim.x) red[k] = 0.0;
        __syncthreads();

        double vec[WS][2], v[WS][2], dd[WS][2], o_next[WS], pn[WS][2];
        int symA[WS];
        LogAcc acc[WS];
        auto frame_row = [&](int z, int s) -> long long {
            int t = t0[z] - maxpre[z] + s;
            t = min(max(t, tstart[z] + (mode[z] == 2 ? 1 : 0)), tend[z] - 1);
            return trow[z] + t;
        };
#pragma unroll
        for (int z = 0; z < WS; ++z) {
            vec[z][0] = vec[z][1] = v[z][0] = v[z][1] = dd[z][0] = dd[z][1] = 0.0;
            o_next[z] = 0.0; pn[z][0] = pn[z][1] = 0.0; symA[z] = 0;
            if (have[z] && mode[z] == 2) {
                const double* hv = chain_start_vec(a.ch, a.hand_end, c[z], c[z] - 1, N);
                if (ok0) vec[z][0] = hv[s0];
                if (ok1) vec[z][1] = hv[s0 + 1];
            }
            if (have[z]) {
                if (EM == EM_GAUSS) o_next[z] = a.em.obs[frame_row(z, 0)];
                if (EM == EM_DISC) {
                    wide_table2<EM>(a.em, 0, a.em.sym[frame_row(z, 0)], N, s0, ok0, ok1, pn[z]);
                    symA[z] = a.em.sym[frame_row(z, 1)];
                }
                if (EM == EM_POBS) wide_table2<EM>(a.em, frame_row(z, 0), 0, N, s0, ok0, ok1, pn[z]);
            }
        }

        for (int s = 0; s <= total; ++s) {
            const int cur = s & 1, prev = cur ^ 1;
            double rc[WS];
            bool use_d[WS];
            // ---- finish frame s-1 of both sets: the chains' sums are complete, normalise, store
#pragma unroll
            for (int z = 0; z < WS; ++z) {
                rc[z] = 1.0;
                use_d[z] = false;
                if (s > 0) {
                    const int tp = t0[z] - maxpre[z] + s - 1;
                    const bool onp = have[z] && tp >= tstart[z] && tp < tend[z];
                    const double* rp = red + (size_t)(z * 2 + prev) * NR * NT * PCH;
                    double cs = 0.0, cd = 0.0, nz = 0.0;
#pragma unroll
                    for (int w2 = 0; w2 < NT; w2 += 4)
                        if (w2 + q < NT) {
                            cs += rp[(w2 + q) * PCH + g];
                            if (OUTL) { cd += rp[(NT + w2 + q) * PCH + g]; nz += rp[(2 * NT + w2 + q) * PCH + g]; }
                        }
                    cs = quad_sum(cs);
                    if (OUTL) {
                        cd = quad_sum(cd);
                        nz = quad_sum(nz);
                        if (a.em.ignore_outliers && onp && nz == 0.0) { use_d[z] = true; cs = cd; }   // outputmodel.py:126-130
                    }
                    rc[z] = (cs != 0.0) ? 1.0 / cs : 1.0;   // _hidden.c:31-34, :58-61: divide iff c != 0
                    if (onp) {
                        const double out0 = (use_d[z] ? dd[z][0] : v[z][0]) * rc[z], out1 = (use_d[z] ? dd[z][1] : v[z][1]) * rc[z];
                        if (tp >= t0[z]) {
                            if (a.alpha) store2(a.alpha + (trow[z] + tp) * N + s0, out0, out1);
                            if (w == 0 && q == 0) acc[z].add(cs);
                            if (tp == tend[z] - 1) store2(a.hand_end + (long long)c[z] * N + s0, out0, out1);
                        } else if (tp == t0[z] - 1) {
                            store2(a.hand_used + (long long)c[z] * N + s0, out0, out1);
                        }
                    }
                }
            }
            if (s == total) break;

            // ---- frame s of both sets
#pragma unroll
            for (int z = 0; z < WS; ++z) {
                const int t = t0[z] - maxpre[z] + s;
                const bool on = have[z] && t >= tstart[z] && t < tend[z];
                const bool init = on && t == tstart[z];
                double p[2] = {0.0, 0.0};
                if (have[z]) {
                    if (EM == EM_GAUSS) {
                        const double o = o_next[z];
                        o_next[z] = a.em.obs[frame_row(z, s + 1)];
                        wide_gauss2(o, mu, isg, lnrm, ok0, ok1, p);
                    } else {
                        p[0] = pn[z][0]; p[1] = pn[z][1];
                        if (EM == EM_DISC) {
                            wide_table2<EM>(a.em, 0, symA[z], N, s0, ok0, ok1, pn[z]);
                            symA[z] = a.em.sym[frame_row(z, s + 2)];
                        } else {
                            wide_table2<EM>(a.em, frame_row(z, s + 1), 0, N, s0, ok0, ok1, pn[z]);
                        }
                    }
                }
                const double* src = ((OUTL && use_d[z]) ? Sd : Sx) + (size_t)(z * 2 + prev) * ROW + g * NPS;
                double e[4][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};   // four accumulator pairs: short dependent DMMA chains
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) dmma(e[ks & 3][0], e[ks & 3][1], src[4 * ks + q], Bf[ks]);
                const double d0 = ((e[0][0] + e[1][0]) + (e[2][0] + e[3][0])) * rc[z];   // the raw vector's product, scaled once
                const double d1 = ((e[0][1] + e[1][1]) + (e[2][1] + e[3][1])) * rc[z];
                bool nzflag = (p[0] != 0.0) || (p[1] != 0.0);
                if (init) {
                    if (mode[z] == 0) { dd[z][0] = ok0 ? a.pi[s0] : 0.0; dd[z][1] = ok1 ? a.pi[s0 + 1] : 0.0; }
                    else if (mode[z] == 1) { dd[z][0] = ok0 ? 1.0 : 0.0; dd[z][1] = ok1 ? 1.0 : 0.0; }
                    else { dd[z][0] = vec[z][0]; dd[z][1] = vec[z][1]; }
                    if (mode[z] == 2) { v[z][0] = vec[z][0]; v[z][1] = vec[z][1]; nzflag = true; }
                    else { v[z][0] = dd[z][0] * p[0]; v[z][1] = dd[z][1] * p[1]; }
                } else if (on) {
                    dd[z][0] = d0; dd[z][1] = d1;
                    v[z][0] = d0 * p[0]; v[z][1] = d1 * p[1];
                } else {
                    dd[z][0] = dd[z][1] = v[z][0] = v[z][1] = 0.0;
                    nzflag = false;
                }
                const double pv = quad_sum(v[z][0] + v[z][1]);
                *reinterpret_cast<double2*>(Sx + (size_t)(z * 2 + cur) * ROW + g * NPS + s0) = make_double2(v[z][0], v[z][1]);
                double* rp = red + (size_t)(z * 2 + cur) * NR * NT * PCH;
                if (OUTL) {
                    const double pd = quad_sum(dd[z][0] + dd[z][1]);
                    const bool nzq = (__ballot_sync(FULL, nzflag) & qmask) != 0u;
                    *reinterpret_cast<double2*>(Sd + (size_t)(z * 2 + cur) * ROW + g * NPS + s0) = make_double2(dd[z][0], dd[z][1]);
                    if (q == 0) { rp[(NT + w) * PCH + g] = pd; rp[(2 * NT + w) * PCH + g] = nzq ? 1.0 : 0.0; }
                }
                if (q == 0) rp[w * PCH + g] = pv;
            }
            __syncthreads();
        }
#pragma unroll
        for (int z = 0; z < WS; ++z)
            if (have[z] && w == 0 && q == 0) a.chain_ll[c[z]] = acc[z].value();
        __syncthreads();                                    // the buffers are cleared for the next chain groups
    }
}

template <int NT, bool OUTL, bool BSM, int WS>
constexpr size_t wide2_backward_smem()
{
    return sizeof(double) * ((size_t)WS * 2 * PCH * WideGeom<NT>::NPS * (OUTL ? 2 : 1)       // Sw (, Sb)
                             + (size_t)WS * PCH * WideGeom<NT>::NPS                          // Su
                             + (size_t)WS * 2 * NT * PCH + (OUTL ? (size_t)WS * NT * PCH : 0)   // red (, redn)
                             + (BSM ? (size_t)NT * WideGeom<NT>::KS * 32 : 0));              // B fragments
}

// Backward + statistics, two chain sets per block.  Per step and set (frame f downwards): publish w = p_f bn (and bn for
// the outlier rule) -- barrier 1 -- xi product of the previous step, d = A w for the warp's tile, partial sums of
// alpha_{f-1} d and of d -- barrier 2 -- S and sum d complete: u = alpha_{f-1} / S published, gamma and moments, bn = d / sum d.
template <int EM, int NT, bool OUTL, bool BSM, int WS>
__global__ void WIDE_KERNEL_ATTR(NT) k_backward_stats_wide2(const BwdArgs a)
{
    constexpr int KS = WideGeom<NT>::KS, NPS = WideGeom<NT>::NPS, ROW = PCH * NPS;
    PANEL_DYN_SMEM(wsm);
    double* const Sw = wsm;                                 // [WS][2][ROW]
    double* const Sb = Sw + WS * 2 * ROW;                   // [WS][2][ROW]  (OUTL only)
    double* const Su = Sb + (OUTL ? WS * 2 * ROW : 0);      // [WS][ROW]
    double* const red = Su + WS * ROW;                      // [WS][2][NT][PCH] partial S, partial sum of d
    double* const redn = red + WS * 2 * NT * PCH;           // [WS][NT][PCH]    any density != 0 (OUTL only)
    double* const Bsm = redn + (OUTL ? WS * NT * PCH : 0);  // [NT][KS][32]     B fragments (BSM only)
    const int N = a.N;
    const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3, w = threadIdx.x >> 5;
    const unsigned qmask = 0xFu << (4 * g);
    const int s0 = 8 * w + 2 * q;
    const bool ok0 = s0 < N, ok1 = s0 + 1 < N;
    const bool pair_ok = ((N & 1) == 0) && ((reinterpret_cast<uintptr_t>(a.alpha) & 15u) == 0);
    // d = A w: contraction index j = 4 ks + q, output i = 8 w + g
    double Bt[BSM ? 1 : KS];
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
        const int j = 4 * ks + q, i = 8 * w + g;
        const double x = (i < N && j < N) ? a.A[i * N + j] : 0.0;
        if (BSM) Bsm[(w * KS + ks) * 32 + lane] = x;
        else Bt[BSM ? 0 : ks] = x;
    }
    const double* const Bw = Bsm + (size_t)w * KS * 32 + lane;
    double X[NT][2];
#pragma unroll
    for (int mt = 0; mt < NT; ++mt) { X[mt][0] = 0.0; X[mt][1] = 0.0; }
    double mu[2] = {0.0, 0.0}, isg[2] = {1.0, 1.0}, lnrm[2] = {0.0, 0.0};
    if (EM == EM_GAUSS) {
#pragma unroll
        for (int r = 0; r < 2; ++r)
            if (s0 + r < N) {
                const double sg = a.em.sigma[s0 + r];
                mu[r] = a.em.mu[s0 + r];
                isg[r] = 1.0 / (sqrt(2.0) * sg);
                lnrm[r] = log(1.0 / (sqrt(2.0 * 3.14159265358979323846) * sg));
            }
    }
    double st_g[2] = {0.0, 0.0}, st_gd[2] = {0.0, 0.0}, st_gdd[2] = {0.0, 0.0};
    const long long nstat = (long long)N * N + 4 * N;
    double* out = a.partials + (long long)blockIdx.x * nstat;
    for (int j = threadIdx.x; j < N; j += blockDim.x) out[(long long)N * N + j] = 0.0;   // gamma0: atomics below
    __syncthreads();

    auto load2 = [&](const double* src, double& x0, double& x1) {   // src -> element s0 of a (rows, N) row
        if (pair_ok && ok1) { const double2 t = *reinterpret_cast<const double2*>(src); x0 = t.x; x1 = t.y; }
        else { x0 = ok0 ? src[0] : 0.0; x1 = ok1 ? src[1] : 0.0; }
    };
    auto xi_product = [&](int z, int buf) {
        const double* sw = Sw + (size_t)(z * 2 + buf) * ROW;
        const double* su = Su + (size_t)z * ROW;
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
            const double wb = sw[(4 * kk + q) * NPS + 8 * w + g];
#pragma unroll
            for (int mt = 0; mt < NT; ++mt) dmma(X[mt][0], X[mt][1], su[(4 * kk + q) * NPS + 8 * mt + g], wb);
        }
    };

    for (int base = blockIdx.x * (WS * PCH); base < a.ch.n; base += gridDim.x * (WS * PCH)) {
        bool have[WS], virt[WS], pending_xi[WS];
        int c[WS], t0[WS], T[WS], e[WS], fstart[WS], mode[WS], maxpre[WS];
        long long trow[WS];
        int total = 0;
#pragma unroll
        for (int z = 0; z < WS; ++z) {
            const int idx = base + z * PCH + g;
            have[z] = idx < a.ch.n;
            c[z] = -1; t0[z] = 0; T[z] = 0; e[z] = 0; fstart[z] = 0; mode[z] = 0; virt[z] = false; trow[z] = 0;
            pending_xi[z] = false;
            if (have[z]) {
                c[z] = a.ch.list ? a.ch.list[idx] : idx;
                const int len = a.ch.len[c[z]];
                t0[z] = a.ch.t0[c[z]];
                T[z] = a.ch.T[c[z]];
                trow[z] = a.ch.row0[c[z]] - t0[z];
                e[z] = t0[z] + len;
                if (e[z] >= T[z]) { virt[z] = true; fstart[z] = T[z]; }
                else if (chain_exact_start(a.ch, c[z])) { fstart[z] = e[z]; mode[z] = 2; }
                else { fstart[z] = min(T[z] - 1, e[z] + (a.ch.warmv ? a.ch.warmv[c[z]] : a.ch.warm) - 1); }
            }
            maxpre[z] = __reduce_max_sync(FULL, have[z] ? (fstart[z] - (e[z] - 1)) : 0);
            total = max(total, maxpre[z] + __reduce_max_sync(FULL, have[z] ? (e[z] - (t0[z] + 1)) : 0));
        }
        for (int k = threadIdx.x; k < WS * 2 * ROW; k += blockDim.x) { Sw[k] = 0.0; if (OUTL) Sb[k] = 0.0; }
        for (int k = threadIdx.x; k < WS * ROW; k += blockDim.x) Su[k] = 0.0;
        __syncthreads();

        double bn[WS][2], o_next[WS], al_next[WS][2], pn[WS][2];
        int symA[WS];
        auto frame_of = [&](int z, int s) -> int { return (e[z] - 1) + maxpre[z] - s; };
        auto em_row = [&](int z, int s) -> long long { return trow[z] + min(max(frame_of(z, s), t0[z]), T[z] - 1); };
        auto al_row = [&](int z, int s) -> long long { return trow[z] + min(max(frame_of(z, s) - 1, t0[z]), e[z] - 1); };
#pragma unroll
        for (int z = 0; z < WS; ++z) {
            bn[z][0] = ok0 ? 1.0 / N : 0.0;                  // beta_{T-1} = 1/N (_hidden.c:76-77); warm-up start
            bn[z][1] = ok1 ? 1.0 / N : 0.0;
            o_next[z] = 0.0; al_next[z][0] = al_next[z][1] = 0.0; pn[z][0] = pn[z][1] = 0.0; symA[z] = 0;
            if (have[z] && mode[z] == 2) {
                const double* hv = chain_start_vec(a.ch, a.hand_end, c[z], c[z] + 1, N);
                if (ok0) bn[z][0] = hv[s0];
                if (ok1) bn[z][1] = hv[s0 + 1];
            }
            if (have[z]) {
                if (EM == EM_GAUSS) o_next[z] = a.em.obs[em_row(z, 0)];
                if (EM == EM_DISC) {
                    wide_table2<EM>(a.em, 0, a.em.sym[em_row(z, 0)], N, s0, ok0, ok1, pn[z]);
                    symA[z] = a.em.sym[em_row(z, 1)];
                }
                if (EM == EM_POBS) wide_table2<EM>(a.em, em_row(z, 0), 0, N, s0, ok0, ok1, pn[z]);
                load2(a.alpha + al_row(z, 0) * N + s0, al_next[z][0], al_next[z][1]);
            }
        }

        for (int s = 0; s < total; ++s) {
            const int cur = s & 1;
            int f[WS], sym_emit[WS];
            bool on[WS], isvirt[WS], act[WS];
            double al[WS][2], wv[WS][2], d[WS][2], gq[WS][2];
            // ---- publish w = p bn (and bn) of both sets
#pragma unroll
            for (int z = 0; z < WS; ++z) {
                f[z] = frame_of(z, s);
                on[z] = have[z] && f[z] <= fstart[z] && f[z] >= t0[z] + 1;
                isvirt[z] = on[z] && virt[z] && f[z] == T[z];
                al[z][0] = al_next[z][0]; al[z][1] = al_next[z][1];
                double p[2] = {0.0, 0.0};
                sym_emit[z] = 0;                            // symbol of frame f-1, the frame this step emits
                if (have[z]) {
                    load2(a.alpha + al_row(z, s + 1) * N + s0, al_next[z][0], al_next[z][1]);
                    if (EM == EM_GAUSS) {
                        const double o = o_next[z];
                        o_next[z] = a.em.obs[em_row(z, s + 1)];   // frame f-1: also the emitted frame's observation
                        wide_gauss2(o, mu, isg, lnrm, ok0, ok1, p);
                    } else {
                        p[0] = pn[z][0]; p[1] = pn[z][1];
                        if (EM == EM_DISC) {
                            sym_emit[z] = symA[z];
                            wide_table2<EM>(a.em, 0, symA[z], N, s0, ok0, ok1, pn[z]);
                            symA[z] = a.em.sym[em_row(z, s + 2)];
                        } else {
                            wide_table2<EM>(a.em, em_row(z, s + 1), 0, N, s0, ok0, ok1, pn[z]);
                        }
                    }
                }
                act[z] = on[z] && !isvirt[z];
                wv[z][0] = act[z] ? p[0] * bn[z][0] : 0.0;
                wv[z][1] = act[z] ? p[1] * bn[z][1] : 0.0;
                *reinterpret_cast<double2*>(Sw + (size_t)(z * 2 + cur) * ROW + g * NPS + s0) = make_double2(wv[z][0], wv[z][1]);
                if (OUTL) {
                    const bool nzq = (__ballot_sync(FULL, (p[0] != 0.0) || (p[1] != 0.0)) & qmask) != 0u;
                    *reinterpret_cast<double2*>(Sb + (size_t)(z * 2 + cur) * ROW + g * NPS + s0) =
                        make_double2(act[z] ? bn[z][0] : 0.0, act[z] ? bn[z][1] : 0.0);
                    if (q == 0) redn[(z * NT + w) * PCH + g] = nzq ? 1.0 : 0.0;
                }
            }
            __syncthreads();                                // ---- barrier 1

#pragma unroll
            for (int z = 0; z < WS; ++z)
                if (pending_xi[z]) xi_product(z, cur ^ 1);

            // ---- d = A w for both sets with one pass over the B fragments
            bool use_b[WS];
            const double* src[WS];
#pragma unroll
            for (int z = 0; z < WS; ++z) {
                use_b[z] = false;
                if (OUTL) {
                    double nz = 0.0;
#pragma unroll
                    for (int w2 = 0; w2 < NT; w2 += 4)
                        if (w2 + q < NT) nz += redn[(z * NT + w2 + q) * PCH + g];
                    nz = quad_sum(nz);
                    use_b[z] = a.em.ignore_outliers && act[z] && nz == 0.0;   // outputmodel.py:126-130
                }
                src[z] = ((OUTL && use_b[z]) ? Sb : Sw) + (size_t)(z * 2 + cur) * ROW + g * NPS;
            }
            double acc[WS][2][2];
#pragma unroll
            for (int z = 0; z < WS; ++z) { acc[z][0][0] = acc[z][0][1] = acc[z][1][0] = acc[z][1][1] = 0.0; }
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                const double b = BSM ? Bw[ks * 32] : Bt[BSM ? 0 : ks];
#pragma unroll
                for (int z = 0; z < WS; ++z) dmma(acc[z][ks & 1][0], acc[z][ks & 1][1], src[z][4 * ks + q], b);
            }
#pragma unroll
            for (int z = 0; z < WS; ++z) {
                d[z][0] = acc[z][0][0] + acc[z][1][0];
                d[z][1] = acc[z][0][1] + acc[z][1][1];
                if (isvirt[z]) { d[z][0] = ok0 ? 1.0 : 0.0; d[z][1] = ok1 ? 1.0 : 0.0; }
                if (OUTL && use_b[z]) {                      // the xi product of the next step reads W from Sw
                    wv[z][0] = act[z] ? bn[z][0] : 0.0; wv[z][1] = act[z] ? bn[z][1] : 0.0;
                    *reinterpret_cast<double2*>(Sw + (size_t)(z * 2 + cur) * ROW + g * NPS + s0) = make_double2(wv[z][0], wv[z][1]);
                }
                if (act[z] && f[z] == e[z]) {
                    if (ok0) a.hand_used[(long long)c[z] * N + s0] = bn[z][0];
                    if (ok1) a.hand_used[(long long)c[z] * N + s0 + 1] = bn[z][1];
                }
                const bool emit = on[z] && (f[z] - 1) < e[z];
                gq[z][0] = emit ? al[z][0] * d[z][0] : 0.0;
                gq[z][1] = emit ? al[z][1] * d[z][1] : 0.0;
                const double pS = quad_sum(gq[z][0] + gq[z][1]), pb = quad_sum(d[z][0] + d[z][1]);
                if (q == 0) { red[((z * 2 + 0) * NT + w) * PCH + g] = pS; red[((z * 2 + 1) * NT + w) * PCH + g] = pb; }
            }
            __syncthreads();                                // ---- barrier 2

#pragma unroll
            for (int z = 0; z < WS; ++z) {
                const bool emit = on[z] && (f[z] - 1) < e[z];
                const bool xi = emit && !isvirt[z];
                double S = 0.0, sbn = 0.0;
#pragma unroll
                for (int w2 = 0; w2 < NT; w2 += 4)
                    if (w2 + q < NT) { S += red[((z * 2 + 0) * NT + w2 + q) * PCH + g]; sbn += red[((z * 2 + 1) * NT + w2 + q) * PCH + g]; }
                S = quad_sum(S);
                sbn = quad_sum(sbn);
                const double rS = 1.0 / S;
                *reinterpret_cast<double2*>(Su + (size_t)z * ROW + g * NPS + s0) =
                    make_double2(xi ? al[z][0] * rS : 0.0, xi ? al[z][1] * rS : 0.0);
                pending_xi[z] = __any_sync(FULL, xi);
                if (emit) {
                    const long long orow = trow[z] + (f[z] - 1);
                    const double gam[2] = {gq[z][0] * rS, gq[z][1] * rS};
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        if (s0 + r >= N) continue;
                        st_g[r] += gam[r];
                        if (f[z] - 1 == 0) atomicAdd(out + (long long)N * N + s0 + r, gam[r]);
                        if (EM == EM_GAUSS) {
                            const double dv = o_next[z] - mu[r];
                            st_gd[r] = fma(gam[r], dv, st_gd[r]);
                            st_gdd[r] = fma(gam[r], dv * dv, st_gdd[r]);
                        }
                        if (EM == EM_DISC && a.Bnum) atomicAdd(a.Bnum + (long long)(s0 + r) * a.em.M + sym_emit[z], gam[r]);
                        if (a.gamma) a.gamma[orow * N + s0 + r] = gam[r];
                    }
                    if (f[z] - 1 == t0[z] && t0[z] > 0) {
                        const double r2 = (sbn != 0.0) ? 1.0 / sbn : 1.0;
                        if (ok0) a.hand_end[(long long)c[z] * N + s0] = d[z][0] * r2;
                        if (ok1) a.hand_end[(long long)c[z] * N + s0 + 1] = d[z][1] * r2;
                    }
                }
                if (on[z]) {
                    const double r2 = (sbn != 0.0) ? 1.0 / sbn : 1.0;          // _hidden.c:104-107
                    bn[z][0] = d[z][0] * r2;
                    bn[z][1] = d[z][1] * r2;
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int z = 0; z < WS; ++z)
            if (pending_xi[z]) xi_product(z, (total - 1) & 1);
        __syncthreads();                                    // the buffers are cleared for the next chain groups
    }

    // ---- the block's row of partial statistics: [X (N*N) | gamma0 (N) | sum gamma | sum gamma d | sum gamma d^2]
#pragma unroll
    for (int mt = 0; mt < NT; ++mt) {
        const int i = 8 * mt + g;
        if (i < N) {
            if (ok0) out[(long long)i * N + s0] = X[mt][0];
            if (ok1) out[(long long)i * N + s0 + 1] = X[mt][1];
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
#pragma unroll
        for (int off = 4; off < 32; off <<= 1) {
            st_g[r] += __shfl_xor_sync(FULL, st_g[r], off);
            st_gd[r] += __shfl_xor_sync(FULL, st_gd[r], off);
            st_gdd[r] += __shfl_xor_sync(FULL, st_gdd[r], off);
        }
        if (g == 0 && s0 + r < N) {
            out[(long long)N * N + N + s0 + r] = st_g[r];
            out[(long long)N * N + 2 * N + s0 + r] = st_gd[r];
            out[(long long)N * N + 3 * N + s0 + r] = st_gdd[r];
        }
    }
}

// ================================================================================================
// Viterbi for 32 < N <= 104 with the transition-matrix column in registers (same opt-in as the panel kernels).
// k_viterbi_team walks its two N-long loops (first-maximum scan, sequential row sum) one shared-memory round trip at a
// time: ~6000 cycles per frame at N = 100 (C4: 4.27 s for 4096 x 1e5 frames).  Here thread j keeps A[:, j] in registers, the
// scan runs as four independent first-maximum scans over index blocks that are combined in block order with the same
// strict '>' (the earliest index among equal maxima wins either way, _hidden.c:186-200), and the row sum -- sequential by
// definition of bit-exactness (_hidden.c:254-259) -- is an unrolled chain of additions fed by 16-byte loads.  Padded states
// hold exact zeros, which neither win a strict comparison against a non-negative maximum nor change a sum.
// Output: the shifted back-pointer map F[t][s'] of k_viterbi_team's CHASE mode (uint8), resolved by the k_chase_* kernels.
// ================================================================================================
template <int EM, int NMAX>
__global__ void __launch_bounds__(((NMAX + 31) / 32) * 32) k_viterbi_regs(const VitArgs a)
{
    constexpr int Q = NMAX / 4;
    __shared__ __align__(16) double ub[NMAX];              // unnormalised row
    __shared__ __align__(16) double vb[NMAX];              // normalised row
    const int N = a.N, j = threadIdx.x;
    const bool jv = j < N;
    double Acol[NMAX];
#pragma unroll
    for (int i = 0; i < NMAX; ++i) Acol[i] = (jv && i < N) ? a.A[i * N + j] : 0.0;
    double mu = 0.0, sigma = 1.0;
    if (EM == EM_GAUSS && jv) { mu = a.em.mu[j]; sigma = a.em.sigma[j]; }
    const double pi_j = jv ? a.pi[j] : 0.0;
    unsigned char* bp = reinterpret_cast<unsigned char*>(a.backptr);
    for (int i = threadIdx.x; i < NMAX; i += blockDim.x) { ub[i] = 0.0; vb[i] = 0.0; }
    __syncthreads();

    auto em_raw = [&](long long row) -> double {
        if (EM == EM_POBS) return a.em.pobs[row * N + j];
        if (EM == EM_GAUSS) return a.em.obs[row];
        return a.em.Bt[(long long)a.em.sym[row] * N + j];
    };

    for (int k = blockIdx.x; k < a.K; k += gridDim.x) {
        const long long row0 = a.offsets[k];
        const int T = (int)(a.offsets[k + 1] - row0);
        double raw_next = (jv && T > 0) ? em_raw(row0) : 0.0;
        for (int t = 0; t < T; ++t) {
            const double raw = raw_next;
            if (jv && t + 1 < T) raw_next = em_raw(row0 + t + 1);
            double p = 0.0;
            if (jv) p = (EM == EM_GAUSS) ? gauss_pdf(raw, mu, sigma) : raw;
            if (EM != EM_POBS && a.em.ignore_outliers) {
                if (!__syncthreads_or(p != 0.0 ? 1 : 0)) p = jv ? 1.0 : 0.0;       // outputmodel.py:126-130
            }
            double vn = 0.0;
            int best = 0;
            if (t == 0) {
                vn = __dmul_rn(p, pi_j);
            } else {
                double m[4], vbest[4], abest[4];
                int bi[4];
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    vbest[b] = vb[b * Q];
                    abest[b] = Acol[b * Q];
                    m[b] = __dmul_rn(vbest[b], abest[b]);
                    bi[b] = b * Q;
                }
#pragma unroll
                for (int ii = 1; ii < Q; ++ii) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const double v = vb[b * Q + ii];
                        const double h = __dmul_rn(v, Acol[b * Q + ii]);
                        if (h > m[b]) { m[b] = h; bi[b] = b * Q + ii; vbest[b] = v; abest[b] = Acol[b * Q + ii]; }
                    }
                }
                double mm = m[0], vsel = vbest[0], asel = abest[0];
                best = bi[0];
#pragma unroll
                for (int b = 1; b < 4; ++b)
                    if (m[b] > mm) { mm = m[b]; best = bi[b]; vsel = vbest[b]; asel = abest[b]; }
                if (jv) {
                    bp[(row0 + t - 1) * N + j] = (unsigned char)best;
                    vn = __dmul_rn(__dmul_rn(p, vsel), asel);                    // (p_j v_best) A[best][j], _hidden.c:247-250
                }
            }
            if (jv) ub[j] = vn;
            __syncthreads();
            double ssum = 0.0;
#pragma unroll
            for (int i = 0; i < NMAX; ++i) ssum = __dadd_rn(ssum, ub[i]);        // j-sequential, + 0.0 for the padding
            if (jv) vb[j] = __ddiv_rn(vn, ssum);
            __syncthreads();
        }
        // path[T-1] = first maximum of the last row (_hidden.c:268): the last row of the map holds it for every s'
        if (T > 0) {
            int best = 0;
            double m = vb[0];
            for (int i = 1; i < N; ++i)
                if (vb[i] > m) { m = vb[i]; best = i; }
            if (jv) bp[(row0 + T - 1) * N + j] = (unsigned char)best;
        }
        __syncthreads();
    }
}

// ================================================================================================
// Viterbi for 32 < N <= 128 with the transition matrix in SHARED memory and R trajectories per block ("k_viterbi_multi").
//
// k_viterbi_regs keeps A[:, j] in registers: 208 registers per thread, two blocks (= two trajectories) per SM, and every
// frame is one long dependent chain -- compare-select scan, then the 104-long sequential row sum: measured 4.2-4.7 s for C4's
// 4.096e8 frames, no faster than the team kernel.  Here thread j still owns state j, but A is read from shared memory
// (row-major with a padded stride: thread j reads A[i][j], consecutive words, conflict-free) and is shared by the R
// trajectories the block walks in lock step: the loaded entry is used R times, the R scans and the R sequential sums are
// independent instruction streams that fill each other's latency, and only the running maximum and its index are carried
// through the scan (the winning v_i and A_ij are re-read from shared memory afterwards instead of being dragged along by
// selects).  Warp r computes the sequential sum of trajectory r.  Arithmetic and order are _hidden.c:229-265's: products
// v_i A_ij, first maximum with strict '>', (p_j v_best) A_best,j, j-sequential sum, true division: bit-exact.
// Output: the shifted back-pointer map of k_viterbi_team's CHASE mode (uint8), resolved by the k_chase_* kernels.
// ================================================================================================
// SUB independent groups of `sthr` threads ("sub-blocks") share ONE copy of the transition matrix in shared memory: the
// matrix (83 KB at N = 100) limits an SM to two blocks, and with one group per block that is two warps per scheduler; four
// groups per block make it eight.  The groups synchronise among themselves with named barriers (bar.sync id, sthr).
__device__ __forceinline__ void sub_barrier(int sub, int sthr, int nsub)
{
#ifdef PANEL_HOST_EMU
    __syncthreads();                                        // the emulated build runs one group per block
#else
    if (nsub == 1) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(sub + 1), "r"(sthr) : "memory");
#endif
}

#ifndef VITERBI_MULTI_MINB
#define VITERBI_MULTI_MINB 1
#endif
template <int EM, int R>
__global__ void __launch_bounds__(512, VITERBI_MULTI_MINB) k_viterbi_multi(const VitArgs a, int NPS, int sthr)
{
    PANEL_DYN_SMEM(vsm);
    const int N = a.N, nsub = blockDim.x / sthr, sub = threadIdx.x / sthr;
    const int j = threadIdx.x - sub * sthr, nthr = sthr, wid = j >> 5, nwarp = sthr >> 5;
    double* const As = vsm;                                 // [N][NPS], shared by the groups
    const size_t per_sub = 2 * (size_t)R * NPS + R + 2 * R; // doubles per group: vb, ub, ssum, anynz (as 4 R ints)
    double* const vb = As + (size_t)N * NPS + sub * per_sub;   // [R][NPS] normalised rows
    double* const ub = vb + R * NPS;                        // [R][NPS] unnormalised rows
    double* const ssum = ub + R * NPS;                      // [R]
    int* const anynz = reinterpret_cast<int*>(ssum + R);    // [R][4] per warp: any density != 0 (outlier rule)
    const bool jv = j < N;
    for (int k = threadIdx.x; k < N * NPS; k += blockDim.x) {
        const int i = k / NPS, c = k - i * NPS;
        As[k] = (c < N) ? a.A[i * N + c] : 0.0;
    }
    for (int k = j; k < 2 * R * NPS; k += nthr) vb[k] = 0.0;
    double mu = 0.0, sigma = 1.0;
    if (EM == EM_GAUSS && jv) { mu = a.em.mu[j]; sigma = a.em.sigma[j]; }
    const double pi_j = jv ? a.pi[j] : 0.0;
    unsigned char* bp = reinterpret_cast<unsigned char*>(a.backptr);
    const bool outl = (EM != EM_POBS) && a.em.ignore_outliers;
    __syncthreads();

    for (int k0 = (blockIdx.x * nsub + sub) * R; k0 < a.K; k0 += gridDim.x * nsub * R) {
        long long row0[R];
        int T[R], Tmax = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int k = k0 + r;
            row0[r] = (k < a.K) ? a.offsets[k] : 0;
            T[r] = (k < a.K) ? (int)(a.offsets[k + 1] - row0[r]) : 0;
            Tmax = max(Tmax, T[r]);
        }
        auto em_raw = [&](int r, int t) -> double {
            if (!jv || t >= T[r]) return 0.0;
            const long long row = row0[r] + t;
            if (EM == EM_POBS) return a.em.pobs[row * N + j];
            if (EM == EM_GAUSS) return a.em.obs[row];
            return a.em.Bt[(long long)a.em.sym[row] * N + j];
        };
        double raw_next[R];
#pragma unroll
        for (int r = 0; r < R; ++r) raw_next[r] = em_raw(r, 0);
        for (int t = 0; t < Tmax; ++t) {
            double p[R], vn[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const double raw = raw_next[r];
                raw_next[r] = em_raw(r, t + 1);
                p[r] = 0.0;
                if (jv && t < T[r]) p[r] = (EM == EM_GAUSS) ? gauss_pdf(raw, mu, sigma) : raw;
            }
            if (outl) {                                     // outputmodel.py:126-130, one vote per trajectory
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const unsigned nzw = __ballot_sync(FULL, p[r] != 0.0);
                    if ((j & 31) == 0) anynz[r * 4 + wid] = nzw != 0u;
                }
                sub_barrier(sub, sthr, nsub);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    int any = 0;
                    for (int w2 = 0; w2 < nwarp; ++w2) any |= anynz[r * 4 + w2];
                    if (!any) p[r] = (jv && t < T[r]) ? 1.0 : 0.0;
                }
            }
            if (t == 0) {
#pragma unroll
                for (int r = 0; r < R; ++r) vn[r] = __dmul_rn(p[r], pi_j);
            } else {
                double m[R];
                int bi[R];
#pragma unroll
                for (int r = 0; r < R; ++r) { m[r] = __dmul_rn(vb[r * NPS], As[j]); bi[r] = 0; }
                // two predecessor states per step: the rows' entries arrive as one 16-byte broadcast load per trajectory (the
                // scan is bound by the LSU wavefronts of these loads, 2 per LDS.64 against 2.4 per LDS.128)
                int i = 1;
                if (N > 1) {
                    const double a1 = As[NPS + j];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const double h = __dmul_rn(vb[r * NPS + 1], a1);
                        if (h > m[r]) { m[r] = h; bi[r] = 1; }              // first maximum, _hidden.c:186-200
                    }
                    i = 2;
                }
#pragma unroll 2
                for (; i + 1 < N; i += 2) {
                    const double a0 = As[i * NPS + j], a1 = As[(i + 1) * NPS + j];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const double2 v2 = *reinterpret_cast<const double2*>(vb + r * NPS + i);
                        const double h0 = __dmul_rn(v2.x, a0), h1 = __dmul_rn(v2.y, a1);
                        if (h0 > m[r]) { m[r] = h0; bi[r] = i; }
                        if (h1 > m[r]) { m[r] = h1; bi[r] = i + 1; }
                    }
                }
                if (i < N) {
                    const double a0 = As[i * NPS + j];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const double h = __dmul_rn(vb[r * NPS + i], a0);
                        if (h > m[r]) { m[r] = h; bi[r] = i; }
                    }
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    if (jv && t < T[r]) bp[(row0[r] + t - 1) * N + j] = (unsigned char)bi[r];
                    vn[r] = __dmul_rn(__dmul_rn(p[r], vb[r * NPS + bi[r]]), As[bi[r] * NPS + j]);   // _hidden.c:247-250
                }
            }
            // (ub's readers -- the sums of the previous frame -- finished before that frame's third barrier)
            if (j < NPS) {
#pragma unroll
                for (int r = 0; r < R; ++r) ub[r * NPS + j] = (jv && t < T[r]) ? vn[r] : 0.0;
            }
            sub_barrier(sub, sthr, nsub);
            {   // j-sequential sums (_hidden.c:254-259): warp w adds up the rows w, w + nwarp, ... -- up to four independent
                // chains of additions interleaved in one loop
                constexpr int RW = (R + 1) / 2;             // rows per warp at two warps per block (the fewest)
                double sacc[RW];
#pragma unroll
                for (int q = 0; q < RW; ++q) sacc[q] = 0.0;
                for (int i = 0; i < N; ++i) {
#pragma unroll
                    for (int q = 0; q < RW; ++q) {
                        const int r = wid + q * nwarp;
                        if (r < R) sacc[q] = __dadd_rn(sacc[q], ub[r * NPS + i]);
                    }
                }
                if ((j & 31) == 0) {
#pragma unroll
                    for (int q = 0; q < RW; ++q)
                        if (wid + q * nwarp < R) ssum[wid + q * nwarp] = sacc[q];
                }
            }
            sub_barrier(sub, sthr, nsub);
            if (j < NPS) {
#pragma unroll
                for (int r = 0; r < R; ++r)
                    if (t < T[r]) vb[r * NPS + j] = jv ? __ddiv_rn(vn[r], ssum[r]) : 0.0;
            }
            sub_barrier(sub, sthr, nsub);
        }
        // path[T-1] = first maximum of the last row (_hidden.c:268): the last row of the map holds it for every s'
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (T[r] <= 0) continue;
            int best = 0;
            double mm = vb[r * NPS];
            for (int i = 1; i < N; ++i) {
                const double x = vb[r * NPS + i];
                if (x > mm) { mm = x; best = i; }
            }
            if (jv) bp[(row0[r] + T[r] - 1) * N + j] = (unsigned char)best;
        }
        sub_barrier(sub, sthr, nsub);
        for (int k = j; k < 2 * R * NPS; k += nthr) vb[k] = 0.0;
        sub_barrier(sub, sthr, nsub);
    }
}

// ================================================================================================
// Time-chunked Viterbi, N <= 32 (C5: one trajectory of 1e9 frames, where the strictly sequential recursion of
// k_viterbi_team would take minutes).  One warp per chain, lane j = state j, A[:, j] in registers.  A chain that does not
// start its trajectory warms its normalised max-product vector up on the frames before it (the max-product filter forgets
// its start like the sum-product one once the survivor paths have coalesced); the hand-over is certified afterwards by
// the same component-wise relative comparison as the forward filter's (certify.cu), with exact re-runs of the chains that
// fail.  Arithmetic per frame is exactly k_viterbi_team's (_hidden.c:229-265 operation order).  Because a certified
// hand-over still differs from the sequential one in the last digits, a decision (arg max over predecessors) is only
// provably the sequential one if its best and second-best candidates differ by more than that: every decision whose
// relative margin is below margin_min sets its bit in `flagmap`.  Only decisions ON the resolved path can change it (by
// induction from the last frame backwards), so after the path chase k_viterbi_path_flags counts the flagged decisions the
// path went through; if there is one, the caller recomputes the map with the sequential kernel -- a returned path is always
// the reference's.  (Measured on dalton data: P(margin < eps) = 0.25 eps per decision but 0.01 eps per ON-PATH decision, i.e.
// 1e-4 expected fallbacks for 1e9 frames at eps = 1e-11, against 8 flagged decisions if every decision counted at 1e-9.)
// ================================================================================================
template <int EM>
__global__ void __launch_bounds__(PW * 32) k_viterbi_chain32(const VitChainArgs a)
{
    __shared__ __align__(16) double ub[PW][32];
    __shared__ __align__(16) double vb[PW][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int gw = blockIdx.x * PW + wib, nw = gridDim.x * PW;
    const int N = a.N, j = lane;
    const bool jv = j < N;
    double* u = ub[wib];
    double* v = vb[wib];
    double Acol[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) Acol[i] = (jv && i < N) ? a.A[i * N + j] : 0.0;
    double mu = 0.0, sigma = 1.0;
    if (EM == EM_GAUSS && jv) { mu = a.em.mu[j]; sigma = a.em.sigma[j]; }
    const double pi_j = jv ? a.pi[j] : 0.0;
    unsigned char* bp = reinterpret_cast<unsigned char*>(a.backptr);

    auto em_raw = [&](long long row) -> double {
        if (EM == EM_POBS) return a.em.pobs[row * N + j];
        if (EM == EM_GAUSS) return a.em.obs[row];
        return a.em.Bt[(long long)a.em.sym[row] * N + j];
    };

    for (int idx = gw; idx < a.ch.n; idx += nw) {
        const int c = a.ch.list ? a.ch.list[idx] : idx;
        const int len = a.ch.len[c], t0 = a.ch.t0[c], T = a.ch.T[c];
        const long long trow = a.ch.row0[c] - t0;
        const int tend = t0 + len;
        int tstart = 0, mode = 0;                           // mode 0: pi at frame 0, 1: uniform warm-up start, 2: exact vector
        if (t0 == 0) { tstart = 0; mode = 0; }
        else if (chain_exact_start(a.ch, c)) { tstart = t0 - 1; mode = 2; }
        else { tstart = max(0, t0 - (a.ch.warmv ? a.ch.warmv[c] : a.ch.warm)); mode = (tstart == 0) ? 0 : 1; }
        u[lane] = 0.0;
        v[lane] = 0.0;
        __syncwarp();
        if (mode == 2) {
            if (jv) {
                const double x = chain_start_vec(a.ch, a.hand_end, c, c - 1, N)[j];
                v[j] = x;
                a.hand_used[(long long)c * N + j] = x;
            }
            __syncwarp();
        }
        const int tfirst = (mode == 2) ? t0 : tstart;
        double raw_next = jv ? em_raw(trow + tfirst) : 0.0;
        for (int t = tfirst; t < tend; ++t) {
            const double raw = raw_next;
            if (jv && t + 1 < tend) raw_next = em_raw(trow + t + 1);
            double p = 0.0;
            if (jv) p = (EM == EM_GAUSS) ? gauss_pdf(raw, mu, sigma) : raw;
            if (EM != EM_POBS && a.em.ignore_outliers) {
                if (!__any_sync(FULL, p != 0.0)) p = jv ? 1.0 : 0.0;              // outputmodel.py:126-130
            }
            double vn;
            if (t == tstart && mode != 2) {
                vn = (mode == 0) ? __dmul_rn(p, pi_j) : p;
            } else {
                double m[4], m2[4], vbest[4], abest[4];
                int bi[4];
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    vbest[b] = v[8 * b];
                    abest[b] = Acol[8 * b];
                    m[b] = __dmul_rn(vbest[b], abest[b]);
                    m2[b] = -1.0;
                    bi[b] = 8 * b;
                }
#pragma unroll
                for (int ii = 1; ii < 8; ++ii) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const double x = v[8 * b + ii];
                        const double h = __dmul_rn(x, Acol[8 * b + ii]);
                        if (h > m[b]) { m2[b] = m[b]; m[b] = h; bi[b] = 8 * b + ii; vbest[b] = x; abest[b] = Acol[8 * b + ii]; }
                        else if (h > m2[b]) m2[b] = h;
                    }
                }
                double mm = m[0], second = m2[0], vsel = vbest[0], asel = abest[0];
                int best = bi[0];
#pragma unroll
                for (int b = 1; b < 4; ++b) {
                    if (m[b] > mm) { second = fmax(second, mm); second = fmax(second, m2[b]); mm = m[b]; best = bi[b]; vsel = vbest[b]; asel = abest[b]; }
                    else second = fmax(second, m[b]);
                }
                if (t >= t0) {
                    if (jv) bp[(trow + t - 1) * N + j] = (unsigned char)best;
                    const bool near = jv && mm > 0.0 && (mm - fmax(second, 0.0)) < a.margin_min * mm;
                    const unsigned word = __ballot_sync(FULL, near);
                    if (lane == 0) a.flagmap[trow + t - 1] = word;
                }
                vn = __dmul_rn(__dmul_rn(p, vsel), asel);
            }
            if (jv) u[j] = vn;
            __syncwarp();
            double ssum = 0.0;
#pragma unroll
            for (int i = 0; i < 32; ++i) ssum = __dadd_rn(ssum, u[i]);
            const double vnew = __ddiv_rn(vn, ssum);
            __syncwarp();                                   // everybody has read u and v of this frame
            if (jv) {
                v[j] = vnew;
                if (t == t0 - 1) a.hand_used[(long long)c * N + j] = vnew;
                if (t == tend - 1) a.hand_end[(long long)c * N + j] = vnew;
            }
            __syncwarp();
        }
        if (tend == T) {                                    // path[T-1] = first maximum of the last row (_hidden.c:268)
            int best = 0;
            double m = v[0], second = -1.0;
            for (int i = 1; i < N; ++i) {
                if (v[i] > m) { second = m; m = v[i]; best = i; }
                else if (v[i] > second) second = v[i];
            }
            if (jv) bp[(trow + T - 1) * N + j] = (unsigned char)best;
            const bool near = m > 0.0 && N > 1 && (m - fmax(second, 0.0)) < a.margin_min * m;
            if (lane == 0) a.flagmap[trow + T - 1] = near ? 0xffffffffu : 0u;
        }
        __syncwarp();
    }
}

// On-path flags of the chunked Viterbi: row r of trajectory k holds the decision "state at r given the state at r+1"
// (bit index = path[r+1]); the last row holds the final arg max (any bit).
__global__ void k_viterbi_path_flags(const unsigned* __restrict__ flagmap, const int* __restrict__ path,
                                     const long long* __restrict__ offsets, int K, long long rows, int* counter)
{
    int hits = 0;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x) {
        const unsigned w = flagmap[r];
        if (w == 0u) continue;
        int lo = 0, hi = K;                                 // trajectory of row r: offsets[lo] <= r < offsets[lo + 1]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (offsets[mid] <= r) lo = mid; else hi = mid;
        }
        const bool last = (r == offsets[lo + 1] - 1);
        if (last || ((w >> path[r + 1]) & 1u)) ++hits;
    }
    if (hits) atomicAdd(counter, hits);
}

// ================================================================================================
// Time-chunked Viterbi, 32 < N <= 128 (a trajectory cut in time across devices at the model sizes of C4).  The contract is
// k_viterbi_chain32's -- start modes (pi at frame 0, uniform warm-up, exact hand-over vector), hand_used at t0 - 1 and
// hand_end at the last frame, back-pointers for t >= t0 only, near-tie flags -- and the layout k_viterbi_multi's: thread j
// owns state j in groups of `sthr` threads, A sits in shared memory with the padded stride NPS, one copy per block shared by
// its nsub groups, and every group walks R chains in lock step (the chains of one plan have nearly equal lengths, so the
// shorter ones idle for at most a warm-up's difference).  Arithmetic per frame is _hidden.c:229-265's, bit for bit: products
// v_i A_ij, first maximum with strict '>', (p_j v_best) A_best,j, j-sequential sum, true division.  The flag map has
// NW = ceil(N / 32) words per row, word w bit b standing for the next state 32 w + b (k_viterbi_path_flags_wide); the last
// row of a trajectory is flagged as a whole.
// ================================================================================================
// doubles of shared memory per group of k_viterbi_chain_wide: vb, ub (R x NPS each), ssum (R), anynz (4 R ints), the chains'
// first rows (R) and descriptions (8 R ints)
__host__ __device__ constexpr size_t chain_wide_group_doubles(int NPS, int R) { return 2 * (size_t)R * NPS + 8 * (size_t)R; }

template <int EM, int R>
__global__ void __launch_bounds__(512, 1) k_viterbi_chain_wide(const VitChainArgs a, int NPS, int sthr)
{
    PANEL_DYN_SMEM(vsm);
    const int N = a.N, nsub = blockDim.x / sthr, sub = threadIdx.x / sthr;
    const int j = threadIdx.x - sub * sthr, nthr = sthr, wid = j >> 5, lane = j & 31, nwarp = sthr >> 5;
    const int NW = (N + 31) >> 5;
    double* const As = vsm;                                 // [N][NPS], shared by the groups
    double* const vb = As + (size_t)N * NPS + sub * chain_wide_group_doubles(NPS, R);   // [R][NPS] normalised rows
    double* const ub = vb + R * NPS;                        // [R][NPS] unnormalised rows
    double* const ssum = ub + R * NPS;                      // [R]
    int* const anynz = reinterpret_cast<int*>(ssum + R);    // [R][4] per warp: any density != 0 (outlier rule)
    // the R chains' descriptions live in shared memory, not in registers (at 128 registers per thread they would spill):
    // row of frame 0, and chain, t0, end frame, trajectory length, start frame, first frame walked, start mode
    long long* const trow = reinterpret_cast<long long*>(anynz + 4 * R);   // [R]
    int* const cd = reinterpret_cast<int*>(trow + R);       // [R][8]
    enum { C_C, C_T0, C_TEND, C_T, C_TSTART, C_TFIRST, C_MODE };
    const bool jv = j < N;
    for (int k = threadIdx.x; k < N * NPS; k += blockDim.x) {
        const int i = k / NPS, c = k - i * NPS;
        As[k] = (c < N) ? a.A[i * N + c] : 0.0;
    }
    double mu = 0.0, sigma = 1.0;
    if (EM == EM_GAUSS && jv) { mu = a.em.mu[j]; sigma = a.em.sigma[j]; }
    const double pi_j = jv ? a.pi[j] : 0.0;
    unsigned char* bp = reinterpret_cast<unsigned char*>(a.backptr);
    const bool outl = (EM != EM_POBS) && a.em.ignore_outliers;
    __syncthreads();

    for (int idx0 = (blockIdx.x * nsub + sub) * R; idx0 < a.ch.n; idx0 += gridDim.x * nsub * R) {
        if (j < R) {                                        // thread r describes chain r
            int* const d = cd + 8 * j;
            int c = -1, t0 = 0, tend = 0, T = 0, tstart = 0, mode = 0;
            long long row = 0;
            if (idx0 + j < a.ch.n) {
                c = a.ch.list ? a.ch.list[idx0 + j] : idx0 + j;
                t0 = a.ch.t0[c];
                T = a.ch.T[c];
                tend = t0 + a.ch.len[c];
                row = a.ch.row0[c] - t0;
                // mode 0: pi at frame 0, 1: uniform warm-up start, 2: exact vector (k_viterbi_chain32)
                if (t0 == 0) { tstart = 0; mode = 0; }
                else if (chain_exact_start(a.ch, c)) { tstart = t0 - 1; mode = 2; }
                else { tstart = max(0, t0 - (a.ch.warmv ? a.ch.warmv[c] : a.ch.warm)); mode = (tstart == 0) ? 0 : 1; }
            }
            d[C_C] = c; d[C_T0] = t0; d[C_TEND] = tend; d[C_T] = T; d[C_TSTART] = tstart;
            d[C_TFIRST] = (mode == 2) ? t0 : tstart; d[C_MODE] = mode;
            trow[j] = row;
        }
        for (int k = j; k < 2 * R * NPS; k += nthr) vb[k] = 0.0;
        sub_barrier(sub, sthr, nsub);
        int steps = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int* const d = cd + 8 * r;
            steps = max(steps, d[C_TEND] - d[C_TFIRST]);
            if (d[C_MODE] == 2 && jv) {
                const double x = chain_start_vec(a.ch, a.hand_end, d[C_C], d[C_C] - 1, N)[j];
                vb[r * NPS + j] = x;
                a.hand_used[(long long)d[C_C] * N + j] = x;
            }
        }
        sub_barrier(sub, sthr, nsub);
        auto em_raw = [&](int r, int t) -> double {
            if (!jv || t >= cd[8 * r + C_TEND]) return 0.0;
            const long long row = trow[r] + t;
            if (EM == EM_POBS) return a.em.pobs[row * N + j];
            if (EM == EM_GAUSS) return a.em.obs[row];
            return a.em.Bt[(long long)a.em.sym[row] * N + j];
        };
        double raw_next[R];
#pragma unroll
        for (int r = 0; r < R; ++r) raw_next[r] = em_raw(r, cd[8 * r + C_TFIRST]);
        for (int s = 0; s < steps; ++s) {
            double p[R], vn[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int t = cd[8 * r + C_TFIRST] + s;
                const double raw = raw_next[r];
                raw_next[r] = em_raw(r, t + 1);
                p[r] = 0.0;
                if (jv && t < cd[8 * r + C_TEND]) p[r] = (EM == EM_GAUSS) ? gauss_pdf(raw, mu, sigma) : raw;
            }
            if (outl) {                                     // outputmodel.py:126-130, one vote per chain
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const unsigned nzw = __ballot_sync(FULL, p[r] != 0.0);
                    if (lane == 0) anynz[r * 4 + wid] = nzw != 0u;
                }
                sub_barrier(sub, sthr, nsub);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    int any = 0;
                    for (int w2 = 0; w2 < nwarp; ++w2) any |= anynz[r * 4 + w2];
                    if (!any) p[r] = (jv && cd[8 * r + C_TFIRST] + s < cd[8 * r + C_TEND]) ? 1.0 : 0.0;
                }
            }
            // the scan of every chain, also of one at its start frame (whose result is not used): best and second-best
            // candidate, the first maximum with strict '>' (_hidden.c:186-200)
            double m[R], m2[R];
            int bi[R];
#pragma unroll
            for (int r = 0; r < R; ++r) { m[r] = __dmul_rn(vb[r * NPS], As[j]); m2[r] = -1.0; bi[r] = 0; }
            {   // N > 32: state 1 alone, then two predecessors per step from one 16-byte broadcast load (k_viterbi_multi)
                const double a1 = As[NPS + j];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const double h = __dmul_rn(vb[r * NPS + 1], a1);
                    if (h > m[r]) { m2[r] = m[r]; m[r] = h; bi[r] = 1; }
                    else if (h > m2[r]) m2[r] = h;
                }
            }
            int i = 2;
#pragma unroll 2
            for (; i + 1 < N; i += 2) {
                const double a0 = As[i * NPS + j], a1 = As[(i + 1) * NPS + j];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const double2 v2 = *reinterpret_cast<const double2*>(vb + r * NPS + i);
                    const double h0 = __dmul_rn(v2.x, a0), h1 = __dmul_rn(v2.y, a1);
                    if (h0 > m[r]) { m2[r] = m[r]; m[r] = h0; bi[r] = i; }
                    else if (h0 > m2[r]) m2[r] = h0;
                    if (h1 > m[r]) { m2[r] = m[r]; m[r] = h1; bi[r] = i + 1; }
                    else if (h1 > m2[r]) m2[r] = h1;
                }
            }
            if (i < N) {
                const double a0 = As[i * NPS + j];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const double h = __dmul_rn(vb[r * NPS + i], a0);
                    if (h > m[r]) { m2[r] = m[r]; m[r] = h; bi[r] = i; }
                    else if (h > m2[r]) m2[r] = h;
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int t = cd[8 * r + C_TFIRST] + s;
                const bool act = t < cd[8 * r + C_TEND], first = act && t == cd[8 * r + C_TSTART] && cd[8 * r + C_MODE] != 2;
                const bool near = jv && m[r] > 0.0 && (m[r] - fmax(m2[r], 0.0)) < a.margin_min * m[r];
                const unsigned word = __ballot_sync(FULL, near);
                if (first) {
                    vn[r] = (cd[8 * r + C_MODE] == 0) ? __dmul_rn(p[r], pi_j) : p[r];
                } else {
                    if (act && t >= cd[8 * r + C_T0]) {
                        if (jv) bp[(trow[r] + t - 1) * N + j] = (unsigned char)bi[r];
                        if (lane == 0 && wid < NW) a.flagmap[(trow[r] + t - 1) * NW + wid] = word;
                    }
                    vn[r] = __dmul_rn(__dmul_rn(p[r], vb[r * NPS + bi[r]]), As[bi[r] * NPS + j]);   // _hidden.c:247-250
                }
            }
            // (ub's readers -- the sums of the previous frame -- finished before that frame's third barrier)
            if (j < NPS) {
#pragma unroll
                for (int r = 0; r < R; ++r) ub[r * NPS + j] = (jv && cd[8 * r + C_TFIRST] + s < cd[8 * r + C_TEND]) ? vn[r] : 0.0;
            }
            sub_barrier(sub, sthr, nsub);
            {   // j-sequential sums (_hidden.c:254-259): warp w adds up the rows w, w + nwarp, ...
                constexpr int RW = (R + 1) / 2;             // rows per warp at two warps per group (the fewest)
                double sacc[RW];
#pragma unroll
                for (int q = 0; q < RW; ++q) sacc[q] = 0.0;
                for (int i = 0; i < N; ++i) {
#pragma unroll
                    for (int q = 0; q < RW; ++q) {
                        const int r = wid + q * nwarp;
                        if (r < R) sacc[q] = __dadd_rn(sacc[q], ub[r * NPS + i]);
                    }
                }
                if (lane == 0) {
#pragma unroll
                    for (int q = 0; q < RW; ++q)
                        if (wid + q * nwarp < R) ssum[wid + q * nwarp] = sacc[q];
                }
            }
            sub_barrier(sub, sthr, nsub);
            if (j < NPS) {
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int t = cd[8 * r + C_TFIRST] + s;
                    if (t >= cd[8 * r + C_TEND]) continue;
                    const double x = jv ? __ddiv_rn(vn[r], ssum[r]) : 0.0;
                    vb[r * NPS + j] = x;
                    if (jv && t == cd[8 * r + C_T0] - 1) a.hand_used[(long long)cd[8 * r + C_C] * N + j] = x;
                    if (jv && t == cd[8 * r + C_TEND] - 1) a.hand_end[(long long)cd[8 * r + C_C] * N + j] = x;
                }
            }
            sub_barrier(sub, sthr, nsub);
        }
        // path[T-1] = first maximum of the last row (_hidden.c:268): the last row of the map holds it for every s'
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (cd[8 * r + C_C] < 0 || cd[8 * r + C_TEND] != cd[8 * r + C_T]) continue;
            int best = 0;
            double mm = vb[r * NPS], second = -1.0;
            for (int i = 1; i < N; ++i) {
                const double x = vb[r * NPS + i];
                if (x > mm) { second = mm; mm = x; best = i; }
                else if (x > second) second = x;
            }
            if (jv) bp[(trow[r] + cd[8 * r + C_T] - 1) * N + j] = (unsigned char)best;
            const bool near = mm > 0.0 && (mm - fmax(second, 0.0)) < a.margin_min * mm;
            if (j < NW) a.flagmap[(trow[r] + cd[8 * r + C_T] - 1) * NW + j] = near ? 0xffffffffu : 0u;
        }
        sub_barrier(sub, sthr, nsub);
    }
}

// On-path flags of the wide chunked Viterbi: row r holds NW words, bit b of word w for the decision "state at r given the
// state 32 w + b at r + 1"; the last row of a trajectory holds the final arg max (any bit).
__global__ void k_viterbi_path_flags_wide(const unsigned* __restrict__ flagmap, int NW, const int* __restrict__ path,
                                          const long long* __restrict__ offsets, int K, long long rows, int* counter)
{
    int hits = 0;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x) {
        const unsigned* w = flagmap + r * NW;
        unsigned any = 0u;
        for (int q = 0; q < NW; ++q) any |= w[q];
        if (any == 0u) continue;
        int lo = 0, hi = K;                                 // trajectory of row r: offsets[lo] <= r < offsets[lo + 1]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (offsets[mid] <= r) lo = mid; else hi = mid;
        }
        const bool last = (r == offsets[lo + 1] - 1);
        if (last || ((w[path[r + 1] >> 5] >> (path[r + 1] & 31)) & 1u)) ++hits;
    }
    if (hits) atomicAdd(counter, hits);
}

#ifndef PANEL_HOST_NO_LAUNCHERS
int panel_sms()
{
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    }
    return n;
}

// resident blocks per SM of the statistics kernel, the more register-hungry of the two (sizes one wave of chains)
int panel_blocks_per_sm()
{
    static int per = 0;
    if (per == 0) {
        int v = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_backward_stats_panel32<EM_GAUSS>, PW * 32, 0) != cudaSuccess
            || v <= 0) v = 2;
        per = v;
    }
    return per;
}

int panel_blocks(int n_chains)
{
    const long long groups = ((long long)n_chains + PW * PCH - 1) / (PW * PCH);
    const long long cap = (long long)panel_sms() * panel_blocks_per_sm();
    return (int)std::max(1LL, std::min(groups, cap));
}

// wide kernels: state tiles (= warps per block) for N, 0 if N is not served (N <= 16 belongs to the lane family)
int wide_tiles(int N) { return (N <= 16) ? 0 : (N <= 32 ? 4 : (N <= 64 ? 8 : (N <= 104 ? 13 : 0))); }

#define WIDE_DISPATCH(NTV, CALL4, CALL8, CALL13) \
    do { if ((NTV) == 4) { CALL4; } else if ((NTV) == 8) { CALL8; } else { CALL13; } } while (0)

// chain sets per block of the backward kernel at NT = 13 (128 registers per thread: two sets spill 200-300 bytes per thread,
// and with 165 KB of the L1 carved out as shared memory the spills go to L2 -- measured: long-scoreboard stalls, no gain)
#ifndef BWS13
#define BWS13 1
#endif
// chains per block: the two-set kernels (wide2) serve NT >= 8, the one-set kernels NT = 4
int wide_cpb(int NT) { return NT >= 8 ? WS * PCH : PCH; }

// dynamic shared memory above 48 KB is an opt-in per kernel; set on every launch (a few microseconds: a cache keyed on the
// function-pointer TYPE -- the first version -- is shared by all instantiations and left most kernels without the attribute)
template <typename K>
int wide2_prepare(K kernel, size_t smem)
{
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        bhmm_set_error(BHMM_ERR_CUDA, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed for a wide2 kernel");
        return BHMM_ERR_CUDA;
    }
    return BHMM_OK;
}

int wide_blocks_per_sm(int NT)
{
    static int per[17] = {0};
    if (per[NT] == 0) {
        int v = 0;
        cudaError_t e = cudaErrorUnknown;
        if (NT == 4) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_backward_stats_wide<EM_GAUSS, 4>, 4 * 32, 0);
        else if (NT == 8) {
            if (wide2_prepare(k_backward_stats_wide2<EM_GAUSS, 8, true, false, 2>, wide2_backward_smem<8, true, false, 2>()) == BHMM_OK)
                e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_backward_stats_wide2<EM_GAUSS, 8, true, false, 2>, 8 * 32,
                                                                  wide2_backward_smem<8, true, false, 2>());
        } else {
            if (wide2_prepare(k_backward_stats_wide2<EM_GAUSS, 13, true, true, BWS13>, wide2_backward_smem<13, true, true, BWS13>()) == BHMM_OK)
                e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, k_backward_stats_wide2<EM_GAUSS, 13, true, true, BWS13>, 13 * 32,
                                                                  wide2_backward_smem<13, true, true, BWS13>());
        }
        per[NT] = (e == cudaSuccess && v > 0) ? v : 1;
    }
    return per[NT];
}

// chains per block and round of the backward + statistics kernel (its grid is the number of rows of partial statistics)
int wide_cpb_bwd(int NT) { return NT > 8 ? BWS13 * PCH : wide_cpb(NT); }

int wide_blocks_bwd(int NT, int n_chains)
{
    const int cpb = wide_cpb_bwd(NT);
    const long long groups = ((long long)n_chains + cpb - 1) / cpb;
    const long long cap = (long long)panel_sms() * wide_blocks_per_sm(NT);
    return (int)std::max(1LL, std::min(groups, cap));
}

int wide_blocks(int NT, int n_chains)
{
    const int cpb = wide_cpb(NT);
    const long long groups = ((long long)n_chains + cpb - 1) / cpb;
    const long long cap = (long long)panel_sms() * wide_blocks_per_sm(NT);
    return (int)std::max(1LL, std::min(groups, cap));
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <int EM, int NT, bool OUTL>
int launch_forward_wide2(const FwdArgs& a, int grid, cudaStream_t st)
{
    constexpr size_t smem = wide2_forward_smem<NT, OUTL>();
    { const int rc_ = wide2_prepare(k_forward_wide2<EM, NT, OUTL>, smem); if (rc_ != BHMM_OK) return rc_; }
    k_forward_wide2<EM, NT, OUTL><<<grid, NT * 32, smem, st>>>(a);
    return BHMM_OK;
}

template <int EM>
int launch_forward_wide_em(const FwdArgs& a, int NT, cudaStream_t st)
{
    const int grid = wide_blocks(NT, a.ch.n);
    if (NT == 4) { k_forward_wide<EM, 4><<<grid, 4 * 32, 0, st>>>(a); return BHMM_OK; }
    const bool outl = (EM != EM_POBS) && a.em.ignore_outliers;
    if (NT == 8) return outl ? launch_forward_wide2<EM, 8, EM != EM_POBS>(a, grid, st) : launch_forward_wide2<EM, 8, false>(a, grid, st);
    return outl ? launch_forward_wide2<EM, 13, EM != EM_POBS>(a, grid, st) : launch_forward_wide2<EM, 13, false>(a, grid, st);
}

template <int EM, int NT, bool OUTL>
int launch_backward_wide2(const BwdArgs& a, cudaStream_t st)
{
    constexpr bool BSM = NT > 8;                            // NT = 13: B fragments + xi accumulators exceed 128 registers
    constexpr int BWS = NT > 8 ? BWS13 : 2;
    constexpr size_t smem = wide2_backward_smem<NT, OUTL, BSM, BWS>();
    { const int rc_ = wide2_prepare(k_backward_stats_wide2<EM, NT, OUTL, BSM, BWS>, smem); if (rc_ != BHMM_OK) return rc_; }
    k_backward_stats_wide2<EM, NT, OUTL, BSM, BWS><<<a.grid, NT * 32, smem, st>>>(a);
    return BHMM_OK;
}

template <int EM>
int launch_backward_wide_em(const BwdArgs& a, int NT, cudaStream_t st)
{
    if (NT == 4) { k_backward_stats_wide<EM, 4><<<a.grid, 4 * 32, 0, st>>>(a); return BHMM_OK; }
    const bool outl = (EM != EM_POBS) && a.em.ignore_outliers;
    if (NT == 8) return outl ? launch_backward_wide2<EM, 8, EM != EM_POBS>(a, st) : launch_backward_wide2<EM, 8, false>(a, st);
    return outl ? launch_backward_wide2<EM, 13, EM != EM_POBS>(a, st) : launch_backward_wide2<EM, 13, false>(a, st);
}
#endif   // PANEL_HOST_NO_LAUNCHERS

}  // namespace

#ifndef PANEL_HOST_NO_LAUNCHERS
// BHMM_B200_PANEL: 0 = off (team kernels); unset / 1 (the default since the family's first B200 runs in round 2: parity,
// memcheck and racecheck green, gpurun_out/c2_*.log) = N = 32 on the one-warp-per-8-chains kernels, 17 <= N <= 104 otherwise on the wide
// kernels; 2 = N = 32 on the wide kernels too (4 warps per 8 chains: a third of the registers, more resident warps)
static int panel_mode()
{
    static int mode = -1;
    if (mode < 0) {
        const char* e = getenv("BHMM_B200_PANEL");
        mode = (e && strcmp(e, "0") == 0) ? 0 : ((e && strcmp(e, "2") == 0) ? 2 : 1);
    }
    return mode;
}
static bool use_panel32(int N) { return N == PN && panel_mode() == 1; }

bool panel_enabled(int N) { return panel_mode() > 0 && wide_tiles(N) > 0; }

// threads per block and chains per row of partial statistics (N = 32: a row per warp; wide: a row per block)
void panel_shape(int N, int* threads, int* chains_per_row)
{
    *threads = use_panel32(N) ? PW * 32 : wide_tiles(N) * 32;
    *chains_per_row = use_panel32(N) ? PCH : wide_cpb(wide_tiles(N));
}

int panel_stats_rows(int N, int n_chains)
{
    return use_panel32(N) ? panel_blocks(n_chains) * PW : wide_blocks_bwd(wide_tiles(N), n_chains);
}

// Viterbi with the matrix column in registers: 32 < N <= 104 (N <= 32 keeps the packed one-warp teams)
bool panel_viterbi_ok(int N) { return panel_mode() > 0 && N > 32 && N <= 104; }

#ifndef VITERBI_MULTI_R
#define VITERBI_MULTI_R 4
#endif

template <int EM>
static int launch_viterbi_regs_em(const VitArgs& a, cudaStream_t st)
{
    if (a.K <= 0) return BHMM_OK;
    static int use_regs = -1;                               // BHMM_B200_VITERBI_REGS=1: the register kernel (comparison)
    if (use_regs < 0) { const char* e = getenv("BHMM_B200_VITERBI_REGS"); use_regs = (e && e[0] == '1') ? 1 : 0; }
    if (!use_regs) {
        constexpr int R = VITERBI_MULTI_R;
        const int sthr = a.N <= 64 ? 64 : 128;              // threads of a group: one per state
#ifdef PANEL_HOST_EMU
        const int nsub = 1;
#else
        const long long groups_all = ((long long)a.K + R - 1) / R;
        const int nsub = (int)std::max<long long>(1, std::min<long long>(512 / sthr, (groups_all + panel_sms() - 1) / panel_sms()));
#endif
        const int NPS = (a.N + 1) & ~1;
        const size_t smem = sizeof(double) * ((size_t)a.N * NPS + (size_t)nsub * (2 * (size_t)R * NPS + R + 2 * R));
        if (cudaFuncSetAttribute(k_viterbi_multi<EM, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            bhmm_set_error(BHMM_ERR_CUDA, "cudaFuncSetAttribute failed for k_viterbi_multi");
            return BHMM_ERR_CUDA;
        }
        int per = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_viterbi_multi<EM, R>, nsub * sthr, smem) != cudaSuccess || per <= 0) per = 1;
        const long long groups = ((long long)a.K + (long long)R * nsub - 1) / ((long long)R * nsub);
        k_viterbi_multi<EM, R><<<(int)std::min<long long>(groups, (long long)panel_sms() * per), nsub * sthr, smem, st>>>(a, NPS, sthr);
        return BHMM_OK;
    }
    int per = 0;
    if (a.N <= 64) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_viterbi_regs<EM, 64>, 64, 0) != cudaSuccess || per <= 0) per = 1;
        k_viterbi_regs<EM, 64><<<(int)std::min<long long>(a.K, (long long)panel_sms() * per), 64, 0, st>>>(a);
    } else {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_viterbi_regs<EM, 104>, 128, 0) != cudaSuccess || per <= 0) per = 1;
        k_viterbi_regs<EM, 104><<<(int)std::min<long long>(a.K, (long long)panel_sms() * per), 128, 0, st>>>(a);
    }
    return BHMM_OK;
}

int launch_viterbi_panel(const VitArgs& a, int em, cudaStream_t st)
{
    switch (em) {
        case EM_POBS: return launch_viterbi_regs_em<EM_POBS>(a, st);
        case EM_GAUSS: return launch_viterbi_regs_em<EM_GAUSS>(a, st);
        case EM_DISC: return launch_viterbi_regs_em<EM_DISC>(a, st);
    }
    return BHMM_ERR_INVALID;
}

bool panel_viterbi_chain_ok(int N) { return panel_mode() > 0 && N >= 1 && N <= 32; }

int launch_viterbi_chain(const VitChainArgs& a, int em, cudaStream_t st)
{
    if (a.N < 1 || a.N > 32) return BHMM_ERR_UNSUPPORTED;
    if (a.ch.n <= 0) return BHMM_OK;
    if (lane_viterbi_ok(a.N)) return launch_viterbi_chain_lane(a, em, st);      // N <= 16: one thread per chain (lane_viterbi.cu)
    const int grid = (int)std::max(1LL, std::min<long long>(((long long)a.ch.n + PW - 1) / PW, (long long)panel_sms() * 4));
    switch (em) {
        case EM_POBS: k_viterbi_chain32<EM_POBS><<<grid, PW * 32, 0, st>>>(a); return BHMM_OK;
        case EM_GAUSS: k_viterbi_chain32<EM_GAUSS><<<grid, PW * 32, 0, st>>>(a); return BHMM_OK;
        case EM_DISC: k_viterbi_chain32<EM_DISC><<<grid, PW * 32, 0, st>>>(a); return BHMM_OK;
    }
    return BHMM_ERR_INVALID;
}

int launch_viterbi_path_flags(const unsigned* flagmap, const int* path, const long long* offsets, int K, long long rows,
                              int* counter, cudaStream_t st)
{
    if (rows <= 0) return BHMM_OK;
    const int grid = (int)std::max(1LL, std::min<long long>((rows + 255) / 256, (long long)panel_sms() * 8));
    k_viterbi_path_flags<<<grid, 256, 0, st>>>(flagmap, path, offsets, K, rows, counter);
    return BHMM_OK;
}

bool panel_viterbi_chain_wide_ok(int N) { return panel_mode() > 0 && N > 32 && N <= 128; }

#ifndef VITERBI_CHAIN_WIDE_R
#define VITERBI_CHAIN_WIDE_R 4
#endif

namespace {
// k_viterbi_chain_wide's shape for N: threads per group (one per state), padded stride, groups per block, dynamic shared memory
struct ChainWideShape { int sthr, NPS, nsub; size_t smem; };
ChainWideShape chain_wide_shape(int N, int nsub)
{
    constexpr int R = VITERBI_CHAIN_WIDE_R;
    ChainWideShape s;
    s.sthr = N <= 64 ? 64 : 128;
    s.NPS = (N + 1) & ~1;
    s.nsub = nsub;
    s.smem = sizeof(double) * ((size_t)N * s.NPS + (size_t)nsub * chain_wide_group_doubles(s.NPS, R));
    return s;
}

template <int EM>
int chain_wide_blocks_per_sm(const ChainWideShape& s, int* per)
{
    constexpr int R = VITERBI_CHAIN_WIDE_R;
    if (cudaFuncSetAttribute(k_viterbi_chain_wide<EM, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s.smem) != cudaSuccess) {
        bhmm_set_error(BHMM_ERR_CUDA, "cudaFuncSetAttribute failed for k_viterbi_chain_wide");
        return BHMM_ERR_CUDA;
    }
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(per, k_viterbi_chain_wide<EM, R>, s.nsub * s.sthr, s.smem) != cudaSuccess
        || *per <= 0)
        *per = 1;
    return BHMM_OK;
}

template <int EM>
int launch_viterbi_chain_wide_em(const VitChainArgs& a, cudaStream_t st)
{
    constexpr int R = VITERBI_CHAIN_WIDE_R;
    const long long groups = ((long long)a.ch.n + R - 1) / R;
#ifdef PANEL_HOST_EMU
    const int nsub = 1;                                     // the emulated build runs one group per block
#else
    const int sthr = a.N <= 64 ? 64 : 128;
    const int nsub = (int)std::max<long long>(1, std::min<long long>(512 / sthr, (groups + panel_sms() - 1) / panel_sms()));
#endif
    const ChainWideShape s = chain_wide_shape(a.N, nsub);
    int per = 1;
    { const int rc_ = chain_wide_blocks_per_sm<EM>(s, &per); if (rc_ != BHMM_OK) return rc_; }
    const long long blocks = (groups + nsub - 1) / nsub;
    k_viterbi_chain_wide<EM, R><<<(int)std::min<long long>(blocks, (long long)panel_sms() * per), nsub * s.sthr, s.smem, st>>>(
        a, s.NPS, s.sthr);
    return BHMM_OK;
}
}  // namespace

int viterbi_chain_wide_wave(int N)
{
    if (!panel_viterbi_chain_wide_ok(N)) return 0;
    const ChainWideShape s = chain_wide_shape(N, N <= 64 ? 8 : 4);
    int per = 1;
    if (chain_wide_blocks_per_sm<EM_GAUSS>(s, &per) != BHMM_OK) { bhmm_set_error(BHMM_OK, ""); per = 1; }
    return panel_sms() * per * s.nsub * VITERBI_CHAIN_WIDE_R;
}

int launch_viterbi_chain_wide(const VitChainArgs& a, int em, cudaStream_t st)
{
    if (a.N <= 32 || a.N > 128) return BHMM_ERR_UNSUPPORTED;
    if (a.ch.n <= 0) return BHMM_OK;
    switch (em) {
        case EM_POBS: return launch_viterbi_chain_wide_em<EM_POBS>(a, st);
        case EM_GAUSS: return launch_viterbi_chain_wide_em<EM_GAUSS>(a, st);
        case EM_DISC: return launch_viterbi_chain_wide_em<EM_DISC>(a, st);
    }
    return BHMM_ERR_INVALID;
}

int launch_viterbi_path_flags_wide(const unsigned* flagmap, int NW, const int* path, const long long* offsets, int K,
                                   long long rows, int* counter, cudaStream_t st)
{
    if (rows <= 0) return BHMM_OK;
    const int grid = (int)std::max(1LL, std::min<long long>((rows + 255) / 256, (long long)panel_sms() * 8));
    k_viterbi_path_flags_wide<<<grid, 256, 0, st>>>(flagmap, NW, path, offsets, K, rows, counter);
    return BHMM_OK;
}

bool panel_forward_ok(const FwdArgs& a, int em)
{
    if (!use_panel32(a.N)) return wide_tiles(a.N) > 0;     // the wide kernels use scalar global accesses only
    bool ok = aligned16(a.A) && aligned16(a.pi) && aligned16(a.hand_end) && aligned16(a.hand_used) && (!a.alpha || aligned16(a.alpha));
    if (em == EM_POBS) ok = ok && aligned16(a.em.pobs);
    if (em == EM_DISC) ok = ok && aligned16(a.em.Bt);
    return ok;
}

bool panel_backward_ok(const BwdArgs& a, int em)
{
    if (!use_panel32(a.N)) return wide_tiles(a.N) > 0 && a.grid > 0;
    bool ok = aligned16(a.A) && aligned16(a.alpha) && aligned16(a.partials) && aligned16(a.hand_end) && aligned16(a.hand_used)
              && (!a.gamma || aligned16(a.gamma)) && a.grid > 0 && a.grid % PW == 0;
    if (em == EM_POBS) ok = ok && aligned16(a.em.pobs);
    if (em == EM_DISC) ok = ok && aligned16(a.em.Bt);
    return ok;
}

int launch_forward_panel(const FwdArgs& a, int em, cudaStream_t st)
{
    if (a.ch.n <= 0) return BHMM_OK;
    if (!use_panel32(a.N)) {
        const int NT = wide_tiles(a.N);
        if (NT == 0) return BHMM_ERR_UNSUPPORTED;
        switch (em) {
            case EM_POBS: return launch_forward_wide_em<EM_POBS>(a, NT, st);
            case EM_GAUSS: return launch_forward_wide_em<EM_GAUSS>(a, NT, st);
            case EM_DISC: return launch_forward_wide_em<EM_DISC>(a, NT, st);
        }
        return BHMM_ERR_INVALID;
    }
    const int grid = panel_blocks(a.ch.n);
    switch (em) {
        case EM_POBS: k_forward_panel32<EM_POBS><<<grid, PW * 32, 0, st>>>(a); return BHMM_OK;
        case EM_GAUSS: k_forward_panel32<EM_GAUSS><<<grid, PW * 32, 0, st>>>(a); return BHMM_OK;
        case EM_DISC: k_forward_panel32<EM_DISC><<<grid, PW * 32, 0, st>>>(a); return BHMM_OK;
    }
    return BHMM_ERR_INVALID;
}

// a.grid = rows of `partials` (panel_stats_rows): warps of the launch at N = 32, blocks for the wide kernels; every
// row is written, chains or not
int launch_backward_stats_panel(const BwdArgs& a, int em, cudaStream_t st)
{
    if (!use_panel32(a.N)) {
        const int NT = wide_tiles(a.N);
        if (NT == 0) return BHMM_ERR_UNSUPPORTED;
        switch (em) {
            case EM_POBS: return launch_backward_wide_em<EM_POBS>(a, NT, st);
            case EM_GAUSS: return launch_backward_wide_em<EM_GAUSS>(a, NT, st);
            case EM_DISC: return launch_backward_wide_em<EM_DISC>(a, NT, st);
        }
        return BHMM_ERR_INVALID;
    }
    const int grid = a.grid / PW;
    switch (em) {
        case EM_POBS: k_backward_stats_panel32<EM_POBS><<<grid, PW * 32, 0, st>>>(a); return BHMM_OK;
        case EM_GAUSS: k_backward_stats_panel32<EM_GAUSS><<<grid, PW * 32, 0, st>>>(a); return BHMM_OK;
        case EM_DISC: k_backward_stats_panel32<EM_DISC><<<grid, PW * 32, 0, st>>>(a); return BHMM_OK;
    }
    return BHMM_ERR_INVALID;
}
#endif   // PANEL_HOST_NO_LAUNCHERS
