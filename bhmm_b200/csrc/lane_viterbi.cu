// bhmm_b200/csrc/lane_viterbi.cu -- time-chunked Viterbi for N <= 16 with ONE THREAD PER CHAIN ("lane" Viterbi).
//
// Replaces _compute_viterbi (bhmm/hidden/impl_c/_hidden.c:203-281, argmax :186-200) for batches whose trajectories the plan
// cuts into chains, fused with the emission (_gaussian.c:45-70 / discrete.py:146-153 / outputmodel.py:119-131).
//
// k_viterbi_chain32 (panel_kernels.cu) gives a chain a whole warp, lane j = state j: at N = 10 two thirds of the lanes
// idle and every frame pays three warp barriers and a 32-long sequential sum (measured, round 2: 0.2 s for the Viterbi
// paths of C3's 1024 x 1e5 frames -- as long as 25 EM iterations).  Here a thread owns a chain: the normalised
// max-product vector lives in registers, the transition matrix is read from shared memory with broadcast loads, a warp
// advances 32 chains per instruction.  Arithmetic per frame is exactly the sequential kernel's (_hidden.c:229-265
// operation order: products v_i A_ij, first maximum with strict '>', vnext_j = (p_j v_best) A_best,j, j-sequential sum,
// true division), so with an exact start a chain reproduces the reference's back-pointers bit for bit.
//
// Chains that do not start their trajectory warm up on the frames before them and are certified / re-run like the
// forward filter's (run_chains_certified); every decision whose relative margin between best and second-best candidate
// is below margin_min sets its bit in `flagmap`, and the caller falls back to the sequential kernel when the resolved
// path went through such a decision (see k_viterbi_chain32 for the argument).  Output layout: the shifted back-pointer
// map of k_viterbi_team's CHASE mode (uint8), resolved by the k_chase_* kernels.
#include <algorithm>

#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int LV_THREADS = 64;

template <int N, int EM>
__global__ void __launch_bounds__(LV_THREADS) k_viterbi_chain_lane(const VitChainArgs a)
{
    __shared__ __align__(16) double As[N * N];
    __shared__ double pis[N], mus[N], sgs[N];
    for (int k = threadIdx.x; k < N * N; k += blockDim.x) As[k] = a.A[k];
    for (int k = threadIdx.x; k < N; k += blockDim.x) {
        pis[k] = a.pi[k];
        mus[k] = (EM == EM_GAUSS) ? a.em.mu[k] : 0.0;
        sgs[k] = (EM == EM_GAUSS) ? a.em.sigma[k] : 1.0;
    }
    __syncthreads();
    unsigned char* bp = reinterpret_cast<unsigned char*>(a.backptr);
    const bool outliers = (EM != EM_POBS) && a.em.ignore_outliers;

    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < a.ch.n; idx += gridDim.x * blockDim.x) {
        const int c = a.ch.list ? a.ch.list[idx] : idx;
        const int len = a.ch.len[c], t0 = a.ch.t0[c], T = a.ch.T[c];
        const long long trow = a.ch.row0[c] - t0;
        const int tend = t0 + len;
        int tstart = 0, mode = 0;                           // mode 0: pi at frame 0, 1: uniform warm-up start, 2: exact vector
        if (t0 == 0) { tstart = 0; mode = 0; }
        else if (chain_exact_start(a.ch, c)) { tstart = t0 - 1; mode = 2; }
        else { tstart = max(0, t0 - (a.ch.warmv ? a.ch.warmv[c] : a.ch.warm)); mode = (tstart == 0) ? 0 : 1; }
        double v[N];
#pragma unroll
        for (int j = 0; j < N; ++j) v[j] = 0.0;
        if (mode == 2) {
            const double* hv = chain_start_vec(a.ch, a.hand_end, c, c - 1, N);
#pragma unroll
            for (int j = 0; j < N; ++j) {
                v[j] = hv[j];
                a.hand_used[(long long)c * N + j] = v[j];
            }
        }
        const int tfirst = (mode == 2) ? t0 : tstart;
        for (int t = tfirst; t < tend; ++t) {
            const long long row = trow + t;
            // ---- emission of frame t
            double p[N];
            if (EM == EM_GAUSS) {
                const double o = a.em.obs[row];
#pragma unroll
                for (int j = 0; j < N; ++j) p[j] = gauss_pdf(o, mus[j], sgs[j]);
            } else if (EM == EM_POBS) {
#pragma unroll
                for (int j = 0; j < N; ++j) p[j] = a.em.pobs[row * N + j];
            } else {
                const double* src = a.em.Bt + (long long)a.em.sym[row] * N;
#pragma unroll
                for (int j = 0; j < N; ++j) p[j] = src[j];
            }
            if (outliers) {                                 // outputmodel.py:126-130
                bool nz = false;
#pragma unroll
                for (int j = 0; j < N; ++j) nz = nz || (p[j] != 0.0);
                if (!nz) {
#pragma unroll
                    for (int j = 0; j < N; ++j) p[j] = 1.0;
                }
            }
            double vn[N];
            if (t == tstart && mode != 2) {
#pragma unroll
                for (int j = 0; j < N; ++j) vn[j] = (mode == 0) ? __dmul_rn(p[j], pis[j]) : p[j];
            } else {
                unsigned near_bits = 0u;
                const bool emit = t >= t0;
#pragma unroll
                for (int j = 0; j < N; ++j) {
                    double vsel = v[0], asel = As[j];
                    double m = __dmul_rn(vsel, asel), m2 = -1.0;
                    int best = 0;
#pragma unroll
                    for (int i = 1; i < N; ++i) {
                        const double aij = As[i * N + j];
                        const double h = __dmul_rn(v[i], aij);
                        if (h > m) { m2 = m; m = h; best = i; vsel = v[i]; asel = aij; }      // first maximum, _hidden.c:186-200
                        else if (h > m2) m2 = h;
                    }
                    if (emit) {
                        bp[(row - 1) * N + j] = (unsigned char)best;
                        if (N > 1 && m > 0.0 && (m - fmax(m2, 0.0)) < a.margin_min * m) near_bits |= 1u << j;
                    }
                    vn[j] = __dmul_rn(__dmul_rn(p[j], vsel), asel);                           // _hidden.c:247-250
                }
                if (emit) a.flagmap[row - 1] = near_bits;
            }
            double ssum = 0.0;
#pragma unroll
            for (int j = 0; j < N; ++j) ssum = __dadd_rn(ssum, vn[j]);                        // j-sequential, _hidden.c:254-259
#pragma unroll
            for (int j = 0; j < N; ++j) v[j] = __ddiv_rn(vn[j], ssum);
            if (t == t0 - 1) {
#pragma unroll
                for (int j = 0; j < N; ++j) a.hand_used[(long long)c * N + j] = v[j];
            }
        }
#pragma unroll
        for (int j = 0; j < N; ++j) a.hand_end[(long long)c * N + j] = v[j];
        if (tend == T) {                                    // path[T-1] = first maximum of the last row (_hidden.c:268)
            int best = 0;
            double m = v[0], second = -1.0;
#pragma unroll
            for (int i = 1; i < N; ++i) {
                if (v[i] > m) { second = m; m = v[i]; best = i; }
                else if (v[i] > second) second = v[i];
            }
#pragma unroll
            for (int j = 0; j < N; ++j) bp[(trow + T - 1) * N + j] = (unsigned char)best;
            const bool near = m > 0.0 && N > 1 && (m - fmax(second, 0.0)) < a.margin_min * m;
            a.flagmap[trow + T - 1] = near ? 0xffffffffu : 0u;
        }
    }
}

template <int N>
int launch_n(const VitChainArgs& a, int em, cudaStream_t st)
{
    const int grid = std::max(1, (a.ch.n + LV_THREADS - 1) / LV_THREADS);
    switch (em) {
        case EM_POBS: k_viterbi_chain_lane<N, EM_POBS><<<grid, LV_THREADS, 0, st>>>(a); return BHMM_OK;
        case EM_GAUSS: k_viterbi_chain_lane<N, EM_GAUSS><<<grid, LV_THREADS, 0, st>>>(a); return BHMM_OK;
        case EM_DISC: k_viterbi_chain_lane<N, EM_DISC><<<grid, LV_THREADS, 0, st>>>(a); return BHMM_OK;
    }
    return BHMM_ERR_INVALID;
}

}  // namespace

bool lane_viterbi_ok(int N)
{
    static int off = -1;
    if (off < 0) {
        const char* e = getenv("BHMM_B200_LANE_VITERBI");
        off = (e && e[0] == '0') ? 1 : 0;
    }
    return !off && N >= 1 && N <= 16;
}

int launch_viterbi_chain_lane(const VitChainArgs& a, int em, cudaStream_t st)
{
    if (a.ch.n <= 0) return BHMM_OK;
    switch (a.N) {
#define CASE(NN) case NN: return launch_n<NN>(a, em, st);
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(11) CASE(12) CASE(13)
        CASE(14) CASE(15) CASE(16)
#undef CASE
    }
    return BHMM_ERR_UNSUPPORTED;
}
