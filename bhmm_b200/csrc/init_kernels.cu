// bhmm_b200/csrc/init_kernels.cu -- the per-frame statistics of the initial-model heuristics (api.init_gaussian_hmm,
// api.init_discrete_hmm) on device-resident trajectories:
//   k_init_subsample   the frames of the mixture fit: owned frames whose index g in the global concatenation of all
//                      trajectories satisfies g % s == 0 (init_gaussian_hmm's pooled[::s], any sharding);
//   k_gmm_pass/_final  one EM iteration of the 1-D Gaussian mixture on the sorted subsample (_gmm_1d);
//   k_init_counts      lag-`lag` pair counts of a frame -> state map, the first-frame histogram and, for the cluster-label
//                      map, the symbol histogram placed at (label(o), o).  Three maps: the Gaussian arg-max assignment,
//                      the symbol itself, and the symbol's cluster label.
// Every kernel covers the OWNED frames of its rows only (ShardRows: own_lo / own_hi per trajectory, NULL = whole
// trajectories; flags & SHARD_STARTS where local frame 0 is the trajectory's frame 0, NULL = everywhere), so the integer
// statistics of the shards of a data set add up to those of the whole.  Integer counters are exact (u64 atomics); the
// mixture's sums run in a fixed order with no floating-point atomics, so identical input gives identical bits on every run.
// The file holds its C ABI too: it can be linked on its own.
#include <cmath>

#include "host_common.h"

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int INIT_THREADS = 256;
constexpr size_t INIT_SMEM_CAP = 96 * 1024;     // privatised counters up to this size (opt-in above 48 KB)
constexpr int GMM_THREADS = 256;
constexpr int GMM_TILE = 256;                    // subsample frames per tile (one per thread in the log-sum-exp phase)
constexpr int GMM_MAX_BLOCKS = 256;              // fixed by n alone: the reduction order does not depend on the device
constexpr size_t GMM_SMEM_CAP = 200 * 1024;

enum { MAP_GAUSSIAN = 0, MAP_SYMBOL = 1, MAP_LABEL = 2 };

__device__ __forceinline__ int row_owner(const long long* __restrict__ offsets, int K, long long row)
{
    int lo = 0, hi = K;          // offsets[lo] <= row < offsets[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (offsets[mid] <= row) lo = mid; else hi = mid;
    }
    return lo;
}

// ------------------------------------------------------------------------------------------------ strided subsample
// out[j], j in [outoff[k], outoff[k+1]): the (j - outoff[k])-th owned frame of trajectory k whose global index is a
// multiple of s.  goff[k] is the global index of local frame 0.
__global__ void k_init_subsample(const double* __restrict__ obs, ShardRows sh, const long long* __restrict__ goff,
                                 const long long* __restrict__ outoff, long long s, long long n, double* __restrict__ out)
{
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int k = row_owner(outoff, sh.K, j);
    const long long glo = goff[k] + (sh.own_lo ? sh.own_lo[k] : 0);
    const long long g = ((glo + s - 1) / s) * s + (j - outoff[k]) * s;
    out[j] = obs[sh.offsets[k] + (g - goff[k])];
}

// ------------------------------------------------------------------------------------------------ 1-D mixture EM
// log p_k(x) exactly as _gmm_1d writes it: (log w_k - (0.5 z) z) - log s_k, z = (x - m_k) / s_k, no contraction
__device__ __forceinline__ double gmm_logp(double x, double lw, double m, double s, double ls)
{
    const double z = __ddiv_rn(__dsub_rn(x, m), s);
    return __dsub_rn(__dsub_rn(lw, __dmul_rn(__dmul_rn(0.5, z), z)), ls);
}

// PASS 0: per block [sum_x r_k (N) | sum_x r_k x (N) | sum_x lse]; PASS 1: per block sum_x r_k (x - mnew_k)^2 (N).  r_k is
// evaluated with the parameters P = [w | m | s] the iteration started from.  A tile of frames is loaded and its log-sum-exp
// formed one frame per thread; then slot q = g N + k (component k, residue class g of the tile's frames mod G) adds its
// frames in order.  The block's partial of component k is the sum over g in order.
template <int PASS>
__global__ void __launch_bounds__(GMM_THREADS) k_gmm_pass(const double* __restrict__ x, long long n, int N,
                                                          const double* __restrict__ P, const double* __restrict__ mnew,
                                                          double* __restrict__ part)
{
    extern __shared__ double sm[];
    double* lw = sm;
    double* ls = lw + N;
    double* mu = ls + N;
    double* sg = mu + N;
    double* mn = sg + N;
    double* xs = mn + N;
    double* lse = xs + GMM_TILE;
    double* acc = lse + GMM_TILE;
    const int tid = threadIdx.x;
    const int G = max(1, (int)blockDim.x / N), slots = G * N;
    for (int k = tid; k < N; k += blockDim.x) {
        lw[k] = log(P[k]);
        mu[k] = P[N + k];
        sg[k] = P[2 * N + k];
        ls[k] = log(P[2 * N + k]);
        mn[k] = PASS == 1 ? mnew[k] : 0.0;
    }
    for (int q = tid; q < 2 * slots; q += blockDim.x) acc[q] = 0.0;
    double llacc = 0.0;
    __syncthreads();
    for (long long t0 = (long long)blockIdx.x * GMM_TILE; t0 < n; t0 += (long long)gridDim.x * GMM_TILE) {
        const int cnt = (int)min((long long)GMM_TILE, n - t0);
        if (tid < cnt) {
            const double xv = x[t0 + tid];
            double mx = -INFINITY;
            for (int k = 0; k < N; ++k) mx = fmax(mx, gmm_logp(xv, lw[k], mu[k], sg[k], ls[k]));
            double se = 0.0;
            for (int k = 0; k < N; ++k) se += exp(gmm_logp(xv, lw[k], mu[k], sg[k], ls[k]) - mx);
            const double l = mx + log(se);
            xs[tid] = xv;
            lse[tid] = l;
            if (PASS == 0) llacc += l;
        }
        __syncthreads();
        for (int q = tid; q < slots; q += blockDim.x) {
            const int k = q % N, g = q / N;
            double a0 = acc[q], a1 = acc[slots + q];
            for (int e = g; e < cnt; e += G) {
                const double r = exp(gmm_logp(xs[e], lw[k], mu[k], sg[k], ls[k]) - lse[e]);
                if (PASS == 0) {
                    a0 += r;
                    a1 += r * xs[e];
                } else {
                    const double d = xs[e] - mn[k];
                    a0 += r * (d * d);
                }
            }
            acc[q] = a0;
            acc[slots + q] = a1;
        }
        __syncthreads();
    }
    const int W = PASS == 0 ? 2 * N + 1 : N;
    for (int k = tid; k < N; k += blockDim.x) {
        double s0 = 0.0, s1 = 0.0;
        for (int g = 0; g < G; ++g) {
            s0 += acc[g * N + k];
            s1 += acc[slots + g * N + k];
        }
        part[(long long)blockIdx.x * W + k] = s0;
        if (PASS == 0) part[(long long)blockIdx.x * W + N + k] = s1;
    }
    if (PASS == 0) {
        xs[tid] = llacc;                         // the tile buffer is free after the last tile's barrier
        __syncthreads();
        if (tid == 0) {
            double l = 0.0;
            for (int t = 0; t < (int)blockDim.x; ++t) l += xs[t];
            part[(long long)blockIdx.x * W + 2 * N] = l;
        }
    }
}

// PASS 0: nk = sum + 1e-300, weights = nk / n, means = sum r x / nk, *ll = sum lse (into wk = [w | m | nk]);
// PASS 1: sigmas = sqrt(max(sum r (x - m)^2 / nk, floor^2)), then P = [w | m | sigmas].  Block sums in block order.
template <int PASS>
__global__ void k_gmm_final(const double* __restrict__ part, int grid, int N, long long n, double floor, double* __restrict__ wk,
                            double* __restrict__ P, double* __restrict__ ll)
{
    const int W = PASS == 0 ? 2 * N + 1 : N;
    for (int k = threadIdx.x; k < N; k += blockDim.x) {
        double s0 = 0.0, s1 = 0.0;
        for (int b = 0; b < grid; ++b) {
            s0 += part[(long long)b * W + k];
            if (PASS == 0) s1 += part[(long long)b * W + N + k];
        }
        if (PASS == 0) {
            const double nk = s0 + 1e-300;
            wk[k] = nk / (double)n;
            wk[N + k] = s1 / nk;
            wk[2 * N + k] = nk;
        } else {
            P[k] = wk[k];
            P[N + k] = wk[N + k];
            P[2 * N + k] = sqrt(fmax(s0 / wk[2 * N + k], floor * floor));
        }
    }
    if (PASS == 0 && threadIdx.x == 0) {
        double l = 0.0;
        for (int b = 0; b < grid; ++b) l += part[(long long)b * W + 2 * N];
        *ll = l;
    }
}

inline int gmm_grid(long long n) { return (int)max(1LL, min((long long)GMM_MAX_BLOCKS, (n + GMM_TILE - 1) / GMM_TILE)); }
inline size_t gmm_smem(int N)
{
    const int G = max(1, GMM_THREADS / N);
    return sizeof(double) * (5 * (size_t)N + 2 * GMM_TILE + 2 * (size_t)G * N);
}

// ------------------------------------------------------------------------------------------------ pair counts
struct InitArgs {
    ShardRows sh;                     // offsets, K, own_lo / own_hi (NULL: whole), flags (NULL: SHARD_STARTS everywhere)
    long long rows;
    int lag;
    int N;                            // hidden states (Gaussian, label)
    int M;                            // symbols (symbol, label)
    const double* obs;                // Gaussian observations
    const int* sym;                   // symbols
    const double* gp;                 // Gaussian [means | sigmas | log weights | log sigmas]
    const int* label;                 // cluster label of every symbol
    unsigned long long* out;          // [pairs (W W) | n0 (W)] (symbol map: pairs only), W = N or M
    unsigned long long* B;            // label map: (N, M) histogram
};

// first arg-max like np.argmax: the first maximum, a NaN before everything else
__device__ __forceinline__ int gauss_state(const double* __restrict__ gp, int N, double x)
{
    int best = 0;
    double bv = 0.0;
    bool nan = false;
    for (int k = 0; k < N; ++k) {
        const double z = __ddiv_rn(__dsub_rn(x, gp[k]), gp[N + k]);
        const double v = __dsub_rn(__dsub_rn(gp[2 * N + k], __dmul_rn(__dmul_rn(0.5, z), z)), gp[3 * N + k]);
        if (nan) continue;
        if (isnan(v)) { best = k; nan = true; }
        else if (k == 0 || v > bv) { best = k; bv = v; }
    }
    return best;
}

template <int MAP>
__device__ __forceinline__ int state_of(const InitArgs& a, long long r)
{
    if (MAP == MAP_GAUSSIAN) return gauss_state(a.gp, a.N, a.obs[r]);
    if (MAP == MAP_SYMBOL) return a.sym[r];
    return a.label[a.sym[r]];
}

// Warp-aggregated add: lanes holding the same key (ka, kb) as the lane before them join its run, and the run's first lane
// adds the run length at table[idx].  ka < 0: nothing to count.  Metastable data gives long runs of one pair.
__device__ __forceinline__ void warp_run_add(int ka, int kb, long long idx, unsigned long long* table, int lane)
{
    const int pa = __shfl_sync(FULL, ka, lane > 0 ? lane - 1 : 0);
    const int pb = __shfl_sync(FULL, kb, lane > 0 ? lane - 1 : 0);
    const bool head = lane == 0 || pa != ka || pb != kb;
    const unsigned heads = __ballot_sync(FULL, head);
    if (head && ka >= 0) {
        const unsigned above = lane == 31 ? 0u : heads & (FULL << (lane + 1));
        const int next = above ? __ffs(above) - 1 : 32;
        atomicAdd(table + idx, (unsigned long long)(next - lane));
    }
}

// One warp covers 32 consecutive rows per step (warp-uniform trip count, so the shuffles see every lane).  The state at
// t + lag comes from lane + lag of the same step when that lane exists, else it is evaluated again.  SMEM: block-private
// counters in shared memory, added to the outputs once per block.
template <int MAP, bool SMEM>
__global__ void __launch_bounds__(INIT_THREADS) k_init_counts(InitArgs a)
{
    extern __shared__ unsigned long long smc[];
    const int W = MAP == MAP_SYMBOL ? a.M : a.N;
    const long long WW = (long long)W * W;
    const long long ntab = WW + (MAP == MAP_SYMBOL ? 0 : W) + (MAP == MAP_LABEL ? a.M : 0);
    unsigned long long* tC = SMEM ? smc : a.out;
    unsigned long long* t0 = tC + WW;
    unsigned long long* tH = SMEM ? t0 + W : a.B;
    if (SMEM) {
        for (long long q = threadIdx.x; q < ntab; q += blockDim.x) smc[q] = 0ULL;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwr = ((long long)gridDim.x * blockDim.x) & ~31LL;
    for (long long base = wid * 32; base < a.rows; base += nwr) {
        const long long r = base + lane;
        int f = -1, tr = 0;
        long long t = 0, len = 0;
        bool own = false;
        if (r < a.rows) {
            tr = row_owner(a.sh.offsets, a.sh.K, r);
            t = r - a.sh.offsets[tr];
            len = a.sh.offsets[tr + 1] - a.sh.offsets[tr];
            own = a.sh.own_lo ? (t >= a.sh.own_lo[tr] && t < a.sh.own_hi[tr]) : true;
            f = state_of<MAP>(a, r);
        }
        const bool near = a.lag < 32 - lane;
        const int fsh = __shfl_sync(FULL, f, near ? lane + a.lag : lane);
        const bool pair = own && t + a.lag < len;
        int fb = -1;
        if (pair) fb = near ? fsh : state_of<MAP>(a, r + a.lag);
        warp_run_add(pair ? f : -1, fb, pair ? (long long)f * W + fb : 0, tC, lane);
        if (MAP != MAP_SYMBOL && own && t == 0 && (!a.sh.flags || (a.sh.flags[tr] & SHARD_STARTS)))
            atomicAdd(t0 + f, 1ULL);
        if (MAP == MAP_LABEL) {
            const int o = own ? a.sym[r] : -1;
            const long long idx = o < 0 ? 0 : (SMEM ? (long long)o : (long long)a.label[o] * a.M + o);
            warp_run_add(o, 0, idx, tH, lane);
        }
    }
    if (SMEM) {
        __syncthreads();
        for (long long q = threadIdx.x; q < WW + (MAP == MAP_SYMBOL ? 0 : W); q += blockDim.x)
            if (smc[q]) atomicAdd(a.out + q, smc[q]);
        if (MAP == MAP_LABEL)
            for (int o = threadIdx.x; o < a.M; o += blockDim.x)
                if (tH[o]) atomicAdd(a.B + (long long)a.label[o] * a.M + o, tH[o]);
    }
}

template <int MAP>
int launch_init_counts(const InitArgs& a, cudaStream_t st)
{
    if (a.rows <= 0) return BHMM_OK;
    const int W = MAP == MAP_SYMBOL ? a.M : a.N;
    const size_t tab = sizeof(unsigned long long) * ((size_t)W * W + (MAP == MAP_SYMBOL ? 0 : W) + (MAP == MAP_LABEL ? a.M : 0));
    const int blocks = (int)min((long long)148 * 8, (a.rows + INIT_THREADS - 1) / INIT_THREADS);
    if (tab <= INIT_SMEM_CAP) {
        if (tab > 48 * 1024)
            CUDA_TRY(cudaFuncSetAttribute(k_init_counts<MAP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tab));
        k_init_counts<MAP, true><<<blocks, INIT_THREADS, tab, st>>>(a);
    } else {
        k_init_counts<MAP, false><<<blocks, INIT_THREADS, 0, st>>>(a);
    }
    return BHMM_OK;
}

bool rows_ok(const long long* offsets, int K, long long rows, int lag)
{
    return offsets && K >= 1 && rows >= 0 && lag >= 1;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI (include/bhmm_b200.h, "initial-model statistics").  All pointers are device pointers.
extern "C" int bhmm_b200_init_subsample_dev(const double* d_obs, const long long* d_offsets, const long long* d_own_lo,
                                            const long long* d_own_hi, const long long* d_goff, const long long* d_outoff,
                                            int K, long long stride, long long n_out, double* d_out, void* stream)
{
    if (!d_obs || !d_offsets || !d_goff || !d_outoff || (n_out > 0 && !d_out) || K < 1 || stride < 1 || n_out < 0 ||
        (!d_own_lo) != (!d_own_hi)) {
        bhmm_set_error(BHMM_ERR_INVALID, "init_subsample: null pointer, K < 1, stride < 1 or n_out < 0");
        return BHMM_ERR_INVALID;
    }
    if (n_out == 0) return BHMM_OK;
    ShardRows sh{};
    sh.offsets = d_offsets;
    sh.K = K;
    sh.own_lo = d_own_lo;
    sh.own_hi = d_own_hi;
    k_init_subsample<<<(unsigned)((n_out + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_obs, sh, d_goff, d_outoff, stride,
                                                                                       n_out, d_out);
    LAUNCHED(1);
    CUDA_TRY(cudaGetLastError());
    return BHMM_OK;
}

extern "C" long long bhmm_b200_gmm_work_doubles(long long n, int N)
{
    if (n < 1 || N < 1) return 0;
    const long long g = gmm_grid(n);
    return g * (2LL * N + 1) + g * N + 3LL * N;
}

extern "C" int bhmm_b200_gmm_em_step_dev(const double* d_x, long long n, int N, double floor, double* d_params,
                                         double* d_work, double* d_ll, void* stream)
{
    if (!d_x || !d_params || !d_work || !d_ll || n < 1 || N < 1) {
        bhmm_set_error(BHMM_ERR_INVALID, "gmm_em_step: null pointer, n < 1 or N < 1");
        return BHMM_ERR_INVALID;
    }
    const size_t smem = gmm_smem(N);
    if (smem > GMM_SMEM_CAP) {
        bhmm_set_error(BHMM_ERR_UNSUPPORTED, "gmm_em_step: too many mixture components");
        return BHMM_ERR_UNSUPPORTED;
    }
    if (smem > 48 * 1024) {
        CUDA_TRY(cudaFuncSetAttribute(k_gmm_pass<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(k_gmm_pass<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    const int grid = gmm_grid(n);
    double* partA = d_work;
    double* partB = partA + (long long)grid * (2 * N + 1);
    double* wk = partB + (long long)grid * N;
    cudaStream_t st = (cudaStream_t)stream;
    k_gmm_pass<0><<<grid, GMM_THREADS, smem, st>>>(d_x, n, N, d_params, nullptr, partA);
    k_gmm_final<0><<<1, 256, 0, st>>>(partA, grid, N, n, floor, wk, d_params, d_ll);
    k_gmm_pass<1><<<grid, GMM_THREADS, smem, st>>>(d_x, n, N, d_params, wk + N, partB);
    k_gmm_final<1><<<1, 256, 0, st>>>(partB, grid, N, n, floor, wk, d_params, d_ll);
    LAUNCHED(4);
    CUDA_TRY(cudaGetLastError());
    return BHMM_OK;
}

static int init_counts(int map, const void* d_obs, const long long* d_offsets, const long long* d_own_lo,
                       const long long* d_own_hi, const int* d_flags, int K, long long rows, int lag, int N, int M,
                       const double* d_gauss, const int* d_label, long long* d_out, long long* d_B, void* stream)
{
    InitArgs a{};
    a.sh.offsets = d_offsets;
    a.sh.K = K;
    a.sh.own_lo = d_own_lo;
    a.sh.own_hi = d_own_hi;
    a.sh.flags = d_flags;
    a.rows = rows;
    a.lag = lag;
    a.N = N;
    a.M = M;
    a.obs = static_cast<const double*>(d_obs);
    a.sym = static_cast<const int*>(d_obs);
    a.gp = d_gauss;
    a.label = d_label;
    a.out = reinterpret_cast<unsigned long long*>(d_out);
    a.B = reinterpret_cast<unsigned long long*>(d_B);
    cudaStream_t st = (cudaStream_t)stream;
    if (map == MAP_GAUSSIAN) RC_TRY(launch_init_counts<MAP_GAUSSIAN>(a, st));
    else if (map == MAP_SYMBOL) RC_TRY(launch_init_counts<MAP_SYMBOL>(a, st));
    else RC_TRY(launch_init_counts<MAP_LABEL>(a, st));
    LAUNCHED(rows > 0 ? 1 : 0);
    CUDA_TRY(cudaGetLastError());
    return BHMM_OK;
}

extern "C" int bhmm_b200_init_counts_gaussian_dev(const double* d_obs, const long long* d_offsets, const long long* d_own_lo,
                                                  const long long* d_own_hi, const int* d_flags, int K, long long rows, int lag,
                                                  int N, const double* d_gauss, long long* d_out, void* stream)
{
    if (!d_obs || !rows_ok(d_offsets, K, rows, lag) || N < 1 || !d_gauss || !d_out || (!d_own_lo) != (!d_own_hi)) {
        bhmm_set_error(BHMM_ERR_INVALID, "init_counts_gaussian: null pointer, K < 1, N < 1 or lag < 1");
        return BHMM_ERR_INVALID;
    }
    return init_counts(MAP_GAUSSIAN, d_obs, d_offsets, d_own_lo, d_own_hi, d_flags, K, rows, lag, N, 0, d_gauss, nullptr, d_out,
                       nullptr, stream);
}

extern "C" int bhmm_b200_init_counts_symbols_dev(const int* d_sym, const long long* d_offsets, const long long* d_own_lo,
                                                 const long long* d_own_hi, int K, long long rows, int lag, int M,
                                                 long long* d_out, void* stream)
{
    if (!d_sym || !rows_ok(d_offsets, K, rows, lag) || M < 1 || !d_out || (!d_own_lo) != (!d_own_hi)) {
        bhmm_set_error(BHMM_ERR_INVALID, "init_counts_symbols: null pointer, K < 1, M < 1 or lag < 1");
        return BHMM_ERR_INVALID;
    }
    return init_counts(MAP_SYMBOL, d_sym, d_offsets, d_own_lo, d_own_hi, nullptr, K, rows, lag, 0, M, nullptr, nullptr, d_out,
                       nullptr, stream);
}

extern "C" int bhmm_b200_init_counts_labels_dev(const int* d_sym, const long long* d_offsets, const long long* d_own_lo,
                                                const long long* d_own_hi, const int* d_flags, int K, long long rows, int lag,
                                                int N, int M, const int* d_label, long long* d_out, long long* d_B,
                                                void* stream)
{
    if (!d_sym || !rows_ok(d_offsets, K, rows, lag) || N < 1 || M < 1 || !d_label || !d_out || !d_B ||
        (!d_own_lo) != (!d_own_hi)) {
        bhmm_set_error(BHMM_ERR_INVALID, "init_counts_labels: null pointer, K < 1, N < 1, M < 1 or lag < 1");
        return BHMM_ERR_INVALID;
    }
    return init_counts(MAP_LABEL, d_sym, d_offsets, d_own_lo, d_own_hi, d_flags, K, rows, lag, N, M, nullptr, d_label, d_out,
                       d_B, stream);
}
