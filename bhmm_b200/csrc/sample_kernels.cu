// bhmm_b200/csrc/sample_kernels.cu -- forward-filter / backward-sample, restructured to be parallel in time
// while staying bit-exact with the serial reference (_sample_path, _hidden.c:330-378).
//
// The reference draws s_{T-1} ~ alpha_{T-1}, then s_t given s_{t+1} with ONE uniform per frame.  Given the
// uniform u_t, the draw at frame t is a deterministic function  s_t = F_t(s_{t+1})  of the next state only:
// F_t(s') = first i with cumsum_i( alpha_t[i]*A[i][s'] / sum ) >= u_t   (_normalize :307-319, _random_choice
// :283-305).  So
//   1. k_sample_table   evaluates F_t(s') for every frame and every s' in parallel (N values per frame),
//                       using exactly the reference's operation order (__dmul_rn/__dadd_rn/__ddiv_rn);
//   2. the path is the composition of those maps, resolved segment-wise:
//        k_chase_map   per (segment, entering state) -> state at the segment's first frame,
//        k_chase_link  per trajectory, walks its segments from the last to the first,
//        k_chase_path  per segment, follows the maps from the now-known entering state and writes the path.
// Device Philox4x32-10 supplies the uniforms in production; an explicit uniform array reproduces the
// reference's glibc stream for parity.  The same Philox stream and link step also drive the forward simulation of
// synthetic trajectories (k_gen_*, k_emit_*: the generate_synthetic_* API).
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

namespace {

__device__ __forceinline__ void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0,
                                             uint32_t k1)
{
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}

// Philox4x32-10 block keyed by `seed`, counter (row, ctr): c = {row lo, row hi, ctr lo, ctr hi} on entry
__device__ __forceinline__ void philox_block(unsigned long long seed, unsigned long long ctr, long long row, uint32_t& c0,
                                             uint32_t& c1, uint32_t& c2, uint32_t& c3)
{
    c0 = (uint32_t)row; c1 = (uint32_t)((unsigned long long)row >> 32);
    c2 = (uint32_t)ctr; c3 = (uint32_t)(ctr >> 32);
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

// uniform in [0,1) from Philox4x32-10 keyed by `seed`, counter (ctr, row)
__device__ __forceinline__ double philox_uniform(unsigned long long seed, unsigned long long ctr, long long row)
{
    uint32_t c0, c1, c2, c3;
    philox_block(seed, ctr, row, c0, c1, c2, c3);
    const unsigned long long bits = ((unsigned long long)c0 << 32) | c1;
    return (double)(bits >> 11) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ int traj_of_row(const long long* __restrict__ offsets, int K, long long row)
{
    int lo = 0, hi = K;          // offsets[lo] <= row < offsets[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (offsets[mid] <= row) lo = mid; else hi = mid;
    }
    return lo;
}

// frame t of local trajectory k of a time shard: the owned range, the Philox row and whether the next frame exists
__device__ __forceinline__ bool shard_owned(const ShardRows& sh, int tr, long long t)
{
    return t >= sh.own_lo[tr] && t < sh.own_hi[tr];
}

// SHARD: a sampling batch of a time shard (ShardRows): only owned rows get a table, frame t of trajectory k draws the Philox
// row base[k] + t, and the last local row of a trajectory that continues past the shard is an ordinary row
template <bool PHILOX, bool SHARD>
__global__ void k_sample_table(const double* __restrict__ alpha, const double* __restrict__ A,
                               const double* __restrict__ u, unsigned long long seed, unsigned long long ctr,
                               const long long* __restrict__ offsets, int K, int N, long long rows,
                               unsigned char* __restrict__ F, int* __restrict__ err, ShardRows sh)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= rows * N) return;
    const long long row = k / N;
    const int sp = (int)(k - row * N);          // hypothetical state of the next frame
    const int tr = traj_of_row(offsets, K, row);
    bool last = (row + 1 == offsets[tr + 1]);
    long long prow = row;
    if (SHARD) {
        const long long t = row - offsets[tr];
        if (!shard_owned(sh, tr, t)) return;
        if (sh.flags[tr] & SHARD_CONTINUES) last = false;
        if (sh.base) prow = sh.base[tr] + t;
    }
    const double r = PHILOX ? philox_uniform(seed, ctr, prow) : u[row];
    const double* a = alpha + row * N;
    double s = 0.0;
    for (int i = 0; i < N; ++i) {
        const double pv = last ? a[i] : __dmul_rn(a[i], A[i * N + sp]);
        s = __dadd_rn(s, pv);
    }
    double acc = 0.0;
    int pick = -1;
    for (int i = 0; i < N; ++i) {
        const double pv = last ? a[i] : __dmul_rn(a[i], A[i * N + sp]);
        acc = __dadd_rn(acc, __ddiv_rn(pv, s));
        if (acc >= r) { pick = i; break; }
    }
    if (pick < 0) { pick = N - 1; atomicExch(err, BHMM_ERR_SAMPLE); }
    F[k] = (unsigned char)pick;
}

// segment tables: same layout as the chain table (row0, len, t0, T), ordered by (trajectory, t0)
__global__ void k_chase_map(const unsigned char* __restrict__ F, Chains seg, int N, unsigned char* __restrict__ map)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= (long long)seg.n * N) return;
    const int sidx = (int)(k / N);
    int s = (int)(k - (long long)sidx * N);
    const long long r0 = seg.row0[sidx];
    for (long long r = r0 + seg.len[sidx] - 1; r >= r0; --r) s = F[r * N + s];
    map[k] = (unsigned char)s;
}

// ENTER: the walk starts from the state handed in for the trajectory (time shards, ShardRows.enter; -1 = none) instead of 0
__device__ __forceinline__ int link_start(const ShardRows& sh, const Chains& seg, int sidx)
{
    const int e = sh.enter[traj_of_row(sh.offsets, sh.K, seg.row0[sidx])];
    return e >= 0 ? e : 0;
}

template <bool ENTER>
__global__ void k_chase_link(Chains seg, int N, const unsigned char* __restrict__ map, int* __restrict__ enter, ShardRows sh)
{
    const int sidx = blockIdx.x * blockDim.x + threadIdx.x;
    if (sidx >= seg.n) return;
    if (seg.t0[sidx] + seg.len[sidx] < seg.T[sidx]) return;   // only the last segment of a trajectory walks
    int s = ENTER ? link_start(sh, seg, sidx) : 0;            // F at the last frame ignores the entering state
    int cur = sidx;
    for (;;) {
        enter[cur] = s;
        s = map[(long long)cur * N + s];
        if (seg.t0[cur] == 0) break;
        --cur;
    }
}

// The same link step for batches with very many segments (one 1e9-frame trajectory has 3.9e6 of them: the walk above is
// that many DEPENDENT global loads, of the order of seconds).  One warp per trajectory end: the map rows of the next 32
// segments are contiguous, the warp copies them into shared memory with coalesced loads whose addresses do not depend on
// the walk, lane 0 walks the 32 rows there (one shared-memory round trip per segment), the lanes store the 32 entering
// states.  Chosen by the launchers when the batch has at least chase_tiled_threshold() segments.
template <bool ENTER>
__global__ void k_chase_link_tiled(Chains seg, int N, const unsigned char* __restrict__ map, int* __restrict__ enter,
                                   ShardRows sh)
{
    __shared__ unsigned char tile[32 * 256];
    __shared__ int states[32];
    const int lane = threadIdx.x;
    const int sidx = blockIdx.x * 32 + lane;
    const bool is_last = sidx < seg.n && (seg.t0[sidx] + seg.len[sidx] >= seg.T[sidx]);
    unsigned todo = __ballot_sync(0xffffffffu, is_last);
    while (todo) {
        const int l0 = __ffs(todo) - 1;
        todo &= todo - 1;
        int cur = blockIdx.x * 32 + l0;                       // the last segment of one trajectory
        int s = ENTER ? link_start(sh, seg, cur) : 0;         // F at the last frame ignores the entering state
        for (;;) {
            const int lo = max(cur - 31, 0);
            const int nrows = cur - lo + 1;
            for (int k = lane; k < nrows * N; k += 32) {      // tile row l = segment cur - l
                const int r = k / N, c = k - r * N;
                tile[(cur - lo - r) * N + c] = map[(long long)lo * N + k];
            }
            const int idx = cur - lane;
            const unsigned fm = __ballot_sync(0xffffffffu, idx >= 0 && seg.t0[idx] == 0);
            const int stop = fm ? (__ffs(fm) - 1) : 31;       // the trajectory's first segment, if it lies in this tile
            __syncwarp();
            if (lane == 0) {
                for (int l = 0; l <= stop; ++l) {
                    states[l] = s;
                    s = tile[l * N + s];
                }
            }
            __syncwarp();
            if (lane <= stop) enter[cur - lane] = states[lane];
            s = __shfl_sync(0xffffffffu, s, 0);
            if (fm) break;
            cur -= 32;
            __syncwarp();
        }
    }
}

__global__ void k_chase_path(const unsigned char* __restrict__ F, Chains seg, int N, const int* __restrict__ enter,
                             int* __restrict__ path)
{
    const int sidx = blockIdx.x * blockDim.x + threadIdx.x;
    if (sidx >= seg.n) return;
    int s = enter[sidx];
    const long long r0 = seg.row0[sidx];
    for (long long r = r0 + seg.len[sidx] - 1; r >= r0; --r) {
        s = F[r * N + s];
        path[r] = s;
    }
}

// One level of the whole-shard map reduction: output map g is the composition of the source maps [beg[g], beg[g] + len[g])
// -- consecutive segments of one trajectory in time order, so the state entering from the right goes through the last one
// first -- and len 0 is the identity (a trajectory with no owned frames passes the state through).
__global__ void k_compose_maps(const unsigned char* __restrict__ src, const long long* __restrict__ beg,
                               const int* __restrict__ len, int n, int N, unsigned char* __restrict__ dst)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= (long long)n * N) return;
    const int g = (int)(k / N);
    int s = (int)(k - (long long)g * N);
    const long long b = beg[g];
    for (int j = len[g] - 1; j >= 0; --j) s = src[(b + j) * N + s];
    dst[k] = (unsigned char)s;
}

// Gibbs path statistics (HMM.count_matrix / count_init / collect_observations_in_state,
// bhmm/hmm/generic_hmm.py:297-334,398-431): integer lag-1 transition counts, first-state histogram, frames per
// state, and sum(o), sum(o^2) per state.  Block-private shared-memory counters, then one global atomic each.
// SHARD: owned frames only; the first frame counts in n0 only where the local trajectory starts the global one
// (SHARD_STARTS), and the last owned frame of a trajectory that continues counts its transition into the handed-in state.
template <bool SHARD>
__global__ void k_path_stats(const int* __restrict__ path, const double* __restrict__ obs,
                             const long long* __restrict__ offsets, int K, int N, long long rows,
                             unsigned long long* __restrict__ Cint, unsigned long long* __restrict__ n0,
                             unsigned long long* __restrict__ cnt, double* __restrict__ so, double* __restrict__ soo,
                             int use_smem, ShardRows shr)
{
    extern __shared__ unsigned long long sh[];
    unsigned long long* sC = sh;                    // N*N
    unsigned long long* s0 = sC + N * N;            // N
    unsigned long long* sc = s0 + N;                // N
    double* sso = reinterpret_cast<double*>(sc + N);   // N
    double* ssoo = sso + N;                            // N
    if (use_smem) {
        for (int k = threadIdx.x; k < N * N + 2 * N; k += blockDim.x) sh[k] = 0ULL;
        for (int k = threadIdx.x; k < 2 * N; k += blockDim.x) sso[k] = 0.0;
        __syncthreads();
    }
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += stride) {
        const int tr = traj_of_row(offsets, K, r);
        bool first = (r == offsets[tr]);
        bool last = (r + 1 == offsets[tr + 1]);
        int next = -1;                                   // SHARD: the handed-in state after the last local frame
        if (SHARD) {
            if (!shard_owned(shr, tr, r - offsets[tr])) continue;
            first = first && (shr.flags[tr] & SHARD_STARTS);
            if (last && (shr.flags[tr] & SHARD_CONTINUES)) { last = false; next = shr.enter[tr]; }
        }
        const int s = path[r];
        const double o = obs ? obs[r] : 0.0;
        if (use_smem) {
            atomicAdd(sc + s, 1ULL);
            if (first) atomicAdd(s0 + s, 1ULL);
            if (!last) atomicAdd(sC + s * N + (next >= 0 ? next : path[r + 1]), 1ULL);
            if (obs) { atomicAdd(sso + s, o); atomicAdd(ssoo + s, o * o); }
        } else {
            atomicAdd(cnt + s, 1ULL);
            if (first) atomicAdd(n0 + s, 1ULL);
            if (!last) atomicAdd(Cint + (long long)s * N + (next >= 0 ? next : path[r + 1]), 1ULL);
            if (obs) { atomicAdd(so + s, o); atomicAdd(soo + s, o * o); }
        }
    }
    if (use_smem) {
        __syncthreads();
        for (int k = threadIdx.x; k < N * N; k += blockDim.x) if (sC[k]) atomicAdd(Cint + k, sC[k]);
        for (int k = threadIdx.x; k < N; k += blockDim.x) {
            if (s0[k]) atomicAdd(n0 + k, s0[k]);
            if (sc[k]) atomicAdd(cnt + k, sc[k]);
            if (obs) { atomicAdd(so + k, sso[k]); atomicAdd(soo + k, ssoo[k]); }
        }
    }
}

__global__ void k_symbol_histogram(const int* __restrict__ path, const int* __restrict__ sym, long long rows, int M,
                                   unsigned long long* __restrict__ hist)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    atomicAdd(hist + (long long)path[r] * M + sym[r], 1ULL);
}

// ---- synthetic trajectories: forward simulation of the hidden chain, parallel in time and exact
// Given the frame's uniform u_t = U(seed, 0, row), the state is a fixed function of the previous one,
//   s_t = G_t(s_{t-1}) = draw(cumA[s_{t-1}], u_t),   s_0 = draw(cum0, u_0) or the caller's start,
// so the chase above applies with time running forwards:
//   k_gen_map     per (segment, entering state) -> state at the segment's last frame, G_t evaluated on the fly;
//   link_segments per trajectory, on a segment table in REVERSED time order (t0 counted from the trajectory's end), so
//                 that its walk from the "last" segment down to the one with t0 == 0 goes from the first in time to the last;
//   k_gen_replay  per segment, from the now-known entering state, writes the states.
// Only comparisons of Philox uniforms with host-built cumulative tables are involved: every segmentation, and a single
// serial thread, give the same states bit for bit.

// smallest i with u < cum[i] (cum non-decreasing, cum[n-1] = 1 > u): never a zero-probability entry, even at u = 0
__device__ __forceinline__ int draw_cum(const double* cum, int n, double u)
{
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (u < cum[mid]) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// state at frame t of a trajectory from the previous state and the frame's uniform (start < 0: draw from cum0)
__device__ __forceinline__ int gen_step(const double* cum0, const double* cumA, int N, int t, int start, int prev, double u)
{
    if (t > 0) return draw_cum(cumA + prev * N, N, u);
    return start >= 0 ? start : draw_cum(cum0, N, u);
}

// first frame, within its trajectory, of segment sidx of the reversed table
__device__ __forceinline__ int gen_t0(const Chains& seg, int sidx) { return seg.T[sidx] - seg.t0[sidx] - seg.len[sidx]; }

// One warp per segment for N <= 32 (4 segments per block), a block of ceil(N/32) warps per segment above.  Lane j carries
// entering state j through the segment; lane l computes the uniform of the l-th frame of every 32 and the warp shares it.
template <bool SMEM>
__global__ void k_gen_map(Chains seg, int N, const double* __restrict__ cum0g, const double* __restrict__ cumAg,
                          const int* __restrict__ seg_start, unsigned long long seed, unsigned char* __restrict__ map)
{
    extern __shared__ double gen_sh[];
    const double* cum0 = cum0g;
    const double* cumA = cumAg;
    if (SMEM) {
        for (int k = threadIdx.x; k < N + N * N; k += blockDim.x) gen_sh[k] = k < N ? cum0g[k] : cumAg[k - N];
        __syncthreads();
        cum0 = gen_sh;
        cumA = gen_sh + N;
    }
    const int W = (N + 31) >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sidx = blockIdx.x * ((blockDim.x >> 5) / W) + warp / W;
    if (sidx >= seg.n) return;                                // whole warps leave together
    const int j = (warp % W) * 32 + lane;
    const long long r0 = seg.row0[sidx];
    const int len = seg.len[sidx], t0 = gen_t0(seg, sidx);
    const int start = seg_start ? seg_start[sidx] : -1;
    int s = j < N ? j : 0;                                    // the first segment of a trajectory ignores it (t == 0)
    for (int b = 0; b < len; b += 32) {
        const int nb = min(32, len - b);
        const double u = lane < nb ? philox_uniform(seed, 0ULL, r0 + b + lane) : 0.0;
        for (int i = 0; i < nb; ++i) s = gen_step(cum0, cumA, N, t0 + b + i, start, s, __shfl_sync(0xffffffffu, u, i));
    }
    if (j < N) map[(long long)sidx * N + j] = (unsigned char)s;
}

// one thread per segment; enter == NULL: every segment starts its trajectory (one segment per trajectory)
template <bool SMEM>
__global__ void k_gen_replay(Chains seg, int N, const double* __restrict__ cum0g, const double* __restrict__ cumAg,
                             const int* __restrict__ seg_start, unsigned long long seed, const int* __restrict__ enter,
                             int* __restrict__ states)
{
    extern __shared__ double gen_sh[];
    const double* cum0 = cum0g;
    const double* cumA = cumAg;
    if (SMEM) {
        for (int k = threadIdx.x; k < N + N * N; k += blockDim.x) gen_sh[k] = k < N ? cum0g[k] : cumAg[k - N];
        __syncthreads();
        cum0 = gen_sh;
        cumA = gen_sh + N;
    }
    const int sidx = blockIdx.x * blockDim.x + threadIdx.x;
    if (sidx >= seg.n) return;
    int s = enter ? enter[sidx] : 0;
    const long long r0 = seg.row0[sidx];
    const int len = seg.len[sidx], t0 = gen_t0(seg, sidx);
    const int start = seg_start ? seg_start[sidx] : -1;
    for (int i = 0; i < len; ++i) {
        s = gen_step(cum0, cumA, N, t0 + i, start, s, philox_uniform(seed, 0ULL, r0 + i));
        states[r0 + i] = s;
    }
}

#ifdef PANEL_HOST_EMU
// the CPU emulation (tests/emu) has no cospi; its Gaussian draws are compared with a tolerance
inline double cospi(double x) { return cos(3.14159265358979323846 * x); }
#endif

// Box-Muller on one Philox block (seed, 1, row): u1 in (0,1], u2 in [0,1); o = mu + sigma z without contraction
__global__ void k_emit_gaussian(const int* __restrict__ states, long long rows, int N, const double* __restrict__ mu,
                                const double* __restrict__ sigma, unsigned long long seed, double* __restrict__ obs,
                                int* __restrict__ err)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const int s = states[r];
    if (s < 0 || s >= N) { obs[r] = NAN; atomicExch(err, BHMM_ERR_INVALID); return; }
    uint32_t c0, c1, c2, c3;
    philox_block(seed, 1ULL, r, c0, c1, c2, c3);
    const double u1 = (double)(((((unsigned long long)c0 << 32) | c1) >> 11) + 1) * (1.0 / 9007199254740992.0);
    const double u2 = (double)((((unsigned long long)c2 << 32) | c3) >> 11) * (1.0 / 9007199254740992.0);
    const double z = __dmul_rn(sqrt(-2.0 * log(u1)), cospi(2.0 * u2));
    obs[r] = __dadd_rn(mu[s], __dmul_rn(sigma[s], z));
}

__global__ void k_emit_discrete(const int* __restrict__ states, long long rows, int N, int M,
                                const double* __restrict__ cumB, unsigned long long seed, int* __restrict__ obs,
                                int* __restrict__ err)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const int s = states[r];
    if (s < 0 || s >= N) { obs[r] = -1; atomicExch(err, BHMM_ERR_INVALID); return; }
    obs[r] = draw_cum(cumB + (long long)s * M, M, philox_uniform(seed, 1ULL, r));
}

inline unsigned nblk(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

}  // namespace

int launch_sample_table(const double* alpha, const double* A, const double* u, const long long* offsets, int K,
                        int N, long long rows, unsigned char* F, int* err, cudaStream_t st)
{
    if (N > 256) return BHMM_ERR_UNSUPPORTED;
    if (rows <= 0) return BHMM_OK;
    k_sample_table<false, false><<<nblk(rows * N, 256), 256, 0, st>>>(alpha, A, u, 0ULL, 0ULL, offsets, K, N, rows, F, err,
                                                                      ShardRows{});
    return BHMM_OK;
}

int launch_sample_table_philox(const double* alpha, const double* A, unsigned long long seed, unsigned long long ctr,
                               const long long* offsets, int K, int N, long long rows, unsigned char* F, int* err,
                               cudaStream_t st)
{
    if (N > 256) return BHMM_ERR_UNSUPPORTED;
    if (rows <= 0) return BHMM_OK;
    k_sample_table<true, false><<<nblk(rows * N, 256), 256, 0, st>>>(alpha, A, nullptr, seed, ctr, offsets, K, N, rows, F,
                                                                       err, ShardRows{});
    return BHMM_OK;
}

// segments from which the tiled link kernel is used: 65536 (16.8 M frames in the batch) unless BHMM_B200_CHASE_TILED says
// otherwise (the CPU emulation tests force it with 1)
static int chase_tiled_threshold()
{
    static int t = -1;
    if (t < 0) {
        const char* e = getenv("BHMM_B200_CHASE_TILED");
        t = (e && atoi(e) > 0) ? atoi(e) : (1 << 16);
    }
    return t;
}

static void link_segments(const Chains& seg, int N, const unsigned char* seg_map, int* seg_enter, cudaStream_t st)
{
    if (seg.n >= chase_tiled_threshold() && N <= 256) k_chase_link_tiled<false><<<nblk(seg.n, 32), 32, 0, st>>>(seg, N, seg_map, seg_enter, ShardRows{});
    else k_chase_link<false><<<nblk(seg.n, 128), 128, 0, st>>>(seg, N, seg_map, seg_enter, ShardRows{});
}

int launch_chase(const unsigned char* F, const Chains& seg, int N, unsigned char* seg_map, int* seg_enter, int* path,
                 cudaStream_t st)
{
    if (seg.n <= 0) return BHMM_OK;
    k_chase_map<<<nblk((long long)seg.n * N, 128), 128, 0, st>>>(F, seg, N, seg_map);
    link_segments(seg, N, seg_map, seg_enter, st);
    k_chase_path<<<nblk(seg.n, 128), 128, 0, st>>>(F, seg, N, seg_enter, path);
    return BHMM_OK;
}

int launch_chase_link(const Chains& seg, int N, const unsigned char* seg_map, int* seg_enter, cudaStream_t st)
{
    if (seg.n <= 0) return BHMM_OK;
    link_segments(seg, N, seg_map, seg_enter, st);
    return BHMM_OK;
}

template <bool SHARD>
static int path_stats(const int* path, const double* obs, const long long* offsets, int K, int N, long long rows,
                      long long* Cint, long long* n0, long long* cnt, double* so, double* soo, const ShardRows& sh,
                      cudaStream_t st)
{
    if (rows <= 0) return BHMM_OK;
    const int use_smem = (N <= 64) ? 1 : 0;
    const size_t smem = use_smem ? sizeof(unsigned long long) * ((size_t)N * N + 2 * N) + sizeof(double) * 2 * N : 0;
    const int blocks = (int)min((long long)148 * 8, (rows + 255) / 256);
    k_path_stats<SHARD><<<blocks, 256, smem, st>>>(path, obs, offsets, K, N, rows,
                                                   reinterpret_cast<unsigned long long*>(Cint),
                                                   reinterpret_cast<unsigned long long*>(n0),
                                                   reinterpret_cast<unsigned long long*>(cnt), so, soo, use_smem, sh);
    return BHMM_OK;
}

int launch_path_stats(const int* path, const double* obs, const long long* offsets, int K, int N, long long rows,
                      long long* Cint, long long* n0, long long* cnt, double* so, double* soo, cudaStream_t st)
{
    return path_stats<false>(path, obs, offsets, K, N, rows, Cint, n0, cnt, so, soo, ShardRows{}, st);
}

// ---- Gibbs sweep on a time shard (engine.cu: gibbs_shard)
int launch_sample_table_shard(const double* alpha, const double* A, const double* u, unsigned long long seed,
                              unsigned long long ctr, const long long* offsets, int K, int N, long long rows,
                              unsigned char* F, int* err, const ShardRows& sh, cudaStream_t st)
{
    if (N > 256) return BHMM_ERR_UNSUPPORTED;
    if (rows <= 0) return BHMM_OK;
    if (u) k_sample_table<false, true><<<nblk(rows * N, 256), 256, 0, st>>>(alpha, A, u, 0ULL, 0ULL, offsets, K, N, rows, F, err, sh);
    else k_sample_table<true, true><<<nblk(rows * N, 256), 256, 0, st>>>(alpha, A, nullptr, seed, ctr, offsets, K, N, rows, F, err, sh);
    return BHMM_OK;
}

int launch_chase_maps(const unsigned char* F, const Chains& seg, int N, unsigned char* seg_map, cudaStream_t st)
{
    if (seg.n <= 0) return BHMM_OK;
    k_chase_map<<<nblk((long long)seg.n * N, 128), 128, 0, st>>>(F, seg, N, seg_map);
    return BHMM_OK;
}

int launch_compose_maps(const unsigned char* src, const long long* beg, const int* len, int n, int N, unsigned char* dst,
                        cudaStream_t st)
{
    if (n <= 0) return BHMM_OK;
    k_compose_maps<<<nblk((long long)n * N, 128), 128, 0, st>>>(src, beg, len, n, N, dst);
    return BHMM_OK;
}

int launch_chase_resolve_shard(const unsigned char* F, const Chains& seg, int N, const unsigned char* seg_map, int* seg_enter,
                               int* path, const ShardRows& sh, cudaStream_t st)
{
    if (seg.n <= 0) return BHMM_OK;
    if (seg.n >= chase_tiled_threshold()) k_chase_link_tiled<true><<<nblk(seg.n, 32), 32, 0, st>>>(seg, N, seg_map, seg_enter, sh);
    else k_chase_link<true><<<nblk(seg.n, 128), 128, 0, st>>>(seg, N, seg_map, seg_enter, sh);
    k_chase_path<<<nblk(seg.n, 128), 128, 0, st>>>(F, seg, N, seg_enter, path);
    return BHMM_OK;
}

int launch_path_stats_shard(const int* path, const double* obs, const long long* offsets, int K, int N, long long rows,
                            long long* Cint, long long* n0, long long* cnt, double* so, double* soo, const ShardRows& sh,
                            cudaStream_t st)
{
    return path_stats<true>(path, obs, offsets, K, N, rows, Cint, n0, cnt, so, soo, sh, st);
}

int launch_symbol_histogram(const int* path, const int* sym, long long rows, int N, int M, long long* hist,
                            cudaStream_t st)
{
    (void)N;
    if (rows <= 0) return BHMM_OK;
    k_symbol_histogram<<<nblk(rows, 256), 256, 0, st>>>(path, sym, rows, M, reinterpret_cast<unsigned long long*>(hist));
    return BHMM_OK;
}

// cum0 + cumA in shared memory up to 100 KB (N <= 112), read through L1 above
static size_t gen_smem_bytes(int N)
{
    const size_t b = sizeof(double) * ((size_t)N * N + N);
    return b <= 100 * 1024 ? b : 0;
}

int launch_generate_states(const Chains& seg, int N, const double* cum0, const double* cumA, const int* seg_start,
                           unsigned long long seed, bool whole, unsigned char* seg_map, int* seg_enter, int* states,
                           cudaStream_t st)
{
    if (N > 256) return BHMM_ERR_UNSUPPORTED;
    if (seg.n <= 0) return BHMM_OK;
    const size_t smem = gen_smem_bytes(N);
    if (smem > 48 * 1024) {
        cudaFuncSetAttribute(k_gen_map<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_gen_replay<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    if (!whole) {
        const int W = (N + 31) / 32, spb = (W == 1) ? 4 : 1;    // segments per block
        if (smem) k_gen_map<true><<<nblk(seg.n, spb), 32 * W * spb, smem, st>>>(seg, N, cum0, cumA, seg_start, seed, seg_map);
        else k_gen_map<false><<<nblk(seg.n, spb), 32 * W * spb, 0, st>>>(seg, N, cum0, cumA, seg_start, seed, seg_map);
        link_segments(seg, N, seg_map, seg_enter, st);
    }
    const int* enter = whole ? nullptr : seg_enter;
    if (smem) k_gen_replay<true><<<nblk(seg.n, 128), 128, smem, st>>>(seg, N, cum0, cumA, seg_start, seed, enter, states);
    else k_gen_replay<false><<<nblk(seg.n, 128), 128, 0, st>>>(seg, N, cum0, cumA, seg_start, seed, enter, states);
    return BHMM_OK;
}

int launch_emit_gaussian(const int* states, long long rows, int N, const double* mu, const double* sigma,
                         unsigned long long seed, double* obs, int* err, cudaStream_t st)
{
    if (rows <= 0) return BHMM_OK;
    k_emit_gaussian<<<nblk(rows, 256), 256, 0, st>>>(states, rows, N, mu, sigma, seed, obs, err);
    return BHMM_OK;
}

int launch_emit_discrete(const int* states, long long rows, int N, int M, const double* cumB, unsigned long long seed,
                         int* obs, int* err, cudaStream_t st)
{
    if (rows <= 0) return BHMM_OK;
    k_emit_discrete<<<nblk(rows, 256), 256, 0, st>>>(states, rows, N, M, cumB, seed, obs, err);
    return BHMM_OK;
}
