// bhmm_b200/csrc/engine.cu -- C ABI, part 2: the batched, device-resident engine (bhmm_b200_batch_*).
//
// All trajectories of a data set are concatenated in device memory ("rows"); one call runs a whole E-step,
// Viterbi pass or Gibbs hidden-path sweep over every trajectory.  This replaces the per-trajectory Python loops
// of MaximumLikelihoodEstimator.fit (maximum_likelihood.py:383-385), compute_viterbi_paths (:332-352) and
// BayesianHMMSampler._updateHiddenStateTrajectories (bayesian_sampling.py:283-291).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "host_common.h"
#include "../../include/bhmm_b200.h"

struct bhmm_b200_batch {
    int K = 0, N = 0;
    long long rows = 0;
    std::vector<long long> offsets;
    int chunk = 0, warm_f = 0, warm_b = 0, warm_min = 32;
    int req_chunk = 0, req_warm = 0;   // what the caller asked for (0 = automatic); kept for re-planning
    // Viterbi on a time shard (owned ranges): phase 0 = map + path in one call, 1 = back-pointer map only, 2 = path only;
    // vit_end[k] >= 0: the state of trajectory k at its last local frame, handed over by the shard that owns the next frames
    int vit_phase = 0;
    bool vit_map_chunked = false;
    std::vector<int> vit_end;
    // Gibbs sweep on a time shard (gibbs_shard): phase 1 = forward, table and whole-shard maps, 2 = link, replay and
    // statistics; the segment table then covers the owned frames only (gibbs_seg)
    int gibbs_phase = 0;
    bool gibbs_seg = false, gibbs_mapped = false, gsh_ready = false;
    std::vector<long long> philox_base;      // per trajectory: Philox row of local frame 0 (empty: the batch row)
    std::vector<int> gibbs_flags, gibbs_enter;
    std::vector<unsigned char> shard_map;   // (K, N) whole-shard maps of the last phase 1
    std::vector<int> lev_n;                 // map composition: groups per level ...
    std::vector<size_t> lev_off;            // ... and where each level's (beg, len) table starts
    Arena gsh;                              // device: own ranges, Philox bases, flags, entering states, level tables, maps
    long long *d_own_lo = nullptr, *d_own_hi = nullptr, *d_base = nullptr, *d_beg = nullptr;
    int *d_flags = nullptr, *d_enter = nullptr, *d_len = nullptr;
    unsigned char* d_lev[2] = {nullptr, nullptr};
    bool lane = false;          // small-N fast path (lane_kernels.cuh) instead of the team family
    bool no_alpha = false;      // Viterbi-only batch: no (rows, N) forward variables in the workspace
    double* d_g0buf = nullptr;
    int partial_rows = 0;
    HostPlan plan, segplan;
    Arena arena;
    bool carved = false;
    char* cw_base = nullptr;    // where the chain work (tables, hand-over vectors) is carved
    // carved device pointers
    ChainWork w;
    Chains seg{};
    unsigned char* seg_map = nullptr;
    int* seg_enter = nullptr;
    long long* d_offsets = nullptr;
    double* d_A = nullptr;
    double* d_pi = nullptr;
    double* d_mu = nullptr;
    double* d_sigma = nullptr;
    double edge_f[2] = {0.0, 0.0}, edge_b[2] = {0.0, 0.0};   // adapt_warm state per direction: remembered need, age
    std::vector<long long> own_lo, own_hi;   // owned frame range per trajectory (empty: whole trajectories)
    double* d_alpha = nullptr;
    unsigned char* d_F = nullptr;
    double* d_partials = nullptr;
    int stats_grid = 0;
    int* d_err = nullptr;
    unsigned* d_vflag = nullptr;   // chunked Viterbi: near-tie flags per row of the back-pointer map
    Arena disc;                 // B staging + Bt for the discrete model (sized on first use)
    Arena scan;                 // transfer operators of the exact-scan fallback (scan_kernels.cu; allocated when first needed)
    // border starts of a time shard (bhmm_b200_batch_set_border_starts): per trajectory an exact alpha at own_lo - 1 and / or
    // beta at own_hi (host, K x N each), and their device tables for the E-step (chain -> row, rows)
    std::vector<double> bs_f, bs_b;
    std::vector<char> has_f, has_b;
    bool bst_ok = false;        // the device tables match the plan and the starts
    Arena bst;
    int *d_gidx_f = nullptr, *d_gidx_b = nullptr;
    double *d_gvec_f = nullptr, *d_gvec_b = nullptr;
    RunInfo info;
    // optional per-kernel timing (CUDA events on the launching stream)
    bool profile = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    double kernel_ms[4] = {0, 0, 0, 0};   // forward (incl. certification), backward+statistics kernel, whole call, unused
};

namespace {

constexpr int SEG_FRAMES = 256;   // frames per segment of the path chase

// the chain-parallel Viterbi of a time shard with 32 < N <= 128 (k_viterbi_chain_wide); whole-trajectory batches with N > 32
// keep the sequential kernels, chunked or not
bool vit_wide(const bhmm_b200_batch* b) { return !b->own_lo.empty() && panel_viterbi_chain_wide_ok(b->N); }

// words per row of the near-tie flag map: one for N <= 32, ceil(N / 32) for k_viterbi_chain_wide
int vflag_row_words(int N) { return N <= 32 ? 1 : (N + 31) / 32; }

size_t batch_layout(bhmm_b200_batch* b, char* base)
{
    const int N = b->N;
    const int n = b->plan.n, ns = b->segplan.n;
    Carver cv;
    const size_t o_offs = cv.add<long long>(b->K + 1);
    const size_t o_cw = cv.add<char>(chainwork_bytes(n, N));
    const size_t o_srow = cv.add<long long>(ns), o_slen = cv.add<int>(ns), o_st0 = cv.add<int>(ns), o_sT = cv.add<int>(ns);
    const size_t o_smap = cv.add<unsigned char>((size_t)std::max(ns, n) * N);   // also per-chain maps (lane sampler)
    const size_t o_sent = cv.add<int>(std::max(ns, n));
    const size_t o_A = cv.add<double>((size_t)N * N), o_pi = cv.add<double>(N), o_mu = cv.add<double>(N),
                 o_sg = cv.add<double>(N);
    b->stats_grid = backward_stats_grid(N, n);
    b->partial_rows = std::max(b->stats_grid, lane_blocks(n));
    const size_t o_part = cv.add<double>((size_t)b->partial_rows * ((size_t)N * N + 4 * N));
    const size_t o_g0 = cv.add<double>((size_t)n * N);
    const size_t o_err = cv.add<int>(4);
    // forward variables: row-major (rows,N), or interleaved [chain/32][frame][state/2][chain%32] double2 (lane family)
    size_t alpha_doubles = (size_t)b->rows * N;
    if (b->lane) alpha_doubles = std::max(alpha_doubles, (size_t)((n + 31) / 32) * b->chunk * ((N + 1) / 2) * 64);
    if (b->no_alpha) alpha_doubles = 32;      // Viterbi needs the observations, the back-pointer map and the path only
    const size_t o_alpha = cv.add<double>(alpha_doubles);
    const size_t o_F = cv.add<unsigned char>((size_t)b->rows * N * (N > 256 ? 2 : 1));
    size_t vflag_words = panel_viterbi_chain_ok(N) ? (size_t)b->rows : 1;
    if (vit_wide(b)) vflag_words = (size_t)b->rows * vflag_row_words(N);   // time shard, 32 < N <= 128: k_viterbi_chain_wide
    const size_t o_vflag = cv.add<unsigned>(vflag_words);
    if (base) {
        b->d_offsets = (long long*)(base + o_offs);
        b->w = ChainWork();
        // chain tables are uploaded by chainwork_setup into base + o_cw
        b->seg.row0 = (const long long*)(base + o_srow);
        b->seg.len = (const int*)(base + o_slen);
        b->seg.t0 = (const int*)(base + o_st0);
        b->seg.T = (const int*)(base + o_sT);
        b->seg.n = ns;
        b->seg_map = (unsigned char*)(base + o_smap);
        b->seg_enter = (int*)(base + o_sent);
        b->d_A = (double*)(base + o_A);
        b->d_pi = (double*)(base + o_pi);
        b->d_mu = (double*)(base + o_mu);
        b->d_sigma = (double*)(base + o_sg);
        b->d_partials = (double*)(base + o_part);
        b->d_g0buf = (double*)(base + o_g0);
        b->d_err = (int*)(base + o_err);
        b->d_alpha = (double*)(base + o_alpha);
        b->d_F = (unsigned char*)(base + o_F);
        b->d_vflag = (unsigned*)(base + o_vflag);
        b->cw_base = base + o_cw;
    }
    return cv.off + 256;
}

int batch_carve(bhmm_b200_batch* b, cudaStream_t st)
{
    if (b->carved) return BHMM_OK;
    const size_t need = batch_layout(b, nullptr);
    RC_TRY(b->arena.ensure(need));
    batch_layout(b, b->arena.base);
    RC_TRY(chainwork_setup(b->w, b->plan, b->N, b->warm_f, b->cw_base, st));
    const int ns = b->segplan.n;
    CUDA_TRY(cudaMemcpyAsync(b->d_offsets, b->offsets.data(), sizeof(long long) * (b->K + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync((void*)b->seg.row0, b->segplan.row0.data(), sizeof(long long) * ns, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync((void*)b->seg.len, b->segplan.len.data(), sizeof(int) * ns, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync((void*)b->seg.t0, b->segplan.t0.data(), sizeof(int) * ns, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync((void*)b->seg.T, b->segplan.T.data(), sizeof(int) * ns, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    b->carved = true;
    return BHMM_OK;
}

void batch_plan(bhmm_b200_batch* b, int chunk, int warm)
{
    b->req_chunk = chunk;
    b->req_warm = warm;
    const int w = warm > 0 ? warm : (b->lane ? auto_warm_lane(b->N) : auto_warm(b->N));
    b->chunk = chunk > 0 ? chunk : (b->lane ? auto_chunk_lane(b->rows, b->N, w) : auto_chunk(b->rows, b->N, w));
    if (chunk <= 0) {
        // the chain kernels run all chains in ONE wave of resident blocks: a few chains too many (every trajectory rounds
        // its chain count up) would double the kernel time, so lengthen the chunk until the count fits
        int sms = 148, dev = 0;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        int tthreads = 32, tcpb = 1;
        team_shape(b->N, &tthreads, &tcpb);
        long long cap = b->lane ? (long long)sms * lane_blocks_per_sm(b->N, EM_GAUSS) * lane_threads()
                                : (long long)backward_stats_grid(b->N, 1 << 28) * tcpb;
        if (b->no_alpha && vit_wide(b)) cap = viterbi_chain_wide_wave(b->N);   // a Viterbi-only shard runs that kernel only
        auto count = [&](long long c) {
            long long n = 0;
            for (int k = 0; k < b->K; ++k) {
                const long long own = b->own_lo.empty() ? b->offsets[k + 1] - b->offsets[k] : b->own_hi[k] - b->own_lo[k];
                n += (own + c - 1) / c;
            }
            return n;
        };
        if (b->lane) {
            for (int it = 0; it < 200; ++it) {
                if (count(b->chunk) <= cap || b->chunk >= (1 << 30)) break;
                b->chunk = (int)std::min<long long>((long long)b->chunk + std::max(1, b->chunk / 100), 1 << 30);
            }
        } else {
            // Persistent blocks walk their chain groups in rounds, and a round that is mostly empty costs as much as a full
            // one (C4 on one GPU, first B200 run of the wide kernels: groups of 1365 whole trajectories on a wave of 1184
            // chains took two rounds, 42 % of the machine idle).  Choose the number of rounds m and the chunk together:
            // the smallest chunk c with at most m x wave chains, cost m x (c + warm-up), cheapest m wins.
            long long maxT = 1;
            for (int k = 0; k < b->K; ++k) maxT = std::max(maxT, b->offsets[k + 1] - b->offsets[k]);
            const long long lo_c = std::max<long long>(64, 2LL * w);
            double best_cost = 1e300;
            long long best_c = std::max<long long>(maxT, 1);
            for (int m = 1; m <= 32; ++m) {
                if (count(maxT) > (long long)m * cap) continue;            // even whole trajectories do not fit m rounds
                long long lo = std::min(lo_c, maxT), hi = maxT;          // smallest c in [lo, hi] with count(c) <= m cap
                while (lo < hi) {
                    const long long mid = (lo + hi) / 2;
                    if (count(mid) <= (long long)m * cap) hi = mid; else lo = mid + 1;
                }
                const double cost = (double)m * ((double)lo + (lo < maxT ? (double)w : 0.0));
                if (cost < best_cost * 0.98) { best_cost = cost; best_c = lo; }   // more rounds only for a real gain
            }
            b->chunk = (int)std::min<long long>(best_c, 1 << 30);
        }
    }
    b->warm_f = b->warm_b = w;
    b->warm_min = warm > 0 ? warm : 32;       // an explicit warm-up length is a floor for the adaptation
    build_plan(b->offsets.data(), b->K, b->chunk, b->plan, b->own_lo.empty() ? nullptr : b->own_lo.data(),
               b->own_hi.empty() ? nullptr : b->own_hi.data());
    if (b->gibbs_seg) {
        // segments over the owned frames, with t0 and T counted from own_lo: the link kernels then see a trajectory that
        // starts at the first owned frame and ends at the last
        build_plan(b->offsets.data(), b->K, SEG_FRAMES, b->segplan, b->own_lo.data(), b->own_hi.data());
        for (int k = 0; k < b->K; ++k)
            for (int q = b->segplan.first_chain[k]; q >= 0 && q <= b->segplan.last_chain[k]; ++q) {
                b->segplan.t0[q] -= (int)b->own_lo[k];
                b->segplan.T[q] = (int)(b->own_hi[k] - b->own_lo[k]);
            }
    } else {
        build_plan(b->offsets.data(), b->K, SEG_FRAMES, b->segplan);
    }
    b->carved = false;
    b->gsh_ready = false;
    b->gibbs_mapped = false;
    b->bst_ok = false;
}

int upload_small(double* dst, const double* src, size_t n, cudaStream_t st)
{
    CUDA_TRY(cudaMemcpyAsync(dst, src, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    return BHMM_OK;
}

// Installs the exact-scan fallback (scan_kernels.cu) on the batch's chain work for the duration of a pass; the callback
// captures the caller's emission by reference, hence the guard that removes it again.
struct ScanGuard {
    bhmm_b200_batch* b;
    ScanGuard(bhmm_b200_batch* b_, const Emission& em, int emkind) : b(b_)
    {
        const int N = b->N;
        static int off = -1;                                // BHMM_B200_EXACT_SCAN=0: repair sweeps only (comparison, tests)
        if (off < 0) { const char* e = getenv("BHMM_B200_EXACT_SCAN"); off = (e && e[0] == '0') ? 1 : 0; }
        if (off || !exact_scan_ok(N) || !b->w.chunked) return;
        b->w.scan = [this, &em, emkind, N](int dir, cudaStream_t st) -> int {
            const size_t need = exact_scan_bytes(b->w.n_total, N);
            if (b->scan.ensure(need) != BHMM_OK) { bhmm_set_error(BHMM_ERR_NO_MEM, "exact scan: device memory for the chain operators"); return BHMM_ERR_NO_MEM; }
            Chains all = b->w.ch;
            return launch_exact_scan(all, b->w.n_total, em, emkind, b->d_A, N, dir, dir > 0 ? b->w.he_f : b->w.he_b,
                                     reinterpret_cast<double*>(b->scan.base), st);
        };
    }
    ~ScanGuard() { b->w.scan = nullptr; }
};

// The E-step's hand-overs are repaired only above the repair tolerance (default 1e-11: still an order below the 1e-10 parity
// bar, and the map is non-expansive), while the warm-up length keeps being steered to the certification tolerance (1e-13):
// in steady state the mismatch sits near 1e-14 and a hand-over that drifts to a few 1e-13 -- the mixing rate moves by a few
// per cent from one EM iteration to the next -- lengthens the next warm-up instead of costing a repair sweep as long as a
// whole kernel (forward) or a second backward pass, for which every other rank of the job would wait in the all-reduce.
// Viterbi and the Gibbs sweep keep the strict tolerance (their outputs are discrete decisions).
struct RepairTolGuard {
    ChainWork& w;
    explicit RepairTolGuard(ChainWork& w_) : w(w_) { w.repair_tol = g_repair_tol; }
    ~RepairTolGuard() { w.repair_tol = 0.0; }
};

void begin_info(bhmm_b200_batch* b)
{
    b->info = RunInfo();
    b->info.chains = b->plan.n;
    b->info.chunk = b->chunk;
    b->info.warm = b->warm_f;
}

int prepare_discrete(bhmm_b200_batch* b, const double* B, int M, Emission& em, cudaStream_t st)
{
    const int N = b->N;
    RC_TRY(b->disc.ensure(sizeof(double) * 2 * (size_t)N * M + 512));
    double* stage = (double*)b->disc.base;
    double* Bt = stage + (((size_t)N * M + 31) & ~(size_t)31);
    CUDA_TRY(cudaMemcpyAsync(stage, B, sizeof(double) * (size_t)N * M, cudaMemcpyHostToDevice, st));
    RC_TRY(launch_transpose(stage, N, M, Bt, st));
    LAUNCHED(1);
    em.Bt = Bt;
    em.M = M;
    return BHMM_OK;
}

bool border_starts_set(const bhmm_b200_batch* b)
{
    for (int k = 0; k < (int)b->has_f.size(); ++k)
        if (b->has_f[k] || b->has_b[k]) return true;
    return false;
}

// Per-chain start tables of a time shard's E-step (Chains.gidx / gvec).  The first owned chain of trajectory k starts its
// forward recursion from row k of gvec_f where a border start is set, the last owned chain its backward recursion from row k
// of gvec_b; without one, a chain whose owned range does not begin at the trajectory's start (forward) or end at its end
// (backward) is marked CHAIN_WARMS_UP: its neighbour in the chain table belongs to another trajectory, so it keeps its halo
// warm-up in the exact passes after the transfer-operator scan as well.  Every other chain: -1.
int border_setup(bhmm_b200_batch* b, cudaStream_t st)
{
    if (b->bst_ok) return BHMM_OK;
    const int K = b->K, N = b->N, n = b->w.n_total;
    const bool given = (int)b->has_f.size() == K;
    if (!given) {
        b->bs_f.assign((size_t)K * N, 0.0); b->bs_b.assign((size_t)K * N, 0.0);
    }
    std::vector<int> gf(std::max(n, 1), -1), gb(std::max(n, 1), -1);
    for (int k = 0; k < K; ++k) {
        const int cf = b->plan.first_chain[k], cl = b->plan.last_chain[k];
        if (cf < 0) continue;
        if (given && b->has_f[k]) gf[cf] = k;
        else if (b->plan.t0[cf] > 0) gf[cf] = CHAIN_WARMS_UP;
        if (given && b->has_b[k]) gb[cl] = k;
        else if (b->plan.t0[cl] + b->plan.len[cl] < b->plan.T[cl]) gb[cl] = CHAIN_WARMS_UP;
    }
    Carver cv;
    const size_t o_if = cv.add<int>(gf.size()), o_ib = cv.add<int>(gb.size());
    const size_t o_vf = cv.add<double>((size_t)K * N), o_vb = cv.add<double>((size_t)K * N);
    RC_TRY(b->bst.ensure(cv.off + 256));
    char* base = b->bst.base;
    b->d_gidx_f = (int*)(base + o_if); b->d_gidx_b = (int*)(base + o_ib);
    b->d_gvec_f = (double*)(base + o_vf); b->d_gvec_b = (double*)(base + o_vb);
    CUDA_TRY(cudaMemcpyAsync(b->d_gidx_f, gf.data(), sizeof(int) * gf.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b->d_gidx_b, gb.data(), sizeof(int) * gb.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b->d_gvec_f, b->bs_f.data(), sizeof(double) * K * N, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b->d_gvec_b, b->bs_b.data(), sizeof(double) * K * N, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));     // the host tables go out of scope
    b->bst_ok = true;
    return BHMM_OK;
}

// Hands the per-chain start tables of one direction to the chain launches of a pass; removed again at the end.
struct BorderGuard {
    ChainWork& w;
    bool on;
    explicit BorderGuard(ChainWork& w_, bool on_) : w(w_), on(on_) {}
    void use(const bhmm_b200_batch* b, int dir)
    {
        w.ch.gidx = (on && dir != 0) ? (dir > 0 ? b->d_gidx_f : b->d_gidx_b) : nullptr;
        w.ch.gvec = (on && dir != 0) ? (dir > 0 ? b->d_gvec_f : b->d_gvec_b) : nullptr;
    }
    ~BorderGuard() { w.ch.gidx = nullptr; w.ch.gvec = nullptr; }
};

// forward + (backward & statistics with whole-pass retry) + finalize
int estep_common(bhmm_b200_batch* b, Emission& em, int emkind, const double* A, const double* pi, const double* mu,
                 const double* sigma, double* d_gamma, double* d_stats, double* d_Bnum, cudaStream_t st)
{
    const int N = b->N;
    if (b->no_alpha) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "Viterbi-only batch: no forward variables"); return BHMM_ERR_UNSUPPORTED; }
    RC_TRY(upload_small(b->d_A, A, (size_t)N * N, st));
    RC_TRY(upload_small(b->d_pi, pi, N, st));
    b->w.ch.warm = b->warm_f;
    ScanGuard scan_guard(b, em, emkind);
    RepairTolGuard repair_guard(b->w);
    const bool borders = !b->own_lo.empty();
    if (borders) RC_TRY(border_setup(b, st));
    BorderGuard border_guard(b->w, borders);
    LaneArgs la{};
    LaneHostParams hp{A, pi, mu, sigma};
    if (b->lane) {
        la.obs = em.obs; la.sym = em.sym; la.Bt = em.Bt; la.M = em.M; la.ignore_outliers = em.ignore_outliers;
        la.alpha_il = b->d_alpha; la.Lmax = b->chunk; la.alpha_rm = nullptr;
        la.chain_ll = b->w.chain_ll; la.g0buf = b->d_g0buf; la.partials = b->d_partials;
        la.Bnum = d_Bnum; la.gamma = d_gamma;
    }
    // ---- the optimistic pass (OPT-IN, BHMM_B200_OPTIMISTIC=1): forward, backward + statistics and both certifications
    // enqueued back to back, ONE synchronisation at the end; any failure falls through to the step-by-step path below, which
    // redoes the E-step with repairs.  Measured (round 2): it saves 0.3 % at one GPU (8.270 vs 8.295 ms per iteration: the two
    // host round trips are cheap) and LOSES 15 % at 8 GPUs (10.5 vs 9.13 ms): a failed forward certification, ~1 % per pass and
    // rank, wastes the backward pass that was already enqueued and every other rank waits for the redo.  Off by default.
    static int optimistic = -1;
    if (optimistic < 0) { const char* e = getenv("BHMM_B200_OPTIMISTIC"); optimistic = (e && e[0] == '1') ? 1 : 0; }
    auto launch_fwd = [&](const Chains& ch, cudaStream_t s2) -> int {
        if (b->lane) {
            LaneArgs x = la;
            x.ch = ch; x.hand_used = b->w.hu_f; x.hand_end = b->w.he_f;
            return launch_lane(x, hp, N, emkind, LANE_FORWARD, s2);
        }
        FwdArgs a{};
        a.ch = ch; a.em = em; a.N = N; a.A = b->d_A; a.pi = b->d_pi; a.alpha = b->d_alpha;
        a.chain_ll = b->w.chain_ll; a.hand_used = b->w.hu_f; a.hand_end = b->w.he_f;
        return launch_forward_team(a, emkind, s2);
    };
    auto launch_bwd = [&](const Chains& ch, cudaStream_t s2) -> int {
        if (b->lane) {
            LaneArgs x = la;
            x.ch = ch; x.hand_used = b->w.hu_b; x.hand_end = b->w.he_b;
            return launch_lane(x, hp, N, emkind, LANE_BACKWARD_STATS, s2);
        }
        BwdArgs a{};
        a.ch = ch;
        a.em = em; a.N = N; a.grid = b->stats_grid; a.A = b->d_A;
        a.alpha = b->d_alpha; a.gamma = d_gamma; a.Bnum = d_Bnum; a.partials = b->d_partials;
        a.hand_used = b->w.hu_b; a.hand_end = b->w.he_b;
        return launch_backward_team(a, emkind, true, s2);
    };
    auto finalize = [&]() -> int {
        const int prow = b->lane ? lane_blocks(b->w.n_total) : b->stats_grid;
        RC_TRY(launch_finalize_stats(b->d_partials, prow, b->w.chain_ll, b->w.n_total, b->d_A, N, d_stats, st));
        LAUNCHED(1);
        if (b->lane) {
            RC_TRY(launch_add_gamma0(b->w.ch, b->w.n_total, N, b->d_g0buf, d_stats, st));
            LAUNCHED(1);
        }
        return BHMM_OK;
    };
    if (optimistic && b->w.chunked && !border_starts_set(b)) {
        Chains all = b->w.ch;
        all.list = nullptr; all.n = b->w.n_total; all.exact = 0; all.warmv = nullptr;
        b->w.need_f = b->w.need_b = 0.0;
        if (b->profile) cudaEventRecord(b->ev[0], st);
        all.warm = b->warm_f;
        RC_TRY(launch_fwd(all, st));
        LAUNCHED(1);
        RC_TRY(certify_async(b->w, N, +1, st));
        if (b->profile) { cudaEventRecord(b->ev[1], st); cudaEventRecord(b->ev[2], st); }
        if (d_Bnum) CUDA_TRY(cudaMemsetAsync(d_Bnum, 0, sizeof(double) * (size_t)N * em.M, st));
        all.warm = b->warm_b;
        RC_TRY(launch_bwd(all, st));
        LAUNCHED(1);
        if (b->profile) cudaEventRecord(b->ev[3], st);
        RC_TRY(certify_async(b->w, N, -1, st));
        RC_TRY(finalize());
        CUDA_TRY(cudaStreamSynchronize(st));
        double wf = 0.0, wb = 0.0;
        const long long ff = certify_collect(b->w, +1, &wf), fb = certify_collect(b->w, -1, &wb);
        if (ff == 0 && fb == 0) {
            b->info.worst_f = wf; b->info.worst_b = wb;
            b->warm_f = adapt_warm(b->warm_f, b->w.need_f, wf, false, b->warm_min, b->plan.maxT, b->edge_f);
            b->warm_b = adapt_warm(b->warm_b, b->w.need_b, wb, false, b->warm_min, b->plan.maxT, b->edge_b);
            b->info.warm = std::max(b->warm_f, b->warm_b);
            return BHMM_OK;
        }
        b->info.rerun += (double)b->w.n_total;               // the whole E-step is redone step by step
        b->w.ch.warm = b->warm_f;
    }

    if (b->profile) cudaEventRecord(b->ev[0], st);
    border_guard.use(b, +1);
    RC_TRY(run_chains_certified(b->w, N, +1, launch_fwd, b->info, st));
    border_guard.use(b, -1);
    if (b->profile) cudaEventRecord(b->ev[1], st);
    if (b->w.chunked) b->warm_f = adapt_warm(b->warm_f, b->w.need_f, b->info.worst_f, b->info.fix_f > 0, b->warm_min, b->plan.maxT, b->edge_f);

    b->w.need_b = 0.0;
    bool exact_bwd = false;
    for (int attempt = 0;; ++attempt) {
        Chains all = b->w.ch;
        all.list = nullptr; all.n = b->w.n_total; all.exact = exact_bwd ? 1 : 0; all.warm = b->warm_b; all.warmv = nullptr;
        if (d_Bnum) CUDA_TRY(cudaMemsetAsync(d_Bnum, 0, sizeof(double) * (size_t)N * em.M, st));
        if (b->profile) cudaEventRecord(b->ev[2], st);
        RC_TRY(launch_bwd(all, st));
        LAUNCHED(1);
        if (b->profile) cudaEventRecord(b->ev[3], st);
        if (!b->w.chunked) break;
        const long long nfail = certify_sync(b->w, N, -1, &b->info.worst_b, st, exact_bwd ? EXACT_SCAN_TOL : 0.0);
        if (nfail < 0) { bhmm_set_error(BHMM_ERR_CUDA, cudaGetErrorString(cudaGetLastError())); return BHMM_ERR_CUDA; }
        if (nfail == 0) { b->warm_b = adapt_warm(b->warm_b, b->w.need_b, b->info.worst_b, false, b->warm_min, b->plan.maxT, b->edge_b); break; }
        // statistics of a failed pass cannot be patched chain by chain: lengthen the warm-up (at least +32 frames, up to
        // the longest trajectory, which is an exact start) and redo the pass.
        // a warm-up as long as the longest trajectory starts every chain from an exact end -- except on a time shard, whose
        // local trajectories end in a halo: there the scan takes over
        const bool capped = b->warm_b >= b->plan.maxT;
        if (exact_bwd || (capped && (b->own_lo.empty() || !b->w.scan))) {
            char msg[160];
            snprintf(msg, sizeof(msg), "backward hand-overs not certified (%lld chains, worst mismatch %.3g%s)", nfail, b->info.worst_b,
                     exact_bwd ? ", after the exact scan" : "");
            bhmm_set_error(BHMM_ERR_NOT_CERTIFIED, msg);
            return BHMM_ERR_NOT_CERTIFIED;
        }
        b->info.fix_b += 1;
        b->info.rerun += (double)b->w.n_total;
        if ((attempt >= 1 || capped) && b->w.scan) {
            // a longer warm-up did not help either: the model does not forget.  Exact starts from the transfer-operator
            // scan (the hand-over vectors the failed pass left behind are exact at the trajectory ends), then the pass once more
            RC_TRY(b->w.scan(-1, st));
            LAUNCHED(2);
            b->w.scans += 1;
            exact_bwd = true;
            continue;
        }
        b->warm_b = adapt_warm(b->warm_b, b->w.need_b, b->info.worst_b, true, b->warm_min, b->plan.maxT, b->edge_b);
    }
    RC_TRY(finalize());
    b->info.warm = std::max(b->warm_f, b->warm_b);
    return BHMM_OK;
}

int finish_stream(cudaStream_t st)
{
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { bhmm_set_error(BHMM_ERR_CUDA, cudaGetErrorString(e)); return BHMM_ERR_CUDA; }
    return BHMM_OK;
}

void collect_times(bhmm_b200_batch* b)
{
    if (!b->profile) return;
    float f = 0.f, g = 0.f, t = 0.f;
    cudaEventElapsedTime(&f, b->ev[0], b->ev[1]);
    cudaEventElapsedTime(&g, b->ev[2], b->ev[3]);
    cudaEventElapsedTime(&t, b->ev[0], b->ev[3]);
    b->kernel_ms[0] = f; b->kernel_ms[1] = g; b->kernel_ms[2] = t;
}

int gibbs_common(bhmm_b200_batch* b, Emission& em, int emkind, const double* A, const double* pi, const double* mu,
                 const double* sigma, const double* d_u,
                 unsigned long long seed, unsigned long long sweep, int* d_path, long long* d_counts, double* d_sums,
                 double* loglik_host, cudaStream_t st)
{
    const int N = b->N;
    if (!b->own_lo.empty()) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "hidden-path sampling needs whole trajectories (batch has owned ranges)"); return BHMM_ERR_UNSUPPORTED; }
    if (b->no_alpha) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "Viterbi-only batch: no forward variables"); return BHMM_ERR_UNSUPPORTED; }
    if (N > 256) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "sampling supports N <= 256"); return BHMM_ERR_UNSUPPORTED; }
    RC_TRY(upload_small(b->d_A, A, (size_t)N * N, st));
    RC_TRY(upload_small(b->d_pi, pi, N, st));
    b->w.ch.warm = b->warm_f;
    ScanGuard scan_guard(b, em, emkind);
    if (b->lane) {
        // lane family: forward on the interleaved layout, then the two-pass hypothesis sampler (lane_kernels.cuh)
        LaneArgs la{};
        LaneHostParams hp{A, pi, mu, sigma};
        la.obs = em.obs; la.sym = em.sym; la.Bt = em.Bt; la.M = em.M; la.ignore_outliers = em.ignore_outliers;
        la.alpha_il = b->d_alpha; la.Lmax = b->chunk; la.chain_ll = b->w.chain_ll;
        la.hand_used = b->w.hu_f; la.hand_end = b->w.he_f;
        RC_TRY(run_chains_certified(b->w, N, +1, [&](const Chains& ch, cudaStream_t s2) {
            LaneArgs x = la;
            x.ch = ch;
            return launch_lane(x, hp, N, emkind, LANE_FORWARD, s2);
        }, b->info, st));
        if (b->w.chunked) b->warm_f = adapt_warm(b->warm_f, b->w.need_f, b->info.worst_f, b->info.fix_f > 0, b->warm_min, b->plan.maxT, b->edge_f);
        CUDA_TRY(cudaMemsetAsync(b->d_err, 0, sizeof(int), st));
        CUDA_TRY(cudaMemsetAsync(d_counts, 0, sizeof(long long) * ((size_t)N * N + 2 * N), st));
        Chains all = b->w.ch;
        all.list = nullptr; all.n = b->w.n_total; all.exact = 0;
        la.ch = all;
        la.u_row = d_u; la.seed = seed; la.sweep = sweep; la.path = d_path;
        la.smap = b->seg_map; la.enter = b->seg_enter; la.coal = b->w.fail_list;
        la.counts = d_counts; la.err = b->d_err; la.partials = d_sums ? b->d_partials : nullptr;
        RC_TRY(launch_lane(la, hp, N, emkind, LANE_SAMPLE_MAP, st));
        RC_TRY(launch_chase_link(all, N, b->seg_map, b->seg_enter, st));
        RC_TRY(launch_lane(la, hp, N, emkind, LANE_SAMPLE_FIX, st));
        LAUNCHED(3);
        if (d_sums) {
            RC_TRY(launch_lane_sum_moments(b->d_partials, 2 * lane_blocks(b->w.n_total), N, d_sums, st));
            LAUNCHED(1);
        }
    } else {
        RC_TRY(run_forward(b->w, em, emkind, N, b->d_A, b->d_pi, b->d_alpha, b->info, st));
        if (b->w.chunked) b->warm_f = adapt_warm(b->warm_f, b->w.need_f, b->info.worst_f, b->info.fix_f > 0, b->warm_min, b->plan.maxT, b->edge_f);
        CUDA_TRY(cudaMemsetAsync(b->d_err, 0, sizeof(int), st));
        if (d_u) RC_TRY(launch_sample_table(b->d_alpha, b->d_A, d_u, b->d_offsets, b->K, N, b->rows, b->d_F, b->d_err, st));
        else RC_TRY(launch_sample_table_philox(b->d_alpha, b->d_A, seed, sweep, b->d_offsets, b->K, N, b->rows, b->d_F, b->d_err, st));
        RC_TRY(launch_chase(b->d_F, b->seg, N, b->seg_map, b->seg_enter, d_path, st));
        LAUNCHED(4);
        CUDA_TRY(cudaMemsetAsync(d_counts, 0, sizeof(long long) * ((size_t)N * N + 2 * N), st));
        if (d_sums) CUDA_TRY(cudaMemsetAsync(d_sums, 0, sizeof(double) * 2 * N, st));
        RC_TRY(launch_path_stats(d_path, d_sums ? em.obs : nullptr, b->d_offsets, b->K, N, b->rows, d_counts,
                                 d_counts + (size_t)N * N, d_counts + (size_t)N * N + N, d_sums, d_sums ? d_sums + N : nullptr,
                                 st));
        LAUNCHED(1);
    }
    std::vector<double> ll(b->w.n_total);
    int err = 0;
    CUDA_TRY(cudaMemcpyAsync(ll.data(), b->w.chain_ll, sizeof(double) * b->w.n_total, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&err, b->d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
    RC_TRY(finish_stream(st));
    if (err) { bhmm_set_error(err, "sample_path: no state could be drawn"); return err; }
    double s = 0.0;
    for (double v : ll) s += v;
    if (loglik_host) *loglik_host = s;
    return BHMM_OK;
}

constexpr int COMPOSE_FAN_IN = 32;   // segment maps composed by one thread per level of the whole-shard map reduction

// Device tables of the sharded sweep: the level tables of the map composition are planned from the segment table once per
// plan.  Level 0 composes each trajectory's segment maps in groups of COMPOSE_FAN_IN, every further level the previous
// level's outputs, until one map per trajectory is left (a trajectory without segments gets the identity at level 0).
int gibbs_shard_setup(bhmm_b200_batch* b, cudaStream_t st)
{
    if (b->gsh_ready) return BHMM_OK;
    const int K = b->K, N = b->N;
    const HostPlan& sp = b->segplan;
    std::vector<long long> start(K), beg;
    std::vector<int> cnt(K), len;
    for (int k = 0; k < K; ++k) {
        start[k] = std::max(sp.first_chain[k], 0);
        cnt[k] = sp.first_chain[k] < 0 ? 0 : sp.last_chain[k] - sp.first_chain[k] + 1;
    }
    b->lev_n.clear(); b->lev_off.clear();
    size_t maxn = 1;
    for (;;) {
        b->lev_off.push_back(beg.size());
        long long o = 0;
        for (int k = 0; k < K; ++k) {
            const int ng = cnt[k] == 0 ? 1 : (cnt[k] + COMPOSE_FAN_IN - 1) / COMPOSE_FAN_IN;
            for (int g = 0; g < ng; ++g) {
                beg.push_back(start[k] + (long long)g * COMPOSE_FAN_IN);
                len.push_back(std::min(COMPOSE_FAN_IN, cnt[k] - g * COMPOSE_FAN_IN));
            }
            start[k] = o; cnt[k] = ng; o += ng;
        }
        b->lev_n.push_back((int)o);
        maxn = std::max(maxn, (size_t)o);
        if (o == K) break;                   // one map per trajectory
    }
    Carver cv;
    const size_t o_lo = cv.add<long long>(K), o_hi = cv.add<long long>(K), o_base = cv.add<long long>(K);
    const size_t o_fl = cv.add<int>(K), o_en = cv.add<int>(K);
    const size_t o_beg = cv.add<long long>(beg.size()), o_len = cv.add<int>(len.size());
    const size_t o_l0 = cv.add<unsigned char>(maxn * N), o_l1 = cv.add<unsigned char>(maxn * N);
    RC_TRY(b->gsh.ensure(cv.off + 256));
    char* base = b->gsh.base;
    b->d_own_lo = (long long*)(base + o_lo); b->d_own_hi = (long long*)(base + o_hi); b->d_base = (long long*)(base + o_base);
    b->d_flags = (int*)(base + o_fl); b->d_enter = (int*)(base + o_en);
    b->d_beg = (long long*)(base + o_beg); b->d_len = (int*)(base + o_len);
    b->d_lev[0] = (unsigned char*)(base + o_l0); b->d_lev[1] = (unsigned char*)(base + o_l1);
    CUDA_TRY(cudaMemcpyAsync(b->d_own_lo, b->own_lo.data(), sizeof(long long) * K, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b->d_own_hi, b->own_hi.data(), sizeof(long long) * K, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b->d_beg, beg.data(), sizeof(long long) * beg.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b->d_len, len.data(), sizeof(int) * len.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));     // the host tables go out of scope
    b->gsh_ready = true;
    return BHMM_OK;
}

ShardRows shard_rows(const bhmm_b200_batch* b)
{
    ShardRows sh{};
    sh.offsets = b->d_offsets; sh.K = b->K;
    sh.own_lo = b->d_own_lo; sh.own_hi = b->d_own_hi;
    sh.base = b->philox_base.empty() ? nullptr : b->d_base;
    sh.flags = b->d_flags; sh.enter = b->d_enter;
    return sh;
}

// Gibbs sweep over the owned frames of a time shard, in two phases with an exchange between them (bhmm_b200.h).
// Phase 1: forward on the team / panel family (warm-up on the halo before the owned range), the table of the owned rows and,
// per trajectory, the map from the state at the frame after the local end to the state at the first owned frame.
// Phase 2: from the handed-in states, link and replay the segments and count the statistics of the owned frames.
int gibbs_shard(bhmm_b200_batch* b, Emission& em, int emkind, const double* A, const double* pi, const double* d_u,
                unsigned long long seed, unsigned long long sweep, int* d_path, long long* d_counts, double* d_sums,
                double* loglik_host, cudaStream_t st)
{
    const int N = b->N, K = b->K;
    if (b->no_alpha) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "Viterbi-only batch: no forward variables"); return BHMM_ERR_UNSUPPORTED; }
    if (N > 256) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "sampling supports N <= 256"); return BHMM_ERR_UNSUPPORTED; }
    if (b->lane) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "sampling on a time shard runs the team family (bhmm_b200_batch_set_family(b, 0))"); return BHMM_ERR_UNSUPPORTED; }
    for (int k = 0; k < K; ++k)
        if (b->own_lo[k] < b->own_hi[k] && b->own_hi[k] != b->offsets[k + 1] - b->offsets[k]) {
            bhmm_set_error(BHMM_ERR_INVALID, "sampling on a time shard: the local trajectory must end with its owned range");
            return BHMM_ERR_INVALID;
        }
    RC_TRY(gibbs_shard_setup(b, st));
    if (b->gibbs_flags.empty()) b->gibbs_flags.assign(K, SHARD_STARTS);
    if (b->gibbs_enter.empty()) b->gibbs_enter.assign(K, -1);
    CUDA_TRY(cudaMemcpyAsync(b->d_flags, b->gibbs_flags.data(), sizeof(int) * K, cudaMemcpyHostToDevice, st));
    if (!b->philox_base.empty())
        CUDA_TRY(cudaMemcpyAsync(b->d_base, b->philox_base.data(), sizeof(long long) * K, cudaMemcpyHostToDevice, st));
    const ShardRows sh0 = shard_rows(b);
    if (b->gibbs_phase == 1) {
        b->gibbs_mapped = false;
        RC_TRY(upload_small(b->d_A, A, (size_t)N * N, st));
        RC_TRY(upload_small(b->d_pi, pi, N, st));
        b->w.ch.warm = b->warm_f;
        ScanGuard scan_guard(b, em, emkind);
        if (b->profile) cudaEventRecord(b->ev[0], st);
        RC_TRY(run_forward(b->w, em, emkind, N, b->d_A, b->d_pi, b->d_alpha, b->info, st));
        if (b->profile) cudaEventRecord(b->ev[1], st);
        if (b->w.chunked) b->warm_f = adapt_warm(b->warm_f, b->w.need_f, b->info.worst_f, b->info.fix_f > 0, b->warm_min, b->plan.maxT, b->edge_f);
        CUDA_TRY(cudaMemsetAsync(b->d_err, 0, sizeof(int), st));
        if (b->profile) cudaEventRecord(b->ev[2], st);
        RC_TRY(launch_sample_table_shard(b->d_alpha, b->d_A, d_u, seed, sweep, b->d_offsets, K, N, b->rows, b->d_F, b->d_err, sh0, st));
        RC_TRY(launch_chase_maps(b->d_F, b->seg, N, b->seg_map, st));
        const unsigned char* src = b->seg_map;
        for (size_t L = 0; L < b->lev_n.size(); ++L) {
            RC_TRY(launch_compose_maps(src, b->d_beg + b->lev_off[L], b->d_len + b->lev_off[L], b->lev_n[L], N, b->d_lev[L & 1], st));
            src = b->d_lev[L & 1];
        }
        if (b->profile) cudaEventRecord(b->ev[3], st);
        LAUNCHED(2 + b->lev_n.size());
        b->shard_map.assign((size_t)K * N, 0);
        int err = 0;
        CUDA_TRY(cudaMemcpyAsync(b->shard_map.data(), src, (size_t)K * N, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(&err, b->d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
        RC_TRY(finish_stream(st));
        if (err) { bhmm_set_error(err, "sample_path: no state could be drawn"); return err; }
        collect_times(b);
        b->gibbs_mapped = true;
        return BHMM_OK;
    }
    if (!b->gibbs_mapped) { bhmm_set_error(BHMM_ERR_INVALID, "Gibbs phase 2 on a time shard needs phase 1 first"); return BHMM_ERR_INVALID; }
    for (int k = 0; k < K; ++k) {
        const bool cont = (b->gibbs_flags[k] & SHARD_CONTINUES) && b->own_lo[k] < b->own_hi[k];
        if (cont && (b->gibbs_enter[k] < 0 || b->gibbs_enter[k] >= N)) {
            bhmm_set_error(BHMM_ERR_INVALID, "Gibbs on a time shard: a trajectory that continues needs its entering state in [0, N)");
            return BHMM_ERR_INVALID;
        }
    }
    CUDA_TRY(cudaMemcpyAsync(b->d_enter, b->gibbs_enter.data(), sizeof(int) * K, cudaMemcpyHostToDevice, st));
    if (b->profile) cudaEventRecord(b->ev[0], st);
    RC_TRY(launch_chase_resolve_shard(b->d_F, b->seg, N, b->seg_map, b->seg_enter, d_path, sh0, st));
    CUDA_TRY(cudaMemsetAsync(d_counts, 0, sizeof(long long) * ((size_t)N * N + 2 * N), st));
    if (d_sums) CUDA_TRY(cudaMemsetAsync(d_sums, 0, sizeof(double) * 2 * N, st));
    RC_TRY(launch_path_stats_shard(d_path, d_sums ? em.obs : nullptr, b->d_offsets, K, N, b->rows, d_counts,
                                   d_counts + (size_t)N * N, d_counts + (size_t)N * N + N, d_sums, d_sums ? d_sums + N : nullptr,
                                   sh0, st));
    if (b->profile) { cudaEventRecord(b->ev[1], st); cudaEventRecord(b->ev[2], st); cudaEventRecord(b->ev[3], st); }
    LAUNCHED(3);
    std::vector<double> ll(b->w.n_total);
    CUDA_TRY(cudaMemcpyAsync(ll.data(), b->w.chain_ll, sizeof(double) * b->w.n_total, cudaMemcpyDeviceToHost, st));
    RC_TRY(finish_stream(st));
    collect_times(b);
    double s = 0.0;
    for (double v : ll) s += v;
    if (loglik_host) *loglik_host = s;
    return BHMM_OK;
}

}  // namespace

extern "C" int bhmm_b200_stats_len_gaussian(int N) { return 1 + N + N * N + 3 * N; }
extern "C" int bhmm_b200_stats_len_discrete(int N) { return 1 + N + N * N + 3 * N; }

extern "C" int bhmm_b200_batch_create_ranges(bhmm_b200_batch** out, const long long* offsets, const long long* own_lo,
                                             const long long* own_hi, int K, int N, int chunk, int warm)
{
    bhmm_set_error(BHMM_OK, "");
    if (!out || !offsets || K < 1 || N < 1 || N > 1024) { bhmm_set_error(BHMM_ERR_INVALID, "bad batch arguments"); return BHMM_ERR_INVALID; }
    for (int k = 0; k < K; ++k)
        if (offsets[k + 1] <= offsets[k] || offsets[k + 1] - offsets[k] > 2000000000LL) {
            bhmm_set_error(BHMM_ERR_INVALID, "trajectories must be non-empty and shorter than 2e9 frames");
            return BHMM_ERR_INVALID;
        }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        bhmm_set_error(BHMM_ERR_CUDA, "no CUDA device available (bhmm_b200 has no CPU fallback)");
        return BHMM_ERR_CUDA;
    }
    bhmm_b200_batch* b = new bhmm_b200_batch();
    b->K = K; b->N = N;
    {
        const char* fam = getenv("BHMM_B200_FAMILY");     // "team" forces the general-N kernels (tests, comparisons)
        b->lane = lane_supported(N, EM_GAUSS) && !(fam && strcmp(fam, "team") == 0);
    }
    b->offsets.assign(offsets, offsets + K + 1);
    if (own_lo && own_hi) {
        for (int k = 0; k < K; ++k) {
            const long long T = offsets[k + 1] - offsets[k];
            if (own_lo[k] < 0 || own_hi[k] > T || own_lo[k] > own_hi[k]) {
                delete b;
                bhmm_set_error(BHMM_ERR_INVALID, "owned range outside its trajectory");
                return BHMM_ERR_INVALID;
            }
        }
        b->own_lo.assign(own_lo, own_lo + K);
        b->own_hi.assign(own_hi, own_hi + K);
    }
    b->rows = offsets[K] - offsets[0];
    if (offsets[0] != 0) { delete b; bhmm_set_error(BHMM_ERR_INVALID, "offsets[0] must be 0"); return BHMM_ERR_INVALID; }
    batch_plan(b, chunk, warm);
    *out = b;
    return BHMM_OK;
}

extern "C" void bhmm_b200_batch_destroy(bhmm_b200_batch* b)
{
    if (!b) return;
    b->arena.release();
    b->disc.release();
    b->scan.release();
    b->bst.release();
    b->gsh.release();
    for (int k = 0; k < 4; ++k) if (b->ev[k]) cudaEventDestroy(b->ev[k]);
    delete b;
}

extern "C" int bhmm_b200_batch_create(bhmm_b200_batch** out, const long long* offsets, int K, int N, int chunk,
                                      int warm)
{
    return bhmm_b200_batch_create_ranges(out, offsets, nullptr, nullptr, K, N, chunk, warm);
}

extern "C" int bhmm_b200_batch_border_handovers(const bhmm_b200_batch* b, int k, double* out)
{
    if (!b || !out || k < 0 || k >= b->K || !b->carved) { bhmm_set_error(BHMM_ERR_INVALID, "border_handovers: bad arguments or no E-step yet"); return BHMM_ERR_INVALID; }
    const int N = b->N, cf = b->plan.first_chain[k], cl = b->plan.last_chain[k];
    for (int i = 0; i < 4 * N; ++i) out[i] = 0.0;
    if (cf < 0) return BHMM_OK;                       // no owned frames in this trajectory
    const double* src[4] = {b->w.hu_f + (size_t)cf * N, b->w.he_f + (size_t)cl * N, b->w.hu_b + (size_t)cl * N,
                            b->w.he_b + (size_t)cf * N};
    for (int q = 0; q < 4; ++q)
        CUDA_TRY(cudaMemcpy(out + q * N, src[q], sizeof(double) * N, cudaMemcpyDeviceToHost));
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_set_border_starts(bhmm_b200_batch* b, int k, const double* fwd, const double* bwd)
{
    bhmm_set_error(BHMM_OK, "");
    if (!b || b->own_lo.empty()) { bhmm_set_error(BHMM_ERR_INVALID, "border starts are for time shards (batches with owned ranges)"); return BHMM_ERR_INVALID; }
    if (k < 0 || k >= b->K) { bhmm_set_error(BHMM_ERR_INVALID, "border starts: trajectory out of range"); return BHMM_ERR_INVALID; }
    const int N = b->N;
    const long long T = b->offsets[k + 1] - b->offsets[k];
    auto bad = [N](const double* v) {
        double s = 0.0;
        for (int i = 0; i < N; ++i) {
            if (!(v[i] >= 0.0) || !std::isfinite(v[i])) return true;         // NaN, negative, infinite
            s += v[i];
        }
        return !(s > 0.0);
    };
    if ((fwd || bwd) && b->own_lo[k] >= b->own_hi[k]) { bhmm_set_error(BHMM_ERR_INVALID, "border starts: the shard owns no frame of this trajectory"); return BHMM_ERR_INVALID; }
    if (fwd && b->own_lo[k] == 0) { bhmm_set_error(BHMM_ERR_INVALID, "forward border start: the owned range starts at local frame 0 (the trajectory's start)"); return BHMM_ERR_INVALID; }
    if (bwd && b->own_hi[k] >= T) { bhmm_set_error(BHMM_ERR_INVALID, "backward border start: the owned range ends with the local trajectory (the trajectory's end)"); return BHMM_ERR_INVALID; }
    if ((fwd && bad(fwd)) || (bwd && bad(bwd))) { bhmm_set_error(BHMM_ERR_INVALID, "border starts must be finite, non-negative and not all zero"); return BHMM_ERR_INVALID; }
    if ((int)b->has_f.size() != b->K) {
        b->has_f.assign(b->K, 0); b->has_b.assign(b->K, 0);
        b->bs_f.assign((size_t)b->K * N, 0.0); b->bs_b.assign((size_t)b->K * N, 0.0);
    }
    b->has_f[k] = fwd != nullptr;
    b->has_b[k] = bwd != nullptr;
    b->bst_ok = false;
    if (fwd) std::copy(fwd, fwd + N, b->bs_f.begin() + (size_t)k * N);
    if (bwd) std::copy(bwd, bwd + N, b->bs_b.begin() + (size_t)k * N);
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_replan(bhmm_b200_batch* b, int chunk, int warm)
{
    if (!b) return BHMM_ERR_INVALID;
    batch_plan(b, chunk, warm);
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_uses_lane_kernels(const bhmm_b200_batch* b) { return b && b->lane ? 1 : 0; }

extern "C" int bhmm_b200_batch_set_family(bhmm_b200_batch* b, int lane)
{
    if (!b) return BHMM_ERR_INVALID;
    const bool want = lane != 0 && lane_supported(b->N, EM_GAUSS);
    if (want == b->lane) return BHMM_OK;
    b->lane = want;
    batch_plan(b, b->req_chunk, b->req_warm);
    return BHMM_OK;
}

// Diagnostic: all hand-over vectors of the last pass, (chains, N) each: dir > 0 forward, dir < 0 backward.
extern "C" int bhmm_b200_batch_debug_handovers(const bhmm_b200_batch* b, int dir, double* used, double* end)
{
    if (!b || !b->carved || !used || !end) return BHMM_ERR_INVALID;
    const size_t n = sizeof(double) * (size_t)b->w.n_total * b->N;
    CUDA_TRY(cudaMemcpy(used, dir > 0 ? b->w.hu_f : b->w.hu_b, n, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(end, dir > 0 ? b->w.he_f : b->w.he_b, n, cudaMemcpyDeviceToHost));
    return BHMM_OK;
}

extern "C" double bhmm_b200_batch_scan_count(const bhmm_b200_batch* b) { return b ? b->w.scans : 0.0; }

extern "C" int bhmm_b200_wave_chains(int N)
{
    if (N < 1 || N > 1024) return 0;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return 0; }
    const char* fam = getenv("BHMM_B200_FAMILY");
    if (lane_supported(N, EM_GAUSS) && !(fam && strcmp(fam, "team") == 0)) {
        int sms = 148, dev = 0;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        return sms * lane_blocks_per_sm(N, EM_GAUSS) * lane_threads();
    }
    int tthreads = 32, tcpb = 1;
    team_shape(N, &tthreads, &tcpb);
    return backward_stats_grid(N, 1 << 28) * tcpb;
}

extern "C" int bhmm_b200_batch_set_viterbi_only(bhmm_b200_batch* b, int on)
{
    if (!b) return BHMM_ERR_INVALID;
    const bool was = b->no_alpha;
    b->no_alpha = on != 0;
    b->carved = false;          // the workspace is laid out again (query bhmm_b200_batch_workspace_bytes after this call)
    if (was != b->no_alpha && vit_wide(b)) batch_plan(b, b->req_chunk, b->req_warm);   // its chain plan follows the Viterbi kernel
    return BHMM_OK;
}

extern "C" size_t bhmm_b200_batch_workspace_bytes(const bhmm_b200_batch* b)
{
    return batch_layout(const_cast<bhmm_b200_batch*>(b), nullptr);
}

extern "C" int bhmm_b200_batch_attach_workspace(bhmm_b200_batch* b, void* d_workspace, size_t bytes)
{
    if (!b || !d_workspace) return BHMM_ERR_INVALID;
    b->arena.release();
    b->arena.base = (char*)d_workspace;
    b->arena.cap = bytes;
    b->arena.owned = false;
    b->carved = false;
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_set_profiling(bhmm_b200_batch* b, int on)
{
    if (!b) return BHMM_ERR_INVALID;
    if (on && !b->ev[0])
        for (int k = 0; k < 4; ++k)
            if (cudaEventCreate(&b->ev[k]) != cudaSuccess) return BHMM_ERR_CUDA;
    b->profile = on != 0;
    return BHMM_OK;
}

extern "C" void bhmm_b200_batch_kernel_ms(const bhmm_b200_batch* b, double ms[4])
{
    for (int k = 0; k < 4; ++k) ms[k] = b->kernel_ms[k];
}

extern "C" void bhmm_b200_batch_info(const bhmm_b200_batch* b, double info[8])
{
    info[0] = b->info.chains; info[1] = b->info.chunk; info[2] = b->info.warm; info[3] = b->info.fix_f;
    info[4] = b->info.fix_b; info[5] = b->info.worst_f; info[6] = b->info.worst_b; info[7] = b->info.rerun;
}

extern "C" int bhmm_b200_estep_gaussian(bhmm_b200_batch* b, const double* d_obs, const double* A, const double* pi,
                                        const double* means, const double* sigmas, int ignore_outliers,
                                        double* d_gamma, double* d_stats, void* stream)
{
    bhmm_set_error(BHMM_OK, "");
    cudaStream_t st = (cudaStream_t)stream;
    RC_TRY(batch_carve(b, st));
    begin_info(b);
    RC_TRY(upload_small(b->d_mu, means, b->N, st));
    RC_TRY(upload_small(b->d_sigma, sigmas, b->N, st));
    Emission em{};
    em.obs = d_obs; em.mu = b->d_mu; em.sigma = b->d_sigma; em.ignore_outliers = ignore_outliers;
    RC_TRY(estep_common(b, em, EM_GAUSS, A, pi, means, sigmas, d_gamma, d_stats, nullptr, st));
    RC_TRY(finish_stream(st));
    collect_times(b);
    return BHMM_OK;
}

extern "C" int bhmm_b200_estep_discrete(bhmm_b200_batch* b, const int* d_obs, const double* A, const double* pi,
                                        const double* B, int M, int ignore_outliers, double* d_gamma,
                                        double* d_stats, double* d_Bnum, void* stream)
{
    bhmm_set_error(BHMM_OK, "");
    cudaStream_t st = (cudaStream_t)stream;
    RC_TRY(batch_carve(b, st));
    begin_info(b);
    Emission em{};
    em.sym = d_obs; em.ignore_outliers = ignore_outliers;
    RC_TRY(prepare_discrete(b, B, M, em, st));
    RC_TRY(estep_common(b, em, EM_DISC, A, pi, nullptr, nullptr, d_gamma, d_stats, d_Bnum, st));
    RC_TRY(finish_stream(st));
    collect_times(b);
    return BHMM_OK;
}

// Operators of the owned frames of every trajectory (bhmm_b200.h): k_chain_operator[_wide] over the batch's chains, then the
// per-trajectory tree reduction (k_compose_operators), forward and backward, into d_out (K, 2, N, N + 1).
static int shard_operators(bhmm_b200_batch* b, Emission& em, int emkind, const double* A, const double* pi, double* d_out,
                           cudaStream_t st)
{
    const int N = b->N, K = b->K;
    const int n = b->w.n_total;
    std::vector<int> pairs, lev_n;
    std::vector<long long> lev_off;
    // level L pairs every chain at offset 2^(L+1) m from its run's first chain with the one 2^L after it (if still in the run)
    for (int s = 1;; s *= 2) {
        const size_t before = pairs.size();
        for (int k = 0; k < K; ++k) {
            const int cf = b->plan.first_chain[k], cl = b->plan.last_chain[k];
            if (cf < 0) continue;
            for (int c = cf; c + s <= cl; c += 2 * s) { pairs.push_back(c); pairs.push_back(c + s); }
        }
        if (pairs.size() == before) break;
        lev_off.push_back((long long)before / 2);
        lev_n.push_back((int)((pairs.size() - before) / 2));
    }
    std::vector<int> first(b->plan.first_chain.begin(), b->plan.first_chain.end());
    const size_t ops_bytes = (exact_scan_bytes(std::max(n, 1), N) + 255) & ~(size_t)255;
    const size_t pair_bytes = ((sizeof(int) * std::max<size_t>(pairs.size(), 2)) + 255) & ~(size_t)255;
    if (b->scan.ensure(ops_bytes + pair_bytes + sizeof(int) * K) != BHMM_OK) {
        bhmm_set_error(BHMM_ERR_NO_MEM, "shard operators: device memory for the chain operators");
        return BHMM_ERR_NO_MEM;
    }
    double* ops = reinterpret_cast<double*>(b->scan.base);
    int* d_pairs = reinterpret_cast<int*>(b->scan.base + ops_bytes);
    int* d_first = reinterpret_cast<int*>(b->scan.base + ops_bytes + pair_bytes);
    RC_TRY(upload_small(b->d_A, A, (size_t)N * N, st));
    RC_TRY(upload_small(b->d_pi, pi, N, st));
    if (!pairs.empty()) CUDA_TRY(cudaMemcpyAsync(d_pairs, pairs.data(), sizeof(int) * pairs.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_first, first.data(), sizeof(int) * K, cudaMemcpyHostToDevice, st));
    const long long kstride = 2LL * N * (N + 1);
    for (int d = 0; d < 2; ++d) {
        RC_TRY(launch_shard_operators(b->w.ch, n, em, emkind, b->d_A, N, d == 0 ? +1 : -1, d_pairs, lev_n, lev_off, d_first,
                                      K, ops, d_out + (size_t)d * N * (N + 1), kstride, st));
        LAUNCHED((n > 0 ? 1 + lev_n.size() : 0) + 1);
    }
    return finish_stream(st);                 // (the host tables above are in use until the copies have run)
}

static int shard_operators_check(bhmm_b200_batch* b, double* d_out)
{
    if (!b || !d_out) { bhmm_set_error(BHMM_ERR_INVALID, "shard operators: null batch or output"); return BHMM_ERR_INVALID; }
    if (b->own_lo.empty()) { bhmm_set_error(BHMM_ERR_INVALID, "shard operators are for time shards (batches with owned ranges)"); return BHMM_ERR_INVALID; }
    if (!exact_scan_ok(b->N)) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "shard operators support N <= 128"); return BHMM_ERR_UNSUPPORTED; }
    return BHMM_OK;
}

extern "C" int bhmm_b200_shard_operators_gaussian(bhmm_b200_batch* b, const double* d_obs, const double* A, const double* pi,
                                                  const double* means, const double* sigmas, int ignore_outliers,
                                                  double* d_out, void* stream)
{
    bhmm_set_error(BHMM_OK, "");
    RC_TRY(shard_operators_check(b, d_out));
    if (!d_obs || !A || !pi || !means || !sigmas) { bhmm_set_error(BHMM_ERR_INVALID, "shard operators: null argument"); return BHMM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    RC_TRY(batch_carve(b, st));
    RC_TRY(upload_small(b->d_mu, means, b->N, st));
    RC_TRY(upload_small(b->d_sigma, sigmas, b->N, st));
    Emission em{};
    em.obs = d_obs; em.mu = b->d_mu; em.sigma = b->d_sigma; em.ignore_outliers = ignore_outliers;
    return shard_operators(b, em, EM_GAUSS, A, pi, d_out, st);
}

extern "C" int bhmm_b200_shard_operators_discrete(bhmm_b200_batch* b, const int* d_obs, const double* A, const double* pi,
                                                  const double* B, int M, int ignore_outliers, double* d_out, void* stream)
{
    bhmm_set_error(BHMM_OK, "");
    RC_TRY(shard_operators_check(b, d_out));
    if (!d_obs || !A || !pi || !B || M < 1) { bhmm_set_error(BHMM_ERR_INVALID, "shard operators: null argument or M < 1"); return BHMM_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    RC_TRY(batch_carve(b, st));
    Emission em{};
    em.sym = d_obs; em.ignore_outliers = ignore_outliers;
    RC_TRY(prepare_discrete(b, B, M, em, st));
    return shard_operators(b, em, EM_DISC, A, pi, d_out, st);
}

static int viterbi_common(bhmm_b200_batch* b, Emission& em, int emkind, const double* A, const double* pi,
                          int* d_path, cudaStream_t st)
{
    const int N = b->N;
    // A batch with owned ranges is a TIME SHARD of longer trajectories (SURVEY 8e, C5): its chains cover the owned frames
    // and warm up on the halo before them; the hand-over at the shard border is certified by the caller across shards
    // (bhmm_b200_batch_border_handovers), the state at the last owned frame comes from the shard that owns the next frames
    // (bhmm_b200_batch_set_viterbi_end_state), and the local trajectory must END with the owned range (no right halo).
    const bool sharded = !b->own_lo.empty();
    const bool wide = vit_wide(b);
    const int NW = wide ? vflag_row_words(N) : 1;            // flag words per row of the map
    const int phase = b->vit_phase;
    if (sharded) {
        if (!panel_viterbi_chain_ok(N) && !wide) { bhmm_set_error(BHMM_ERR_UNSUPPORTED, "Viterbi on a time shard needs the chain-parallel Viterbi kernels (N <= 128, BHMM_B200_PANEL != 0)"); return BHMM_ERR_UNSUPPORTED; }
        for (int k = 0; k < b->K; ++k) {
            if (b->own_hi[k] != b->offsets[k + 1] - b->offsets[k]) { bhmm_set_error(BHMM_ERR_INVALID, "Viterbi on a time shard: the local trajectory must end with its owned range"); return BHMM_ERR_INVALID; }
            if (!b->w.chunked && b->own_lo[k] != 0) { bhmm_set_error(BHMM_ERR_INVALID, "Viterbi on a time shard: plan without chains"); return BHMM_ERR_INVALID; }
        }
    } else if (phase != 0) { bhmm_set_error(BHMM_ERR_INVALID, "Viterbi phases are for time shards"); return BHMM_ERR_INVALID; }
    RC_TRY(upload_small(b->d_A, A, (size_t)N * N, st));
    RC_TRY(upload_small(b->d_pi, pi, N, st));
    // Default (BHMM_B200_PANEL=0 turns it off): trajectories that the plan cuts into chains (one very long trajectory, C5) run their
    // max-product recursions chain-parallel with certified hand-overs.  A decision whose margin is too small to be
    // certified only matters if the resolved path goes through it: that is checked after the path chase, and then -- or when
    // the hand-overs cannot be certified -- the sequential kernel recomputes the whole map.
    bool chunked_map = (phase == 2) ? b->vit_map_chunked : false;
    if (phase != 2 && (panel_viterbi_chain_ok(N) || wide) && b->w.chunked) {
        VitChainArgs va{};
        va.em = em; va.N = N; va.A = b->d_A; va.pi = b->d_pi; va.backptr = b->d_F;
        va.hand_used = b->w.hu_f; va.hand_end = b->w.he_f; va.flagmap = b->d_vflag;
        va.margin_min = std::max(1e-11, 100.0 * g_cert_tol);   // two orders above the certification tolerance (default 1e-13)
        b->w.ch.warm = b->warm_f;
        const int rc = run_chains_certified(b->w, N, +1, [&](const Chains& ch, cudaStream_t s2) {
            VitChainArgs x = va;
            x.ch = ch;
            return wide ? launch_viterbi_chain_wide(x, emkind, s2) : launch_viterbi_chain(x, emkind, s2);
        }, b->info, st);
        if (rc == BHMM_OK) {
            chunked_map = true;
            // the warm-up length learns from this pass like the forward filter's (estep_common)
            b->warm_f = adapt_warm(b->warm_f, b->w.need_f, b->info.worst_f, b->info.fix_f > 0, b->warm_min, b->plan.maxT, b->edge_f);
        }
        else if (rc != BHMM_ERR_NOT_CERTIFIED || sharded) return rc;
        else bhmm_set_error(BHMM_OK, "");
    }
    for (int pass = 0; pass < 2; ++pass) {
        if (!chunked_map && phase != 2) {
            VitArgs a{};
            a.em = em; a.N = N; a.K = b->K; a.offsets = b->d_offsets; a.A = b->d_A; a.pi = b->d_pi;
            a.backptr = b->d_F; a.path = d_path;
            RC_TRY(launch_viterbi_team(a, emkind, st));
            LAUNCHED(1);
        }
        if (phase == 1) { b->vit_map_chunked = chunked_map; break; }
        if (sharded) {
            // rows before the first owned decision were never written: clear map and flags there; a handed-over end state
            // replaces the last row ("the last row holds the final arg max for every s'", k_chase_* convention)
            for (int k = 0; k < b->K; ++k) {
                const long long r0 = b->offsets[k], Tk = b->offsets[k + 1] - r0, lo = b->own_lo[k];
                if (lo > 1) {
                    CUDA_TRY(cudaMemsetAsync(b->d_F + (size_t)r0 * N, 0, (size_t)(lo - 1) * N, st));
                    if (chunked_map) CUDA_TRY(cudaMemsetAsync(b->d_vflag + (size_t)r0 * NW, 0, sizeof(unsigned) * (size_t)(lo - 1) * NW, st));
                }
                const int es = k < (int)b->vit_end.size() ? b->vit_end[k] : -1;
                if (es >= 0) {
                    if (es >= N) { bhmm_set_error(BHMM_ERR_INVALID, "Viterbi end state out of range"); return BHMM_ERR_INVALID; }
                    CUDA_TRY(cudaMemsetAsync(b->d_F + (size_t)(r0 + Tk - 1) * N, es, (size_t)N, st));
                    if (chunked_map) CUDA_TRY(cudaMemsetAsync(b->d_vflag + (size_t)(r0 + Tk - 1) * NW, 0, sizeof(unsigned) * NW, st));
                }
            }
        }
        if (N <= 256) {     // uint8 maps written by the kernel: resolve the paths by segment-wise map composition
            RC_TRY(launch_chase(b->d_F, b->seg, N, b->seg_map, b->seg_enter, d_path, st));
            LAUNCHED(3);
        }
        if (!chunked_map) break;
        int flagged = 0;
        CUDA_TRY(cudaMemsetAsync(b->d_err + 1, 0, sizeof(int), st));
        if (wide) RC_TRY(launch_viterbi_path_flags_wide(b->d_vflag, NW, d_path, b->d_offsets, b->K, b->rows, b->d_err + 1, st));
        else RC_TRY(launch_viterbi_path_flags(b->d_vflag, d_path, b->d_offsets, b->K, b->rows, b->d_err + 1, st));
        LAUNCHED(1);
        CUDA_TRY(cudaMemcpyAsync(&flagged, b->d_err + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (flagged == 0) break;
        if (sharded) {
            bhmm_set_error(BHMM_ERR_NOT_CERTIFIED, "Viterbi on a time shard: the path goes through a decision whose margin is below the certified tolerance; run the trajectory on one device");
            return BHMM_ERR_NOT_CERTIFIED;
        }
        chunked_map = false;                                // a near-tie on the path: sequential kernel, resolve again
    }
    return finish_stream(st);
}

extern "C" int bhmm_b200_batch_set_viterbi_phase(bhmm_b200_batch* b, int phase)
{
    if (!b || phase < 0 || phase > 2) return BHMM_ERR_INVALID;
    b->vit_phase = phase;
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_set_viterbi_end_state(bhmm_b200_batch* b, int k, int state)
{
    if (!b || k < 0 || k >= b->K) return BHMM_ERR_INVALID;
    if ((int)b->vit_end.size() != b->K) b->vit_end.assign(b->K, -1);
    b->vit_end[k] = state;
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_set_gibbs_phase(bhmm_b200_batch* b, int phase)
{
    if (!b || phase < 0 || phase > 2) { bhmm_set_error(BHMM_ERR_INVALID, "Gibbs phase must be 0, 1 or 2"); return BHMM_ERR_INVALID; }
    if (phase != 0 && b->own_lo.empty()) { bhmm_set_error(BHMM_ERR_INVALID, "Gibbs phases are for time shards (batches with owned ranges)"); return BHMM_ERR_INVALID; }
    b->gibbs_phase = phase;
    const bool seg = phase != 0;
    if (seg != b->gibbs_seg) {                  // the segment table changes: re-plan, the workspace is laid out again
        b->gibbs_seg = seg;
        batch_plan(b, b->req_chunk, b->req_warm);
    }
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_set_philox_rows(bhmm_b200_batch* b, const long long* base)
{
    if (!b) return BHMM_ERR_INVALID;
    if (base) b->philox_base.assign(base, base + b->K);
    else b->philox_base.clear();
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_set_gibbs_borders(bhmm_b200_batch* b, const int* flags)
{
    if (!b) return BHMM_ERR_INVALID;
    if (!flags) { b->gibbs_flags.clear(); return BHMM_OK; }
    for (int k = 0; k < b->K; ++k)
        if (flags[k] & ~(SHARD_CONTINUES | SHARD_STARTS)) { bhmm_set_error(BHMM_ERR_INVALID, "unknown Gibbs border flag"); return BHMM_ERR_INVALID; }
    b->gibbs_flags.assign(flags, flags + b->K);
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_set_gibbs_enter_state(bhmm_b200_batch* b, int k, int state)
{
    if (!b || k < 0 || k >= b->K || state < -1 || state >= b->N) { bhmm_set_error(BHMM_ERR_INVALID, "Gibbs entering state: bad trajectory or state"); return BHMM_ERR_INVALID; }
    if ((int)b->gibbs_enter.size() != b->K) b->gibbs_enter.assign(b->K, -1);
    b->gibbs_enter[k] = state;
    return BHMM_OK;
}

extern "C" int bhmm_b200_batch_gibbs_shard_map(const bhmm_b200_batch* b, int k, unsigned char* out)
{
    if (!b || !out || k < 0 || k >= b->K || !b->gibbs_mapped) { bhmm_set_error(BHMM_ERR_INVALID, "gibbs_shard_map: bad arguments or no phase 1 yet"); return BHMM_ERR_INVALID; }
    std::memcpy(out, b->shard_map.data() + (size_t)k * b->N, (size_t)b->N);
    return BHMM_OK;
}

extern "C" int bhmm_b200_viterbi_gaussian(bhmm_b200_batch* b, const double* d_obs, const double* A, const double* pi,
                                          const double* means, const double* sigmas, int ignore_outliers,
                                          int* d_path, void* stream)
{
    bhmm_set_error(BHMM_OK, "");
    cudaStream_t st = (cudaStream_t)stream;
    RC_TRY(batch_carve(b, st));
    begin_info(b);
    RC_TRY(upload_small(b->d_mu, means, b->N, st));
    RC_TRY(upload_small(b->d_sigma, sigmas, b->N, st));
    Emission em{};
    em.obs = d_obs; em.mu = b->d_mu; em.sigma = b->d_sigma; em.ignore_outliers = ignore_outliers;
    return viterbi_common(b, em, EM_GAUSS, A, pi, d_path, st);
}

extern "C" int bhmm_b200_viterbi_discrete(bhmm_b200_batch* b, const int* d_obs, const double* A, const double* pi,
                                          const double* B, int M, int ignore_outliers, int* d_path, void* stream)
{
    bhmm_set_error(BHMM_OK, "");
    cudaStream_t st = (cudaStream_t)stream;
    RC_TRY(batch_carve(b, st));
    begin_info(b);
    Emission em{};
    em.sym = d_obs; em.ignore_outliers = ignore_outliers;
    RC_TRY(prepare_discrete(b, B, M, em, st));
    return viterbi_common(b, em, EM_DISC, A, pi, d_path, st);
}

extern "C" int bhmm_b200_gibbs_gaussian(bhmm_b200_batch* b, const double* d_obs, const double* A, const double* pi,
                                        const double* means, const double* sigmas, int ignore_outliers,
                                        const double* d_u, unsigned long long seed, unsigned long long sweep,
                                        int* d_path, long long* d_counts, double* d_sums, double* loglik_host,
                                        void* stream)
{
    bhmm_set_error(BHMM_OK, "");
    cudaStream_t st = (cudaStream_t)stream;
    RC_TRY(batch_carve(b, st));
    begin_info(b);
    RC_TRY(upload_small(b->d_mu, means, b->N, st));
    RC_TRY(upload_small(b->d_sigma, sigmas, b->N, st));
    Emission em{};
    em.obs = d_obs; em.mu = b->d_mu; em.sigma = b->d_sigma; em.ignore_outliers = ignore_outliers;
    if (b->gibbs_phase) return gibbs_shard(b, em, EM_GAUSS, A, pi, d_u, seed, sweep, d_path, d_counts, d_sums, loglik_host, st);
    return gibbs_common(b, em, EM_GAUSS, A, pi, means, sigmas, d_u, seed, sweep, d_path, d_counts, d_sums, loglik_host, st);
}

extern "C" int bhmm_b200_gibbs_discrete(bhmm_b200_batch* b, const int* d_obs, const double* A, const double* pi,
                                        const double* B, int M, int ignore_outliers, const double* d_u,
                                        unsigned long long seed, unsigned long long sweep, int* d_path,
                                        long long* d_counts, double* loglik_host, void* stream)
{
    bhmm_set_error(BHMM_OK, "");
    cudaStream_t st = (cudaStream_t)stream;
    RC_TRY(batch_carve(b, st));
    begin_info(b);
    Emission em{};
    em.sym = d_obs; em.ignore_outliers = ignore_outliers;
    RC_TRY(prepare_discrete(b, B, M, em, st));
    if (b->gibbs_phase) return gibbs_shard(b, em, EM_DISC, A, pi, d_u, seed, sweep, d_path, d_counts, nullptr, loglik_host, st);
    return gibbs_common(b, em, EM_DISC, A, pi, nullptr, nullptr, d_u, seed, sweep, d_path, d_counts, nullptr, loglik_host, st);
}

extern "C" int bhmm_b200_path_symbol_histogram(const int* d_path, const int* d_obs, long long rows, int N, int M,
                                               long long* d_hist, void* stream)
{
    bhmm_set_error(BHMM_OK, "");
    RC_TRY(launch_symbol_histogram(d_path, d_obs, rows, N, M, d_hist, (cudaStream_t)stream));
    LAUNCHED(1);
    return finish_stream((cudaStream_t)stream);
}
