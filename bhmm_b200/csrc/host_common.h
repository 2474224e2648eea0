// bhmm_b200/csrc/host_common.h -- host-side plumbing shared by capi.cu (literal API) and engine.cu (batched engine).
#pragma once
#include <atomic>
#include <functional>
#include <mutex>
#include <vector>
#include <stdint.h>

#include "common.cuh"
#include "kernels.h"

extern std::atomic<unsigned long long> g_launches;
extern double g_cert_tol, g_repair_tol;
#define LAUNCHED(n) (g_launches.fetch_add((unsigned long long)(n), std::memory_order_relaxed))

#define RC_TRY(expr)                        \
    do {                                    \
        int rc_ = (expr);                   \
        if (rc_ != BHMM_OK) { bhmm_note_error(rc_, #expr); return rc_; } \
    } while (0)

// Grow-only device buffer carved into aligned pieces.  Either owned (cudaMalloc) or attached (caller memory).
struct Arena {
    char* base = nullptr;
    size_t cap = 0;
    bool owned = true;
    int ensure(size_t bytes);
    void release();
};

struct Carver {
    size_t off = 0;
    template <typename T>
    size_t add(size_t n)
    {
        off = (off + 255) & ~(size_t)255;
        const size_t o = off;
        off += n * sizeof(T);
        return o;
    }
};

// Chain table on the host: trajectories cut into chains of `chunk` frames, ordered by (trajectory, t0).
struct HostPlan {
    std::vector<long long> row0;
    std::vector<int> len, t0, T;
    int n = 0;
    int maxT = 0;
    bool chunked = false;       // some chain does not start its trajectory
    std::vector<int> first_chain, last_chain;   // per trajectory: its first / last chain in the table (-1: none)
};
// Chains over the OWNED frame range [own_lo[k], own_hi[k]) of every trajectory (NULL: the whole trajectory).  Frames
// outside the range are a halo: the chains next to the range's borders warm up on them (time-sharded trajectories).
void build_plan(const long long* offsets, int K, int chunk, HostPlan& p, const long long* own_lo = nullptr,
                const long long* own_hi = nullptr);
int auto_warm(int N);
int auto_chunk(long long rows, int N, int warm);

// Device scratch that belongs to one plan.
struct ChainWork {
    Chains ch{};                 // full table (list = NULL, n = all chains)
    int n_total = 0;
    bool chunked = false;
    double* chain_ll = nullptr;
    double* hu_f = nullptr;      // forward hand-over used / end
    double* he_f = nullptr;
    double* hu_b = nullptr;      // backward hand-over used / end
    double* he_b = nullptr;
    int* fail_list = nullptr;
    unsigned long long* cert_out = nullptr;   // device [n_fail, worst bits, sum warm, count]
    int warm_cap = 1;            // longest trajectory: a warm-up that long is an exact start
    double repair_tol = 0.0;     // hand-overs above max(g_cert_tol, this) are repaired (0: the certification tolerance itself)
    double need_f = 0, need_b = 0;   // certification's estimate of the warm-up the hardest hand-over needs
    // Exact fallback for models whose filter does not forget (scan_kernels.cu): fills he_f (dir > 0) or he_b (dir < 0) with
    // the exact hand-over vectors of every chain; set by the engine around a pass, empty when unavailable (N > 128)
    std::function<int(int dir, cudaStream_t st)> scan;
    double scans = 0;            // how many times the fallback ran (reported through bhmm_b200_batch_scan_count)
};
// next warm-up length from the current one, the certification's need estimate and the largest mismatch of the pass
int adapt_warm(int current, double need, double worst, bool failed, int warm_min, int warm_cap, double* edge);
size_t chainwork_bytes(int n_chains, int N);
// carve ChainWork out of `base` (device) and upload the plan; returns bytes used
int chainwork_setup(ChainWork& w, const HostPlan& p, int N, int warm, char* base, cudaStream_t st);

struct RunInfo {
    double chains = 0, chunk = 0, warm = 0, fix_f = 0, fix_b = 0, worst_f = 0, worst_b = 0, rerun = 0;
};

// Launch `launch(chains)` over all chains, then certify the hand-overs (dir = +1 forward, -1 backward) and re-run the
// failing chains from the exact neighbour value (Chains.list / Chains.exact) until none fails.  scan_first (with w.scan
// installed): skip the warm-up pass and start every chain from the exact scan (the Viterbi pass that is redone with a wider
// near-tie margin, engine.cu).
typedef std::function<int(const Chains& ch, cudaStream_t st)> ChainLauncher;
int run_chains_certified(ChainWork& w, int N, int dir, const ChainLauncher& launch, RunInfo& info, cudaStream_t st,
                         bool scan_first = false);
int auto_warm_lane(int N);
int auto_chunk_lane(long long rows, int N, int warm);

// forward over all chains + certification with exact fix-up sweeps.  alpha may be NULL.
int run_forward(ChainWork& w, const Emission& em, int emkind, int N, const double* dA, const double* dpi,
                double* d_alpha, RunInfo& info, cudaStream_t st);
// literal backward (beta written) + certification with exact fix-up sweeps.
int run_backward(ChainWork& w, const Emission& em, int emkind, int N, const double* dA, double* d_beta,
                 RunInfo& info, cudaStream_t st);
// certification read-back: returns number of failing chains (or <0 on CUDA error), updates worst
constexpr double EXACT_SCAN_TOL = 1e-11;   // hand-over tolerance of the pass that follows the exact scan (capi.cu)
long long certify_sync(ChainWork& w, int N, int dir, double* worst, cudaStream_t st, double tol_floor = 0.0);
int certify_async(ChainWork& w, int N, int dir, cudaStream_t st);     // verdict into a pinned slot, no synchronisation
long long certify_collect(ChainWork& w, int dir, double* worst);       // ... read after the stream was synchronised

// glibc srand()/rand() restatement (TYPE_3, r[i] = r[i-31] + r[i-3]); reproduces the reference's uniforms
struct GlibcRand {
    uint32_t ring[34];
    long pos = 0;               // index of the next r[] to produce
    GlibcRand() { seed(1); }
    void seed(unsigned int s);
    int next();                 // like rand(): 31-bit
    double uniform() { return (double)next() / (2147483647.0 + 1.0); }
};
