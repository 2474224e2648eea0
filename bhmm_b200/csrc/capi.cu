// bhmm_b200/csrc/capi.cu -- C ABI, part 1: library state, chain planning, certification drivers and the
// literal per-function API (host-pointer drop-ins and their device-pointer variants).  See include/bhmm_b200.h.
#include <algorithm>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <ctime>

#include "host_common.h"
#include "../../include/bhmm_b200.h"

std::atomic<unsigned long long> g_launches{0};
double g_cert_tol = 1e-13;      // the mismatch the warm-up length is steered to (bhmm_b200_set_certify_tolerance)
double g_repair_tol = 1e-11;    // E-step hand-overs above this are repaired (bhmm_b200_set_repair_tolerance)

static thread_local int t_err = BHMM_OK;
static thread_local char t_msg[512] = "";
static std::mutex g_lit_mutex;          // the literal API shares one scratch arena
static Arena g_lit_arena;
static int g_chunk_override = 0, g_warm_override = 0;
static double g_warm_margin = 0.0;      // added to the safety factors of adapt_warm (bhmm_b200_set_warm_margin)
static RunInfo g_last_info;
static GlibcRand g_rand;
static unsigned long long* g_pinned_cert = nullptr;

void bhmm_set_error(int code, const char* msg)
{
    t_err = code;
    snprintf(t_msg, sizeof(t_msg), "%s", msg ? msg : "");
}

// RC_TRY: keep the innermost message (e.g. the CUDA error string) and append the call site
void bhmm_note_error(int code, const char* where)
{
    if (t_err == code && t_msg[0]) {
        const size_t n = strlen(t_msg);
        if (n + 8 < sizeof(t_msg) && !strstr(t_msg, " <- ")) snprintf(t_msg + n, sizeof(t_msg) - n, " <- %s", where ? where : "");
        return;
    }
    bhmm_set_error(code, where);
}

static inline void clear_error() { t_err = BHMM_OK; t_msg[0] = 0; }

// ------------------------------------------------------------------------------------------------
// arena / planning
// ------------------------------------------------------------------------------------------------
int Arena::ensure(size_t bytes)
{
    if (bytes <= cap) return BHMM_OK;
    if (!owned) return BHMM_ERR_NO_MEM;
    if (base) cudaFree(base);
    base = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 4 + (1 << 20);
    if (cudaMalloc(&base, want) != cudaSuccess) {
        cudaGetLastError();
        if (cudaMalloc(&base, bytes) != cudaSuccess) { cudaGetLastError(); base = nullptr; return BHMM_ERR_NO_MEM; }
        cap = bytes;
        return BHMM_OK;
    }
    cap = want;
    return BHMM_OK;
}

void Arena::release()
{
    if (owned && base) cudaFree(base);
    base = nullptr;
    cap = 0;
}

void build_plan(const long long* offsets, int K, int chunk, HostPlan& p, const long long* own_lo, const long long* own_hi)
{
    p.row0.clear(); p.len.clear(); p.t0.clear(); p.T.clear();
    p.first_chain.assign(K, -1); p.last_chain.assign(K, -1);
    p.maxT = 0;
    p.chunked = false;
    for (int k = 0; k < K; ++k) {
        const long long r0 = offsets[k];
        const int T = (int)(offsets[k + 1] - r0);
        p.maxT = std::max(p.maxT, T);
        const int lo = own_lo ? (int)std::max<long long>(0, own_lo[k]) : 0;
        const int hi = own_hi ? (int)std::min<long long>(T, own_hi[k]) : T;
        for (int t0 = lo; t0 < hi; t0 += chunk) {
            if (p.first_chain[k] < 0) p.first_chain[k] = (int)p.row0.size();
            p.last_chain[k] = (int)p.row0.size();
            p.row0.push_back(r0 + t0);
            p.len.push_back(std::min(chunk, hi - t0));
            p.t0.push_back(t0);
            p.T.push_back(T);
            if (t0 > 0) p.chunked = true;
        }
    }
    p.n = (int)p.row0.size();
}

int auto_warm(int N)
{
    if (g_warm_override > 0) return g_warm_override;
    return std::min(8192, std::max(128, 48 * N));
}

int auto_chunk(long long rows, int N, int warm)
{
    if (g_chunk_override > 0) return g_chunk_override;
    int threads, cpb;
    team_shape(N, &threads, &cpb);
    // chains that fill the machine ONCE: resident blocks of the most demanding kernel (backward + statistics: two N x N
    // shared-memory matrices, one or two blocks per SM at N = 100) times chains per block.  More chains than that run
    // in rounds, and a last round that is mostly empty costs as much as a full one.
    const long long target = (long long)backward_stats_grid(N, 1 << 28) * cpb;
    long long c = (rows + target - 1) / target;
    c = std::max<long long>(c, 2LL * warm);
    c = std::max<long long>(c, 64);
    return (int)std::min<long long>(c, 1 << 30);
}

int auto_warm_lane(int N)
{
    if (g_warm_override > 0) return g_warm_override;
    return std::min(8192, std::max(64, 32 * N));
}

int auto_chunk_lane(long long rows, int N, int warm)
{
    // one thread per chain
    if (g_chunk_override > 0) return g_chunk_override;
    int sms = 148, dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // exactly one wave of resident blocks (occupancy of the register-hungriest lane kernel for this N)
    const long long target = (long long)sms * lane_blocks_per_sm(N, EM_GAUSS) * lane_threads();
    long long c = (rows + target - 1) / target;
    // A step of the lane kernels takes the same time with one resident warp per scheduler as with two (latency bound,
    // DESIGN.md 5.4), so the time of a pass is (chunk + warm-up) steps whatever the number of chains: a full wave of short
    // chains beats fewer, longer ones even when the warm-up exceeds the chunk (strong scaling: C3's 1024 trajectories over
    // 8 GPUs leave 338 frames per chain of a full wave; the old floor of 2 x warm-up ran a third of a wave for 1584 steps
    // instead of a full one for 866).  The floor only keeps the chain tables small for tiny inputs.
    c = std::max<long long>(c, std::max(64, warm / 4));
    return (int)std::min<long long>(c, 1 << 30);
}

int adapt_warm(int current, double need, double worst, bool failed, int warm_min, int warm_cap, double* edge)
{
    // edge[0]: the last warm-up need that was MEASURABLE, edge[1]: passes since it was confirmed.
    //
    // Keep the warm-up 12-15 % above what the hardest hand-over needs.  `need` (= w log tol / log m) is only informative
    // while the mismatch m is above the rounding-noise floor of two independently rounded filters (~1e-14); at the floor
    // the warm-up is known to be more than enough and shrinks slowly -- but not below 1.12 x the remembered need, which
    // is held for 20 passes and then decays by 3 % per pass until the mismatch becomes measurable again and confirms
    // or corrects it.  Without that memory the warm-up oscillates between the floor and the tolerance, and with the
    // mixing rate changing by a few per cent from one EM iteration (and one rank) to the next a hand-over fails every
    // 15-30 passes; a failed forward certification costs a fix-up sweep as long as a whole forward kernel (the repaired
    // chains are walked sequentially) on every rank of the job.  Simulated with 5-8 % jitter of the need
    // (tests/test_host_logic_cpu.py): failure rate 3-5 % -> below 1 % per pass for about 5 % more warm-up frames.
    double target;
    if (failed) {
        if (worst < 0.5) edge[0] = std::max(edge[0], need);      // (m >= 0.5: `need` is only a doubling rule)
        edge[1] = 0.0;
        target = std::max(1.2 * need, current + 32.0);
    } else if (worst <= 1e-14) {
        edge[1] += 1.0;
        if (edge[1] > 20.0) edge[0] *= 0.97;
        target = std::max(0.95 * current, (1.12 + g_warm_margin) * edge[0]);
    } else {
        edge[0] = std::max(need, 0.97 * edge[0]);
        edge[1] = 0.0;
        target = std::max(std::max((1.15 + g_warm_margin) * need, (1.12 + g_warm_margin) * edge[0]), 0.95 * current);
    }
    int w = (int)std::ceil(target / 16.0 - 1e-9) * 16;        // (1.12 x 300 is 336.00000000000006)
    w = std::max(w, warm_min);
    return std::min(w, std::max(warm_cap, 1));
}

// the policy above as a plain host function (no device needed): state[2] = {remembered need, passes since confirmed}
extern "C" int bhmm_b200_adapt_warm(int current, double need, double worst, int failed, int warm_min, int warm_cap,
                                    double* state)
{
    return adapt_warm(current, need, worst, failed != 0, warm_min, warm_cap, state);
}

size_t chainwork_bytes(int n, int N)
{
    Carver cv;
    cv.add<long long>(n);
    cv.add<int>(n); cv.add<int>(n); cv.add<int>(n);
    cv.add<double>(n);
    for (int k = 0; k < 4; ++k) cv.add<double>((size_t)n * N);
    cv.add<int>(n);
    cv.add<unsigned long long>(8);
    return cv.off + 256;
}

int chainwork_setup(ChainWork& w, const HostPlan& p, int N, int warm, char* base, cudaStream_t st)
{
    const int n = p.n;
    Carver cv;
    long long* row0 = (long long*)(base + cv.add<long long>(n));
    int* len = (int*)(base + cv.add<int>(n));
    int* t0 = (int*)(base + cv.add<int>(n));
    int* T = (int*)(base + cv.add<int>(n));
    w.chain_ll = (double*)(base + cv.add<double>(n));
    w.hu_f = (double*)(base + cv.add<double>((size_t)n * N));
    w.he_f = (double*)(base + cv.add<double>((size_t)n * N));
    w.hu_b = (double*)(base + cv.add<double>((size_t)n * N));
    w.he_b = (double*)(base + cv.add<double>((size_t)n * N));
    w.fail_list = (int*)(base + cv.add<int>(n));
    w.cert_out = (unsigned long long*)(base + cv.add<unsigned long long>(8));
    w.warm_cap = std::max(1, p.maxT);
    CUDA_TRY(cudaMemcpyAsync(row0, p.row0.data(), sizeof(long long) * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(len, p.len.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(t0, p.t0.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(T, p.T.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
    // the host vectors may die before the copies run: pageable copies are staged synchronously, so this is safe,
    // but make it explicit
    CUDA_TRY(cudaStreamSynchronize(st));
    w.ch.row0 = row0; w.ch.len = len; w.ch.t0 = t0; w.ch.T = T;
    w.ch.list = nullptr; w.ch.n = n; w.ch.warm = warm; w.ch.exact = 0; w.ch.warmv = nullptr;
    w.n_total = n;
    w.chunked = p.chunked;
    return BHMM_OK;
}

// ------------------------------------------------------------------------------------------------
// certification drivers
// ------------------------------------------------------------------------------------------------
long long certify_sync(ChainWork& w, int N, int dir, double* worst, cudaStream_t st, double tol_floor)
{
    if (!g_pinned_cert) {
        if (cudaMallocHost(&g_pinned_cert, 8 * sizeof(unsigned long long)) != cudaSuccess) return -1;
    }
    Chains full = w.ch;
    full.list = nullptr;
    full.n = w.n_total;
    full.warmv = nullptr;
    launch_certify(full, w.n_total, N, dir, dir > 0 ? w.hu_f : w.hu_b, dir > 0 ? w.he_f : w.he_b, std::max(g_cert_tol, tol_floor),
                   std::max(w.repair_tol, tol_floor), w.fail_list, w.cert_out, st);
    LAUNCHED(1);
    if (cudaMemcpyAsync(g_pinned_cert, w.cert_out, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st) !=
        cudaSuccess)
        return -1;
    if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
    double wv;
    memcpy(&wv, &g_pinned_cert[1], sizeof(double));
    if (worst) *worst = tol_floor > 0.0 ? wv : std::max(*worst, wv);     // after the exact scan: the mismatch of THAT pass
    double& need = dir > 0 ? w.need_f : w.need_b;
    need = std::max(need, (double)g_pinned_cert[2]);       // callers reset it at the start of a pass
    return (long long)g_pinned_cert[0];
}

// Certification WITHOUT a host round trip: the verdict of direction `dir` goes to slot (dir > 0 ? 0 : 1) of the pinned result
// buffer; certify_collect reads it after the caller's next synchronisation of the stream.
int certify_async(ChainWork& w, int N, int dir, cudaStream_t st)
{
    if (!g_pinned_cert) {
        if (cudaMallocHost(&g_pinned_cert, 8 * sizeof(unsigned long long)) != cudaSuccess) return BHMM_ERR_NO_MEM;
    }
    const int slot = dir > 0 ? 0 : 1;
    Chains full = w.ch;
    full.list = nullptr;
    full.n = w.n_total;
    full.warmv = nullptr;
    launch_certify(full, w.n_total, N, dir, dir > 0 ? w.hu_f : w.hu_b, dir > 0 ? w.he_f : w.he_b, g_cert_tol, w.repair_tol, w.fail_list,
                   w.cert_out + 4 * slot, st);
    LAUNCHED(1);
    CUDA_TRY(cudaMemcpyAsync(g_pinned_cert + 4 * slot, w.cert_out + 4 * slot, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    return BHMM_OK;
}

long long certify_collect(ChainWork& w, int dir, double* worst)
{
    const int slot = dir > 0 ? 0 : 1;
    double wv;
    memcpy(&wv, &g_pinned_cert[4 * slot + 1], sizeof(double));
    if (worst) *worst = std::max(*worst, wv);
    double& need = dir > 0 ? w.need_f : w.need_b;
    need = std::max(need, (double)g_pinned_cert[4 * slot + 2]);
    return (long long)g_pinned_cert[4 * slot];
}

int run_chains_certified(ChainWork& w, int N, int dir, const ChainLauncher& launch, RunInfo& info, cudaStream_t st,
                         bool scan_first)
{
    Chains all = w.ch;
    all.list = nullptr; all.n = w.n_total; all.exact = 0;
    all.warmv = nullptr;
    (dir > 0 ? w.need_f : w.need_b) = 0.0;
    double& worst = dir > 0 ? info.worst_f : info.worst_b;
    double& sweeps = dir > 0 ? info.fix_f : info.fix_b;
    auto exact_from_scan = [&]() -> int {
        RC_TRY(w.scan(dir, st));
        LAUNCHED(2);
        w.scans += 1;
        Chains ex = all;
        ex.exact = 1;
        RC_TRY(launch(ex, st));
        LAUNCHED(1);
        return BHMM_OK;
    };
    if (scan_first && w.chunked && w.scan) {
        RC_TRY(exact_from_scan());
    } else {
        RC_TRY(launch(all, st));
        LAUNCHED(1);
    }
    if (!w.chunked) return BHMM_OK;
    // After the exact scan the starts are exact up to the rounding of two different evaluation orders (operator products vs.
    // the vector recursion); a model that does not forget does not contract that difference either (measured: up to
    // 1.2e-13 over 400-frame chains), so the hand-overs of that pass are accepted at 1e-11 -- non-expansive, i.e. still two
    // orders below the 1e-10 parity bar.
    double tol_floor = (scan_first && w.scan) ? EXACT_SCAN_TOL : 0.0;
    for (int sweep = 0;; ++sweep) {
        const long long nfail = certify_sync(w, N, dir, &worst, st, tol_floor);
        if (nfail < 0) { bhmm_set_error(BHMM_ERR_CUDA, cudaGetErrorString(cudaGetLastError())); return BHMM_ERR_CUDA; }
        if (nfail == 0) break;
        if (sweep > w.n_total + 2) { bhmm_set_error(BHMM_ERR_NOT_CERTIFIED, "chain hand-overs not certified"); return BHMM_ERR_NOT_CERTIFIED; }
        if (sweep == 1 && w.scan && nfail > 1 && tol_floor == 0.0) {
            // The first repair sweep did not clear the list: the model does not forget its start within the warm-up, and
            // chain-by-chain repairs would walk the trajectory sequentially.  Exact starts for ALL chains from the
            // transfer-operator scan, then one parallel pass from them.
            RC_TRY(exact_from_scan());
            sweeps += 1;
            info.rerun += (double)w.n_total;
            tol_floor = EXACT_SCAN_TOL;
            continue;
        }
        Chains some = all;
        some.list = w.fail_list; some.n = (int)nfail; some.exact = 1;
        RC_TRY(launch(some, st));
        LAUNCHED(1);
        sweeps += 1;
        info.rerun += (double)nfail;
    }
    return BHMM_OK;
}

int run_forward(ChainWork& w, const Emission& em, int emkind, int N, const double* dA, const double* dpi,
                double* d_alpha, RunInfo& info, cudaStream_t st)
{
    FwdArgs a{};
    a.em = em; a.N = N; a.A = dA; a.pi = dpi; a.alpha = d_alpha;
    a.chain_ll = w.chain_ll; a.hand_used = w.hu_f; a.hand_end = w.he_f;
    return run_chains_certified(w, N, +1, [&](const Chains& ch, cudaStream_t s2) {
        FwdArgs b = a;
        b.ch = ch;
        return launch_forward_team(b, emkind, s2);
    }, info, st);
}

int run_backward(ChainWork& w, const Emission& em, int emkind, int N, const double* dA, double* d_beta,
                 RunInfo& info, cudaStream_t st)
{
    BwdArgs a{};
    a.em = em; a.N = N; a.A = dA; a.beta = d_beta;
    a.hand_used = w.hu_b; a.hand_end = w.he_b;
    return run_chains_certified(w, N, -1, [&](const Chains& ch, cudaStream_t s2) {
        BwdArgs b = a;
        b.ch = ch;
        return launch_backward_team(b, emkind, false, s2);
    }, info, st);
}

// ------------------------------------------------------------------------------------------------
// glibc rand() restatement
// ------------------------------------------------------------------------------------------------
void GlibcRand::seed(unsigned int s)
{
    // published algorithm of glibc random_r.c (TYPE_3): r[0]=seed (0 -> 1); r[i] = 16807*r[i-1] mod (2^31-1) by
    // Schrage's method for i<31; r[i] = r[i-31] for i=31..33; then r[i] = r[i-31] + r[i-3]; the first 310 of
    // those are discarded, output k is r[k+344] >> 1.
    int32_t r[34];
    if (s == 0) s = 1;
    r[0] = (int32_t)s;
    for (int i = 1; i < 31; ++i) {
        const long hi = r[i - 1] / 127773, lo = r[i - 1] % 127773;
        long word = 16807 * lo - 2836 * hi;
        if (word < 0) word += 2147483647;
        r[i] = (int32_t)word;
    }
    for (int i = 31; i < 34; ++i) r[i] = r[i - 31];
    for (int i = 0; i < 34; ++i) ring[i] = (uint32_t)r[i];
    pos = 34;
    for (int i = 34; i < 344; ++i) next();
}

int GlibcRand::next()
{
    const uint32_t v = ring[(pos - 31) % 34] + ring[(pos - 3) % 34];
    ring[pos % 34] = v;
    ++pos;
    return (int)(v >> 1);
}

// ------------------------------------------------------------------------------------------------
// library state
// ------------------------------------------------------------------------------------------------
extern "C" int bhmm_b200_last_error(void) { return t_err; }
extern "C" const char* bhmm_b200_last_error_string(void) { return t_msg; }
extern "C" const char* bhmm_b200_version(void) { return "bhmm_b200 0.1 (sm_100a)"; }
extern "C" int bhmm_b200_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
extern "C" unsigned long long bhmm_b200_launch_count(void) { return g_launches.load(); }
extern "C" void bhmm_b200_set_chunking(int chunk, int warm) { g_chunk_override = chunk; g_warm_override = warm; }
extern "C" void bhmm_b200_set_certify_tolerance(double tol) { g_cert_tol = tol; }
extern "C" void bhmm_b200_set_repair_tolerance(double tol) { g_repair_tol = tol > 0.0 ? tol : 0.0; }
extern "C" void bhmm_b200_set_warm_margin(double extra) { g_warm_margin = extra < 0.0 ? 0.0 : (extra > 2.0 ? 2.0 : extra); }
extern "C" void bhmm_b200_last_info(double info[8])
{
    info[0] = g_last_info.chains; info[1] = g_last_info.chunk; info[2] = g_last_info.warm;
    info[3] = g_last_info.fix_f; info[4] = g_last_info.fix_b; info[5] = g_last_info.worst_f;
    info[6] = g_last_info.worst_b; info[7] = g_last_info.rerun;
}
extern "C" void bhmm_b200_set_seed(int seed)
{
    std::lock_guard<std::mutex> lk(g_lit_mutex);
    g_rand.seed(seed >= 0 ? (unsigned int)seed : (unsigned int)time(nullptr));   // set_seed, _hidden.c:321-327
}
extern "C" void bhmm_b200_glibc_uniforms(int seed, long n, double* u)
{
    GlibcRand r;
    r.seed((unsigned int)seed);
    for (long k = 0; k < n; ++k) u[k] = r.uniform();
}

static size_t chase_scratch_bytes(int N, int T);
static int chase_single(const unsigned char* F, int N, int T, char* scratch, int* d_path, cudaStream_t st);

static int require_device()
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        bhmm_set_error(BHMM_ERR_CUDA, "no CUDA device available (bhmm_b200 has no CPU fallback)");
        return BHMM_ERR_CUDA;
    }
    return BHMM_OK;
}

static int finish(cudaStream_t st)
{
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { bhmm_set_error(BHMM_ERR_CUDA, cudaGetErrorString(e)); return BHMM_ERR_CUDA; }
    return BHMM_OK;
}

// scratch of a single-trajectory literal call: chain plan + extra bytes
struct LitScratch {
    ChainWork w;
    HostPlan plan;
    char* extra = nullptr;
};

static int lit_prepare(LitScratch& s, int N, int T, size_t extra_bytes, bool need_chains, cudaStream_t st)
{
    const int warm = auto_warm(N);
    const int chunk = need_chains ? auto_chunk(T, N, warm) : std::max(T, 1);
    const long long offs[2] = {0, T};
    build_plan(offs, 1, chunk, s.plan);
    const size_t cw = chainwork_bytes(s.plan.n, N);
    RC_TRY(g_lit_arena.ensure(cw + extra_bytes + 512));
    RC_TRY(chainwork_setup(s.w, s.plan, N, warm, g_lit_arena.base, st));
    s.extra = g_lit_arena.base + ((cw + 255) & ~(size_t)255);
    g_last_info = RunInfo();
    g_last_info.chains = s.plan.n; g_last_info.chunk = chunk; g_last_info.warm = warm;
    return BHMM_OK;
}

static double sum_chain_ll(const ChainWork& w, cudaStream_t st, int* rc)
{
    std::vector<double> ll(w.n_total);
    if (cudaMemcpyAsync(ll.data(), w.chain_ll, sizeof(double) * w.n_total, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
        *rc = BHMM_ERR_CUDA;
        return 0.0;
    }
    double s = 0.0;
    for (double v : ll) s += v;
    *rc = BHMM_OK;
    return s;
}

// ------------------------------------------------------------------------------------------------
// (2) device-pointer variants -- the real implementations
// ------------------------------------------------------------------------------------------------
static int forward_dev_locked(double* d_alpha, const double* d_A, const double* d_pobs, const double* d_pi, int N,
                              int T, double* logprob, cudaStream_t st, size_t extra, char** extra_out)
{
    if (N < 1 || T < 1) { bhmm_set_error(BHMM_ERR_INVALID, "N and T must be positive"); return BHMM_ERR_INVALID; }
    LitScratch s;
    RC_TRY(lit_prepare(s, N, T, extra, true, st));
    if (extra_out) *extra_out = s.extra;
    Emission em{};
    em.pobs = d_pobs;
    RC_TRY(run_forward(s.w, em, EM_POBS, N, d_A, d_pi, d_alpha, g_last_info, st));
    int rc;
    const double ll = sum_chain_ll(s.w, st, &rc);
    if (rc) { bhmm_set_error(rc, "log-likelihood read-back failed"); return rc; }
    if (logprob) *logprob = ll;
    return BHMM_OK;
}

extern "C" int bhmm_b200_forward_dev(double* d_alpha, const double* d_A, const double* d_pobs, const double* d_pi,
                                     int N, int T, double* logprob_host, void* stream)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_lit_mutex);
    RC_TRY(forward_dev_locked(d_alpha, d_A, d_pobs, d_pi, N, T, logprob_host, (cudaStream_t)stream, 0, nullptr));
    return finish((cudaStream_t)stream);
}

extern "C" int bhmm_b200_backward_dev(double* d_beta, const double* d_A, const double* d_pobs, int N, int T,
                                      void* stream)
{
    clear_error();
    RC_TRY(require_device());
    if (N < 1 || T < 1) { bhmm_set_error(BHMM_ERR_INVALID, "N and T must be positive"); return BHMM_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(g_lit_mutex);
    cudaStream_t st = (cudaStream_t)stream;
    LitScratch s;
    RC_TRY(lit_prepare(s, N, T, 0, true, st));
    Emission em{};
    em.pobs = d_pobs;
    RC_TRY(run_backward(s.w, em, EM_POBS, N, d_A, d_beta, g_last_info, st));
    return finish(st);
}

extern "C" int bhmm_b200_state_probabilities_dev(double* d_gamma, const double* d_alpha, const double* d_beta,
                                                 int N, int T, void* stream)
{
    clear_error();
    RC_TRY(require_device());
    RC_TRY(launch_state_probabilities(d_alpha, d_beta, N, T, d_gamma, (cudaStream_t)stream));
    LAUNCHED(1);
    return finish((cudaStream_t)stream);
}

extern "C" int bhmm_b200_state_counts_dev(double* d_counts, const double* d_gamma, int N, int T, void* stream)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_lit_mutex);
    const int nb = state_counts_blocks(T);
    RC_TRY(g_lit_arena.ensure(sizeof(double) * (size_t)std::max(nb, 1) * N + 256));
    RC_TRY(launch_state_counts(d_gamma, N, T, d_counts, (double*)g_lit_arena.base, nullptr, (cudaStream_t)stream));
    LAUNCHED(2);
    return finish((cudaStream_t)stream);
}

extern "C" int bhmm_b200_transition_counts_dev(double* d_C, const double* d_A, const double* d_pobs,
                                               const double* d_alpha, const double* d_beta, int N, int T,
                                               void* stream)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_lit_mutex);
    const int nb = std::max(1, transition_counts_blocks(T));
    RC_TRY(g_lit_arena.ensure(sizeof(double) * ((size_t)T + (size_t)nb * N * N) + 256));
    RC_TRY(launch_transition_counts(d_alpha, d_beta, d_A, d_pobs, N, T, d_C, (double*)g_lit_arena.base,
                                    (cudaStream_t)stream));
    LAUNCHED(3);
    return finish((cudaStream_t)stream);
}

extern "C" int bhmm_b200_viterbi_dev(int* d_path, const double* d_A, const double* d_pobs, const double* d_pi,
                                     int N, int T, void* stream)
{
    clear_error();
    RC_TRY(require_device());
    if (N < 1 || T < 1) { bhmm_set_error(BHMM_ERR_INVALID, "N and T must be positive"); return BHMM_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(g_lit_mutex);
    cudaStream_t st = (cudaStream_t)stream;
    const bool chunked = panel_viterbi_chain_ok(N) && T >= 4096;
    Carver cv;
    const size_t o_off = cv.add<long long>(2);
    const size_t o_bp = cv.add<unsigned short>((size_t)T * N);
    const size_t o_chase = cv.add<char>(chase_scratch_bytes(N, T));
    const size_t o_flag = cv.add<int>(4);
    const size_t o_vflag = cv.add<unsigned>(chunked ? (size_t)T : 1);
    // Default (BHMM_B200_PANEL=0 turns it off): a long trajectory is cut into chains whose max-product recursions run in parallel with
    // certified hand-overs (panel_kernels.cu:k_viterbi_chain32); the strictly sequential kernel walks it at ~0.5 us per
    // frame, slower than one CPU core.  Any decision too close to call, or an uncertifiable hand-over: sequential kernel.
    LitScratch s;
    char* base = nullptr;
    if (chunked) {
        RC_TRY(lit_prepare(s, N, T, cv.off + 256, true, st));
        base = s.extra;
    } else {
        RC_TRY(g_lit_arena.ensure(cv.off + 256));
        base = g_lit_arena.base;
    }
    long long* d_offs = (long long*)(base + o_off);
    const long long offs[2] = {0, T};
    CUDA_TRY(cudaMemcpyAsync(d_offs, offs, sizeof(offs), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    VitArgs a{};
    a.em.pobs = d_pobs;
    a.N = N; a.K = 1; a.offsets = d_offs; a.A = d_A; a.pi = d_pi;
    a.backptr = base + o_bp; a.path = d_path;
    bool chunked_map = false;
    int* d_flag = (int*)(base + o_flag);
    unsigned* d_vflag = (unsigned*)(base + o_vflag);
    if (chunked && s.w.chunked) {
        VitChainArgs va{};
        va.em.pobs = d_pobs;
        va.N = N; va.A = d_A; va.pi = d_pi; va.backptr = a.backptr;
        va.hand_used = s.w.hu_f; va.hand_end = s.w.he_f; va.flagmap = d_vflag;
        va.margin_min = std::max(1e-11, 100.0 * g_cert_tol);
        const int rc = run_chains_certified(s.w, N, +1, [&](const Chains& ch, cudaStream_t s2) {
            VitChainArgs x = va;
            x.ch = ch;
            return launch_viterbi_chain(x, EM_POBS, s2);
        }, g_last_info, st);
        if (rc == BHMM_OK) chunked_map = true;
        else if (rc != BHMM_ERR_NOT_CERTIFIED) return rc;
        else clear_error();
    }
    for (int pass = 0; pass < 2; ++pass) {
        if (!chunked_map) {
            RC_TRY(launch_viterbi_team(a, EM_POBS, st));
            LAUNCHED(1);
        }
        if (N <= 256)   // uint8 maps: the path is resolved in parallel; wider back-pointers were backtraced in the kernel
            RC_TRY(chase_single((const unsigned char*)a.backptr, N, T, base + o_chase, d_path, st));
        if (!chunked_map) break;
        int flagged = 0;                                    // near-tie decisions ON the resolved path
        CUDA_TRY(cudaMemsetAsync(d_flag, 0, sizeof(int), st));
        RC_TRY(launch_viterbi_path_flags(d_vflag, d_path, d_offs, 1, T, d_flag, st));
        LAUNCHED(1);
        CUDA_TRY(cudaMemcpyAsync(&flagged, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (flagged == 0) break;
        chunked_map = false;
    }
    return finish(st);
}

// Resolve the path of ONE trajectory from its map table F (T,N): F[t][s'] = state at t given state s' at t+1 (the last
// row ignores s').  Segment-wise map composition (k_chase_*); `scratch` holds chase_scratch_bytes(N, T) bytes.
static size_t chase_scratch_bytes(int N, int T)
{
    const size_t nseg = (size_t)(T + 255) / 256 + 1;
    return nseg * (8 + 12 + N + 4) + 16 + 4096;
}

static int chase_single(const unsigned char* F, int N, int T, char* scratch, int* d_path, cudaStream_t st)
{
    const int seg = 256;
    HostPlan sp;
    const long long offs[2] = {0, T};
    build_plan(offs, 1, seg, sp);
    Carver cv;
    const size_t o_row0 = cv.add<long long>(sp.n);
    const size_t o_len = cv.add<int>(sp.n), o_t0 = cv.add<int>(sp.n), o_T = cv.add<int>(sp.n);
    const size_t o_map = cv.add<unsigned char>((size_t)sp.n * N);
    const size_t o_enter = cv.add<int>(sp.n);
    CUDA_TRY(cudaMemcpyAsync(scratch + o_row0, sp.row0.data(), sizeof(long long) * sp.n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(scratch + o_len, sp.len.data(), sizeof(int) * sp.n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(scratch + o_t0, sp.t0.data(), sizeof(int) * sp.n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(scratch + o_T, sp.T.data(), sizeof(int) * sp.n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    Chains sg{};
    sg.row0 = (const long long*)(scratch + o_row0);
    sg.len = (const int*)(scratch + o_len);
    sg.t0 = (const int*)(scratch + o_t0);
    sg.T = (const int*)(scratch + o_T);
    sg.n = sp.n;
    RC_TRY(launch_chase(F, sg, N, (unsigned char*)(scratch + o_map), (int*)(scratch + o_enter), d_path, st));
    LAUNCHED(3);
    return BHMM_OK;
}

// path from a (T,N) alpha and per-ROW uniforms (u_row[t] is the draw of frame t)
static int sample_rows_locked(int* d_path, const double* d_alpha, const double* d_A, const double* d_urow, int N,
                              int T, char* scratch, cudaStream_t st)
{
    Carver cv;
    const size_t o_off = cv.add<long long>(2);
    const size_t o_F = cv.add<unsigned char>((size_t)T * N);
    const size_t o_err = cv.add<int>(1);
    const size_t o_chase = cv.add<char>(chase_scratch_bytes(N, T));
    long long* d_offs = (long long*)(scratch + o_off);
    const long long offs[2] = {0, T};
    CUDA_TRY(cudaMemcpyAsync(d_offs, offs, sizeof(offs), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(scratch + o_err, 0, sizeof(int), st));
    CUDA_TRY(cudaStreamSynchronize(st));
    unsigned char* F = (unsigned char*)(scratch + o_F);
    RC_TRY(launch_sample_table(d_alpha, d_A, d_urow, d_offs, 1, N, T, F, (int*)(scratch + o_err), st));
    LAUNCHED(1);
    RC_TRY(chase_single(F, N, T, scratch + o_chase, d_path, st));
    int err = 0;
    CUDA_TRY(cudaMemcpyAsync(&err, scratch + o_err, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (err) { bhmm_set_error(err, "sample_path: no state could be drawn (alpha not normalisable?)"); return err; }
    return BHMM_OK;
}

static size_t sample_scratch_bytes(int N, int T)
{
    return (size_t)T * N + chase_scratch_bytes(N, T) + 4096;
}

extern "C" int bhmm_b200_sample_path_dev(int* d_path, const double* d_alpha, const double* d_A, const double* d_u,
                                         int N, int T, void* stream)
{
    // d_u: device, per-ROW uniforms
    clear_error();
    RC_TRY(require_device());
    if (N < 1 || T < 1) { bhmm_set_error(BHMM_ERR_INVALID, "N and T must be positive"); return BHMM_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(g_lit_mutex);
    RC_TRY(g_lit_arena.ensure(sample_scratch_bytes(N, T)));
    RC_TRY(sample_rows_locked(d_path, d_alpha, d_A, d_u, N, T, g_lit_arena.base, (cudaStream_t)stream));
    return finish((cudaStream_t)stream);
}

extern "C" int bhmm_b200_gaussian_p_obs_dev(const double* d_o, const double* d_mus, const double* d_sigmas, int N,
                                            int T, int ignore_outliers, double* d_p, void* stream)
{
    clear_error();
    RC_TRY(require_device());
    RC_TRY(launch_gaussian_pobs(d_o, d_mus, d_sigmas, N, T, ignore_outliers, d_p, (cudaStream_t)stream));
    LAUNCHED(1);
    return finish((cudaStream_t)stream);
}

extern "C" int bhmm_b200_discrete_p_obs_dev(const int* d_obs, const double* d_B, int N, int M, int T,
                                            int ignore_outliers, double* d_p, void* stream)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_lit_mutex);
    RC_TRY(g_lit_arena.ensure(sizeof(double) * (size_t)N * M + 256));
    double* Bt = (double*)g_lit_arena.base;
    RC_TRY(launch_transpose(d_B, N, M, Bt, (cudaStream_t)stream));
    RC_TRY(launch_discrete_pobs(d_obs, Bt, N, M, T, ignore_outliers, d_p, (cudaStream_t)stream));
    LAUNCHED(2);
    return finish((cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------
// (1) host-pointer drop-ins: stage through a private device buffer, call the device variant
// ------------------------------------------------------------------------------------------------
namespace {

// second arena for staged host arrays (the first one is scratch of the device variants)
Arena g_stage;
std::mutex g_stage_mutex;

struct Stage {
    Carver cv;
    std::vector<size_t> offs;
    size_t add(size_t bytes) { offs.push_back(cv.add<char>(bytes)); return offs.size() - 1; }
    int commit() { return g_stage.ensure(cv.off + 256); }
    template <typename T> T* ptr(size_t k) const { return (T*)(g_stage.base + offs[k]); }
};

inline cudaError_t h2d(void* d, const void* h, size_t n) { return cudaMemcpy(d, h, n, cudaMemcpyHostToDevice); }
inline cudaError_t d2h(void* h, const void* d, size_t n) { return cudaMemcpy(h, d, n, cudaMemcpyDeviceToHost); }

}  // namespace

extern "C" double bhmm_b200_forward(double* alpha, const double* A, const double* pobs, const double* pi, int N,
                                    int T)
{
    clear_error();
    if (require_device()) return NAN;
    if (N < 1 || T < 1) { bhmm_set_error(BHMM_ERR_INVALID, "N and T must be positive"); return NAN; }
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N;
    const size_t kA = s.add(sizeof(double) * N * N), kpi = s.add(sizeof(double) * N), kp = s.add(tn), ka = s.add(tn);
    if (s.commit()) { bhmm_set_error(BHMM_ERR_NO_MEM, "device memory"); return NAN; }
    if (h2d(s.ptr<double>(kA), A, sizeof(double) * N * N) || h2d(s.ptr<double>(kpi), pi, sizeof(double) * N) ||
        h2d(s.ptr<double>(kp), pobs, tn)) { bhmm_set_error(BHMM_ERR_CUDA, "H2D copy failed"); return NAN; }
    double ll = NAN;
    if (bhmm_b200_forward_dev(s.ptr<double>(ka), s.ptr<double>(kA), s.ptr<double>(kp), s.ptr<double>(kpi), N, T, &ll,
                              nullptr))
        return NAN;
    if (d2h(alpha, s.ptr<double>(ka), tn)) { bhmm_set_error(BHMM_ERR_CUDA, "D2H copy failed"); return NAN; }
    return ll;
}

extern "C" void bhmm_b200_backward(double* beta, const double* A, const double* pobs, int N, int T)
{
    clear_error();
    if (require_device()) return;
    if (N < 1 || T < 1) { bhmm_set_error(BHMM_ERR_INVALID, "N and T must be positive"); return; }
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N;
    const size_t kA = s.add(sizeof(double) * N * N), kp = s.add(tn), kb = s.add(tn);
    if (s.commit()) { bhmm_set_error(BHMM_ERR_NO_MEM, "device memory"); return; }
    if (h2d(s.ptr<double>(kA), A, sizeof(double) * N * N) || h2d(s.ptr<double>(kp), pobs, tn)) {
        bhmm_set_error(BHMM_ERR_CUDA, "H2D copy failed");
        return;
    }
    if (bhmm_b200_backward_dev(s.ptr<double>(kb), s.ptr<double>(kA), s.ptr<double>(kp), N, T, nullptr)) return;
    if (d2h(beta, s.ptr<double>(kb), tn)) bhmm_set_error(BHMM_ERR_CUDA, "D2H copy failed");
}

extern "C" int bhmm_b200_state_probabilities(double* gamma, const double* alpha, const double* beta, int N, int T)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N;
    const size_t ka = s.add(tn), kb = s.add(tn), kg = s.add(tn);
    RC_TRY(s.commit());
    CUDA_TRY(h2d(s.ptr<double>(ka), alpha, tn));
    CUDA_TRY(h2d(s.ptr<double>(kb), beta, tn));
    RC_TRY(bhmm_b200_state_probabilities_dev(s.ptr<double>(kg), s.ptr<double>(ka), s.ptr<double>(kb), N, T, nullptr));
    CUDA_TRY(d2h(gamma, s.ptr<double>(kg), tn));
    return BHMM_OK;
}

extern "C" int bhmm_b200_state_counts(double* counts, const double* gamma, int N, int T)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N;
    const size_t kg = s.add(tn), kc = s.add(sizeof(double) * N);
    RC_TRY(s.commit());
    CUDA_TRY(h2d(s.ptr<double>(kg), gamma, tn));
    RC_TRY(bhmm_b200_state_counts_dev(s.ptr<double>(kc), s.ptr<double>(kg), N, T, nullptr));
    CUDA_TRY(d2h(counts, s.ptr<double>(kc), sizeof(double) * N));
    return BHMM_OK;
}

extern "C" int bhmm_b200_transition_counts(double* C, const double* A, const double* pobs, const double* alpha,
                                           const double* beta, int N, int T)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N, nn = sizeof(double) * (size_t)N * N;
    const size_t kA = s.add(nn), kp = s.add(tn), ka = s.add(tn), kb = s.add(tn), kC = s.add(nn);
    RC_TRY(s.commit());
    CUDA_TRY(h2d(s.ptr<double>(kA), A, nn));
    CUDA_TRY(h2d(s.ptr<double>(kp), pobs, tn));
    CUDA_TRY(h2d(s.ptr<double>(ka), alpha, tn));
    CUDA_TRY(h2d(s.ptr<double>(kb), beta, tn));
    RC_TRY(bhmm_b200_transition_counts_dev(s.ptr<double>(kC), s.ptr<double>(kA), s.ptr<double>(kp), s.ptr<double>(ka),
                                           s.ptr<double>(kb), N, T, nullptr));
    CUDA_TRY(d2h(C, s.ptr<double>(kC), nn));
    return BHMM_OK;
}

extern "C" int bhmm_b200_viterbi(int* path, const double* A, const double* pobs, const double* pi, int N, int T)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N, nn = sizeof(double) * (size_t)N * N;
    const size_t kA = s.add(nn), kpi = s.add(sizeof(double) * N), kp = s.add(tn), kpath = s.add(sizeof(int) * (size_t)T);
    RC_TRY(s.commit());
    CUDA_TRY(h2d(s.ptr<double>(kA), A, nn));
    CUDA_TRY(h2d(s.ptr<double>(kpi), pi, sizeof(double) * N));
    CUDA_TRY(h2d(s.ptr<double>(kp), pobs, tn));
    RC_TRY(bhmm_b200_viterbi_dev(s.ptr<int>(kpath), s.ptr<double>(kA), s.ptr<double>(kp), s.ptr<double>(kpi), N, T,
                                 nullptr));
    CUDA_TRY(d2h(path, s.ptr<int>(kpath), sizeof(int) * (size_t)T));
    return BHMM_OK;
}

extern "C" int bhmm_b200_sample_path_u(int* path, const double* alpha, const double* A, const double* u, int N,
                                       int T)
{
    clear_error();
    RC_TRY(require_device());
    if (N < 1 || T < 1) { bhmm_set_error(BHMM_ERR_INVALID, "N and T must be positive"); return BHMM_ERR_INVALID; }
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N, nn = sizeof(double) * (size_t)N * N;
    const size_t kA = s.add(nn), ka = s.add(tn), ku = s.add(sizeof(double) * (size_t)T),
                 kpath = s.add(sizeof(int) * (size_t)T);
    RC_TRY(s.commit());
    std::vector<double> urow(T);
    for (int t = 0; t < T; ++t) urow[t] = u[T - 1 - t];       // draw k belongs to frame T-1-k (_hidden.c:356-372)
    CUDA_TRY(h2d(s.ptr<double>(kA), A, nn));
    CUDA_TRY(h2d(s.ptr<double>(ka), alpha, tn));
    CUDA_TRY(h2d(s.ptr<double>(ku), urow.data(), sizeof(double) * (size_t)T));
    RC_TRY(bhmm_b200_sample_path_dev(s.ptr<int>(kpath), s.ptr<double>(ka), s.ptr<double>(kA), s.ptr<double>(ku), N, T,
                                     nullptr));
    CUDA_TRY(d2h(path, s.ptr<int>(kpath), sizeof(int) * (size_t)T));
    return BHMM_OK;
}

extern "C" int bhmm_b200_sample_path(int* path, const double* alpha, const double* A, const double* pobs, int N,
                                     int T)
{
    (void)pobs;   // unused by the reference as well (_hidden.c:330-378)
    if (T < 1) { bhmm_set_error(BHMM_ERR_INVALID, "T must be positive"); return BHMM_ERR_INVALID; }
    std::vector<double> u(T);
    {
        std::lock_guard<std::mutex> lk(g_lit_mutex);
        for (int k = 0; k < T; ++k) u[k] = g_rand.uniform();
    }
    return bhmm_b200_sample_path_u(path, alpha, A, u.data(), N, T);
}

extern "C" int bhmm_b200_gaussian_p_obs_outliers(const double* o, const double* mus, const double* sigmas, int N,
                                                 int T, int ignore_outliers, double* p)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N;
    const size_t ko = s.add(sizeof(double) * (size_t)T), km = s.add(sizeof(double) * N), ks = s.add(sizeof(double) * N),
                 kp = s.add(tn);
    RC_TRY(s.commit());
    CUDA_TRY(h2d(s.ptr<double>(ko), o, sizeof(double) * (size_t)T));
    CUDA_TRY(h2d(s.ptr<double>(km), mus, sizeof(double) * N));
    CUDA_TRY(h2d(s.ptr<double>(ks), sigmas, sizeof(double) * N));
    RC_TRY(bhmm_b200_gaussian_p_obs_dev(s.ptr<double>(ko), s.ptr<double>(km), s.ptr<double>(ks), N, T, ignore_outliers,
                                        s.ptr<double>(kp), nullptr));
    CUDA_TRY(d2h(p, s.ptr<double>(kp), tn));
    return BHMM_OK;
}

extern "C" void bhmm_b200_gaussian_p_obs(const double* o, const double* mus, const double* sigmas, int N, int T,
                                         double* p)
{
    bhmm_b200_gaussian_p_obs_outliers(o, mus, sigmas, N, T, 0, p);
}

extern "C" int bhmm_b200_discrete_p_obs(const int* obs, const double* B, int N, int M, int T, int ignore_outliers,
                                        double* p)
{
    clear_error();
    RC_TRY(require_device());
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N;
    const size_t ko = s.add(sizeof(int) * (size_t)T), kB = s.add(sizeof(double) * (size_t)N * M), kp = s.add(tn);
    RC_TRY(s.commit());
    CUDA_TRY(h2d(s.ptr<int>(ko), obs, sizeof(int) * (size_t)T));
    CUDA_TRY(h2d(s.ptr<double>(kB), B, sizeof(double) * (size_t)N * M));
    RC_TRY(bhmm_b200_discrete_p_obs_dev(s.ptr<int>(ko), s.ptr<double>(kB), N, M, T, ignore_outliers, s.ptr<double>(kp),
                                        nullptr));
    CUDA_TRY(d2h(p, s.ptr<double>(kp), tn));
    return BHMM_OK;
}

extern "C" void bhmm_b200_discrete_update_pout(const int* obs, const double* weights, int T, int N, int M,
                                               double* pout)
{
    clear_error();
    if (require_device()) return;
    std::lock_guard<std::mutex> lk(g_stage_mutex);
    Stage s;
    const size_t tn = sizeof(double) * (size_t)T * N, nm = sizeof(double) * (size_t)N * M;
    const size_t ko = s.add(sizeof(int) * (size_t)T), kw = s.add(tn), kp = s.add(nm);
    if (s.commit()) { bhmm_set_error(BHMM_ERR_NO_MEM, "device memory"); return; }
    if (h2d(s.ptr<int>(ko), obs, sizeof(int) * (size_t)T) || h2d(s.ptr<double>(kw), weights, tn) ||
        h2d(s.ptr<double>(kp), pout, nm)) { bhmm_set_error(BHMM_ERR_CUDA, "H2D copy failed"); return; }
    launch_update_pout(s.ptr<int>(ko), s.ptr<double>(kw), T, N, M, s.ptr<double>(kp), nullptr);
    LAUNCHED(1);
    if (finish(nullptr)) return;
    if (d2h(pout, s.ptr<double>(kp), nm)) bhmm_set_error(BHMM_ERR_CUDA, "D2H copy failed");
}

// ------------------------------------------------------------------------------------------------
// M-step on the device (SURVEY 8f N1): the reduced statistics never leave the GPU except as the updated parameters.
// ------------------------------------------------------------------------------------------------
extern "C" int bhmm_b200_mstep_dev(const double* d_stats, const double* d_means_old, int N, double mincount, double* d_out,
                                   void* stream)
{
    clear_error();
    if (!d_stats || !d_out || N < 1) { bhmm_set_error(BHMM_ERR_INVALID, "mstep: null pointer or N < 1"); return BHMM_ERR_INVALID; }
    RC_TRY(require_device());
    RC_TRY(launch_mstep_hmm(d_stats, d_means_old, N, d_means_old != nullptr, mincount, d_out, (cudaStream_t)stream));
    LAUNCHED(1);
    CUDA_TRY(cudaGetLastError());
    return BHMM_OK;
}

extern "C" int bhmm_b200_mstep_discrete_dev(const double* d_Bnum, int N, int M, double* d_B, double* d_Bt, void* stream)
{
    clear_error();
    if (!d_Bnum || !d_B || N < 1 || M < 1) { bhmm_set_error(BHMM_ERR_INVALID, "mstep_discrete: null pointer or empty shape"); return BHMM_ERR_INVALID; }
    RC_TRY(require_device());
    RC_TRY(launch_mstep_rows(d_Bnum, N, M, d_B, d_Bt, (cudaStream_t)stream));
    LAUNCHED(1);
    CUDA_TRY(cudaGetLastError());
    return BHMM_OK;
}

// ------------------------------------------------------------------------------------------------
// Synthetic trajectories (generate_synthetic_*, bhmm/hmm/generic_hmm.py:433-589): hidden states by exact time-parallel
// forward simulation (sample_kernels.cu:k_gen_*), observations frame-parallel from the states.
// ------------------------------------------------------------------------------------------------
static int gen_fail(int code, const char* msg)
{
    bhmm_set_error(code, msg);
    return code;
}

// Cumulative table of one distribution: sequential float64 sums (what np.cumsum computes), every entry from the last
// positive probability on set to exactly 1.0.  False when p is not a probability vector.
static bool cumulative_row(const double* p, int n, double* cum)
{
    double c = 0.0;
    int last = -1;
    for (int i = 0; i < n; ++i) {
        if (!(p[i] >= 0.0) || !std::isfinite(p[i])) return false;
        c += p[i];
        cum[i] = c;
        if (p[i] > 0.0) last = i;
    }
    if (last < 0 || std::fabs(c - 1.0) > 1e-6) return false;
    for (int i = last; i < n; ++i) cum[i] = 1.0;
    return true;
}

static int gen_check(const long long* offsets, int K, int N, int segment)
{
    if (!offsets || K < 1 || N < 1 || segment < 0) return gen_fail(BHMM_ERR_INVALID, "generate: bad offsets, K, N or segment");
    if (N > 256) return gen_fail(BHMM_ERR_UNSUPPORTED, "generate: at most 256 hidden states (uint8 segment maps)");
    if (offsets[0] != 0) return gen_fail(BHMM_ERR_INVALID, "generate: offsets[0] must be 0");
    for (int k = 0; k < K; ++k) {
        const long long T = offsets[k + 1] - offsets[k];
        if (T < 1) return gen_fail(BHMM_ERR_INVALID, "generate: every trajectory needs at least one frame");
        if (T > 2147483647LL) return gen_fail(BHMM_ERR_INVALID, "generate: trajectories must be shorter than 2^31 frames");
    }
    return BHMM_OK;
}

// Segment length of a call.  Trajectories that fill the GPU on their own (at least two warps per SM for every warp of
// map work a segment would need) run as one segment each: replay alone, the serial generator.  Otherwise segments are cut
// so that there are about as many as the SMs hold 1024 threads, i.e. a few waves of map warps and replay threads.
static int gen_segment_len(const long long* offsets, int K, int N, int segment, bool* whole, long long* nseg)
{
    long long maxT = 0;
    for (int k = 0; k < K; ++k) maxT = std::max(maxT, offsets[k + 1] - offsets[k]);
    long long L = segment;
    if (L <= 0) {
        int sms = 148, dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
            { cudaGetLastError(); sms = 148; }
        const int W = (N + 31) / 32;
        if ((long long)K * W >= 64LL * sms) L = maxT;
        else L = std::max<long long>(32, (offsets[K] + 1024LL * sms - 1) / (1024LL * sms));
    }
    L = std::min(L, maxT);
    *whole = (L >= maxT);
    long long n = 0;
    for (int k = 0; k < K; ++k) n += (offsets[k + 1] - offsets[k] + L - 1) / L;
    *nseg = n;
    return (int)L;
}

struct GenLayout {
    size_t row0, len, t0, T, start, map, enter, cum, bytes;
};

static GenLayout gen_layout(long long nseg, int N, bool whole)
{
    GenLayout g;
    Carver cv;
    g.row0 = cv.add<long long>(nseg);
    g.len = cv.add<int>(nseg);
    g.t0 = cv.add<int>(nseg);
    g.T = cv.add<int>(nseg);
    g.start = cv.add<int>(nseg);
    g.map = cv.add<unsigned char>(whole ? 0 : (size_t)nseg * N);
    g.enter = cv.add<int>(whole ? 0 : nseg);
    g.cum = cv.add<double>((size_t)N + (size_t)N * N);
    g.bytes = cv.off + 256;                  // the base is aligned up to 256 bytes
    return g;
}

extern "C" size_t bhmm_b200_generate_workspace_bytes(const long long* offsets, int K, int N, int segment)
{
    if (gen_check(offsets, K, N, segment) != BHMM_OK) return 0;
    bool whole;
    long long nseg;
    gen_segment_len(offsets, K, N, segment, &whole, &nseg);
    if (nseg > 2147483647LL) return 0;
    return gen_layout(nseg, N, whole).bytes;
}

extern "C" int bhmm_b200_generate_states(int* d_states, const long long* offsets, int K, int N, const double* A,
                                         const double* p0, const int* start, unsigned long long seed, int segment,
                                         void* d_workspace, size_t bytes, void* stream)
{
    clear_error();
    RC_TRY(gen_check(offsets, K, N, segment));
    if (!d_states || !A || (!p0 && !start)) return gen_fail(BHMM_ERR_INVALID, "generate: null states, A or initial distribution");
    std::vector<double> cum((size_t)N + (size_t)N * N, 1.0);
    if (!start && !cumulative_row(p0, N, cum.data()))
        return gen_fail(BHMM_ERR_INVALID, "generate: the initial distribution is not a probability vector");
    for (int i = 0; i < N; ++i)
        if (!cumulative_row(A + (size_t)i * N, N, cum.data() + N + (size_t)i * N))
            return gen_fail(BHMM_ERR_INVALID, "generate: the transition matrix is not row-stochastic");
    if (start)
        for (int k = 0; k < K; ++k)
            if (start[k] < 0 || start[k] >= N) return gen_fail(BHMM_ERR_INVALID, "generate: start state out of range");
    bool whole;
    long long nseg;
    const int L = gen_segment_len(offsets, K, N, segment, &whole, &nseg);
    if (nseg > 2147483647LL) return gen_fail(BHMM_ERR_INVALID, "generate: too many segments (use a longer segment)");
    const GenLayout g = gen_layout(nseg, N, whole);
    if (!d_workspace || bytes < g.bytes) return gen_fail(BHMM_ERR_INVALID, "generate: workspace smaller than bhmm_b200_generate_workspace_bytes");
    RC_TRY(require_device());
    // segments of every trajectory in reversed time order, t0 counted from the trajectory's end (sample_kernels.cu:k_gen_map)
    HostPlan p;
    build_plan(offsets, K, L, p);
    std::vector<long long> row0(p.n);
    std::vector<int> len(p.n), t0r(p.n), T(p.n), sst(p.n, -1);
    int c = 0;
    for (int k = 0; k < K; ++k)
        for (int q = p.last_chain[k]; q >= p.first_chain[k]; --q, ++c) {
            row0[c] = p.row0[q];
            len[c] = p.len[q];
            T[c] = p.T[q];
            t0r[c] = p.T[q] - p.t0[q] - p.len[q];
            if (start && p.t0[q] == 0) sst[c] = start[k];
        }
    char* base = (char*)(((uintptr_t)d_workspace + 255) & ~(uintptr_t)255);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(base + g.row0, row0.data(), sizeof(long long) * p.n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(base + g.len, len.data(), sizeof(int) * p.n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(base + g.t0, t0r.data(), sizeof(int) * p.n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(base + g.T, T.data(), sizeof(int) * p.n, cudaMemcpyHostToDevice, st));
    if (start) CUDA_TRY(cudaMemcpyAsync(base + g.start, sst.data(), sizeof(int) * p.n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(base + g.cum, cum.data(), sizeof(double) * cum.size(), cudaMemcpyHostToDevice, st));
    Chains seg{};
    seg.row0 = (const long long*)(base + g.row0);
    seg.len = (const int*)(base + g.len);
    seg.t0 = (const int*)(base + g.t0);
    seg.T = (const int*)(base + g.T);
    seg.n = p.n;
    const double* d_cum = (const double*)(base + g.cum);
    RC_TRY(launch_generate_states(seg, N, d_cum, d_cum + N, start ? (const int*)(base + g.start) : nullptr, seed, whole,
                                  (unsigned char*)(base + g.map), (int*)(base + g.enter), d_states, st));
    LAUNCHED(whole ? 1 : 3);
    return finish(st);
}

// small host parameters of an emission call go to the literal API's arena; a state outside [0, N) is reported, not read
static int emit_run(const std::vector<double>& params, cudaStream_t st,
                    const std::function<int(const double* d_params, int* d_err)>& launch)
{
    std::lock_guard<std::mutex> lk(g_lit_mutex);
    Carver cv;
    const size_t o_p = cv.add<double>(params.size());
    const size_t o_err = cv.add<int>(1);
    RC_TRY(g_lit_arena.ensure(cv.off + 256));
    char* base = g_lit_arena.base;
    CUDA_TRY(cudaMemcpyAsync(base + o_p, params.data(), sizeof(double) * params.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(base + o_err, 0, sizeof(int), st));
    RC_TRY(launch((const double*)(base + o_p), (int*)(base + o_err)));
    LAUNCHED(1);
    int err = 0;
    CUDA_TRY(cudaMemcpyAsync(&err, base + o_err, sizeof(int), cudaMemcpyDeviceToHost, st));
    RC_TRY(finish(st));
    if (err) return gen_fail(BHMM_ERR_INVALID, "emit: a state is out of range [0, N)");
    return BHMM_OK;
}

extern "C" int bhmm_b200_emit_gaussian(double* d_obs, const int* d_states, long long rows, int N, const double* means,
                                       const double* sigmas, unsigned long long seed, void* stream)
{
    clear_error();
    if (rows < 0 || N < 1 || !means || !sigmas || (rows > 0 && (!d_obs || !d_states)))
        return gen_fail(BHMM_ERR_INVALID, "emit_gaussian: bad arguments");
    std::vector<double> params(2 * (size_t)N);
    for (int i = 0; i < N; ++i) {
        if (!std::isfinite(means[i]) || !std::isfinite(sigmas[i]) || !(sigmas[i] >= 0.0))
            return gen_fail(BHMM_ERR_INVALID, "emit_gaussian: means must be finite, sigmas finite and >= 0");
        params[i] = means[i];
        params[N + i] = sigmas[i];
    }
    RC_TRY(require_device());
    if (rows == 0) return BHMM_OK;
    cudaStream_t st = (cudaStream_t)stream;
    return emit_run(params, st, [&](const double* d_p, int* d_err) {
        return launch_emit_gaussian(d_states, rows, N, d_p, d_p + N, seed, d_obs, d_err, st);
    });
}

extern "C" int bhmm_b200_emit_discrete(int* d_obs, const int* d_states, long long rows, int N, int M, const double* B,
                                       unsigned long long seed, void* stream)
{
    clear_error();
    if (rows < 0 || N < 1 || M < 1 || !B || (rows > 0 && (!d_obs || !d_states)))
        return gen_fail(BHMM_ERR_INVALID, "emit_discrete: bad arguments");
    std::vector<double> cumB((size_t)N * M);
    for (int i = 0; i < N; ++i)
        if (!cumulative_row(B + (size_t)i * M, M, cumB.data() + (size_t)i * M))
            return gen_fail(BHMM_ERR_INVALID, "emit_discrete: the output matrix is not row-stochastic");
    RC_TRY(require_device());
    if (rows == 0) return BHMM_OK;
    cudaStream_t st = (cudaStream_t)stream;
    return emit_run(cumB, st, [&](const double* d_cumB, int* d_err) {
        return launch_emit_discrete(d_states, rows, N, M, d_cumB, seed, d_obs, d_err, st);
    });
}
