// tests/emu/panel_emu.cpp -- the panel kernels' SOURCE (bhmm_b200/csrc/panel_kernels.cu) compiled for the CPU on top of
// warp_emu.h, exported with a flat C interface for tests/test_panel_emulated_cpu.py and test_panel_family_emulated_cpu.py.
// Test infrastructure only.
//   g++ -O1 -std=c++17 -shared -fPIC -I/usr/local/cuda/include -o panel_emu.so panel_emu.cpp
#define PANEL_HOST_EMU 1            // asm (DMMA, prefetch) -> emulator hooks
#define PANEL_HOST_NO_LAUNCHERS 1   // no <<<>>> launchers, no CUDA runtime: the kernels are called directly below
#include "warp_emu.h"

#include <limits>
#include <vector>
// dynamic shared memory of the kernels that use it (wide2, k_viterbi_multi); NaN before every launch, so that a word read
// before the kernel wrote it shows up in the results (on the GPU it holds whatever the previous block left there)
namespace emu {
inline std::vector<double>& dyn_smem_buf() { static std::vector<double> b(1 << 16); return b; }
inline double* dyn_smem() { return dyn_smem_buf().data(); }
inline void poison_dyn_smem(size_t bytes)
{
    if (bytes > dyn_smem_buf().size() * sizeof(double)) { fprintf(stderr, "panel_emu: %zu bytes of shared memory\n", bytes); abort(); }
    std::fill(dyn_smem_buf().begin(), dyn_smem_buf().end(), std::numeric_limits<double>::quiet_NaN());
}
}  // namespace emu

#include "../../bhmm_b200/csrc/panel_kernels.cu"

namespace {

Chains make_chains(const long long* row0, const int* len, const int* t0, const int* T, const int* list, int n_run, int warm,
                   const int* warmv, int exact)
{
    Chains ch{};
    ch.row0 = row0; ch.len = len; ch.t0 = t0; ch.T = T; ch.list = list; ch.n = n_run; ch.warm = warm; ch.warmv = warmv;
    ch.exact = exact;
    return ch;
}

Emission make_emission(const double* pobs, const double* obs, const int* sym, const double* mu, const double* sigma,
                       const double* Bt, int M, int ignore_outliers)
{
    Emission em{};
    em.pobs = pobs; em.obs = obs; em.sym = sym; em.mu = mu; em.sigma = sigma; em.Bt = Bt; em.M = M;
    em.ignore_outliers = ignore_outliers;
    return em;
}

}  // namespace

static int g_force_wide = 0;     // N = 32 on the wide kernels (BHMM_B200_PANEL=2)
extern "C" void panel_emu_force_wide(int on) { g_force_wide = on; }
extern "C" int panel_emu_warps_per_block() { return PW; }
// chains per block of the wide forward kernel and per block and round of the wide backward kernel at N (0: N not served)
extern "C" int panel_emu_wide_cpb(int N) { return wide_tiles(N) ? wide_cpb(wide_tiles(N)) : 0; }
extern "C" int panel_emu_wide_cpb_bwd(int N) { return wide_tiles(N) ? wide_cpb_bwd(wide_tiles(N)) : 0; }

// the wide kernels as launch_forward_wide_em / launch_backward_wide_em dispatch them: the one-set kernels at NT = 4, the
// two-set kernels (wide2) at NT = 8 and 13 with the outlier machinery compiled in only when the rule is on
template <int EM, int NT, bool OUTL>
void forward_wide2(const FwdArgs& a, int grid)
{
    emu::poison_dyn_smem(wide2_forward_smem<NT, OUTL>());
    emu::launch(grid, NT * 32, [&] { k_forward_wide2<EM, NT, OUTL>(a); });
}

template <int EM>
void forward_wide(const FwdArgs& a, int NT, int grid)
{
    const bool outl = (EM != EM_POBS) && a.em.ignore_outliers;
    if (NT == 4) emu::launch(grid, 4 * 32, [&] { k_forward_wide<EM, 4>(a); });
    else if (NT == 8) outl ? forward_wide2<EM, 8, EM != EM_POBS>(a, grid) : forward_wide2<EM, 8, false>(a, grid);
    else outl ? forward_wide2<EM, 13, EM != EM_POBS>(a, grid) : forward_wide2<EM, 13, false>(a, grid);
}

template <int EM, int NT, bool OUTL>
void backward_wide2(const BwdArgs& a, int grid)
{
    constexpr bool BSM = NT > 8;
    constexpr int BWS = NT > 8 ? BWS13 : 2;
    emu::poison_dyn_smem(wide2_backward_smem<NT, OUTL, BSM, BWS>());
    emu::launch(grid, NT * 32, [&] { k_backward_stats_wide2<EM, NT, OUTL, BSM, BWS>(a); });
}

template <int EM>
void backward_wide(const BwdArgs& a, int NT, int grid)
{
    const bool outl = (EM != EM_POBS) && a.em.ignore_outliers;
    if (NT == 4) emu::launch(grid, 4 * 32, [&] { k_backward_stats_wide<EM, 4>(a); });
    else if (NT == 8) outl ? backward_wide2<EM, 8, EM != EM_POBS>(a, grid) : backward_wide2<EM, 8, false>(a, grid);
    else outl ? backward_wide2<EM, 13, EM != EM_POBS>(a, grid) : backward_wide2<EM, 13, false>(a, grid);
}

extern "C" int panel_emu_forward(int N, int em_kind, int grid, const long long* row0, const int* len, const int* t0, const int* T,
                                 const int* list, int n_run, int warm, const int* warmv, int exact, const double* pobs,
                                 const double* obs, const int* sym, const double* mu, const double* sigma, const double* Bt,
                                 int M, int ignore_outliers, const double* A, const double* pi, double* alpha,
                                 double* chain_ll, double* hand_used, double* hand_end)
{
    FwdArgs a{};
    a.ch = make_chains(row0, len, t0, T, list, n_run, warm, warmv, exact);
    a.em = make_emission(pobs, obs, sym, mu, sigma, Bt, M, ignore_outliers);
    a.N = N; a.A = A; a.pi = pi; a.alpha = alpha; a.chain_ll = chain_ll; a.hand_used = hand_used; a.hand_end = hand_end;
    if (N != PN || g_force_wide) {
        const int NT = wide_tiles(N);
        if (NT == 0) return 2;
        switch (em_kind) {
            case EM_POBS: forward_wide<EM_POBS>(a, NT, grid); return 0;
            case EM_GAUSS: forward_wide<EM_GAUSS>(a, NT, grid); return 0;
            case EM_DISC: forward_wide<EM_DISC>(a, NT, grid); return 0;
        }
        return 1;
    }
    switch (em_kind) {
        case EM_POBS: emu::launch(grid, PW * 32, [&] { k_forward_panel32<EM_POBS>(a); }); return 0;
        case EM_GAUSS: emu::launch(grid, PW * 32, [&] { k_forward_panel32<EM_GAUSS>(a); }); return 0;
        case EM_DISC: emu::launch(grid, PW * 32, [&] { k_forward_panel32<EM_DISC>(a); }); return 0;
    }
    return 1;
}

// partials: N = 32: (grid * PW, N*N + 4N), one row per warp; wide kernels: (grid, N*N + 4N), one row per block
extern "C" int panel_emu_backward_stats(int N, int em_kind, int grid, const long long* row0, const int* len, const int* t0,
                                        const int* T, const int* list, int n_run, int warm, const int* warmv, int exact,
                                        const double* pobs, const double* obs, const int* sym, const double* mu,
                                        const double* sigma, const double* Bt, int M, int ignore_outliers, const double* A,
                                        const double* alpha, double* gamma, double* Bnum, double* partials,
                                        double* hand_used, double* hand_end)
{
    BwdArgs a{};
    a.ch = make_chains(row0, len, t0, T, list, n_run, warm, warmv, exact);
    a.em = make_emission(pobs, obs, sym, mu, sigma, Bt, M, ignore_outliers);
    a.N = N; a.grid = (N == PN && !g_force_wide) ? grid * PW : grid; a.A = A; a.alpha = alpha; a.gamma = gamma; a.Bnum = Bnum; a.partials = partials;
    a.hand_used = hand_used; a.hand_end = hand_end;
    if (N != PN || g_force_wide) {
        const int NT = wide_tiles(N);
        if (NT == 0) return 2;
        switch (em_kind) {
            case EM_POBS: backward_wide<EM_POBS>(a, NT, grid); return 0;
            case EM_GAUSS: backward_wide<EM_GAUSS>(a, NT, grid); return 0;
            case EM_DISC: backward_wide<EM_DISC>(a, NT, grid); return 0;
        }
        return 1;
    }
    switch (em_kind) {
        case EM_POBS: emu::launch(grid, PW * 32, [&] { k_backward_stats_panel32<EM_POBS>(a); }); return 0;
        case EM_GAUSS: emu::launch(grid, PW * 32, [&] { k_backward_stats_panel32<EM_GAUSS>(a); }); return 0;
        case EM_DISC: emu::launch(grid, PW * 32, [&] { k_backward_stats_panel32<EM_DISC>(a); }); return 0;
    }
    return 1;
}

// Viterbi with the matrix column in registers (k_viterbi_regs, BHMM_B200_VITERBI_REGS=1); backptr: (rows, N) uint8 shifted back-pointer map (CHASE layout)
extern "C" int panel_emu_viterbi(int N, int em_kind, int grid, int K, const long long* offsets, const double* pobs,
                                 const double* obs, const int* sym, const double* mu, const double* sigma, const double* Bt,
                                 int M, int ignore_outliers, const double* A, const double* pi, unsigned char* backptr)
{
    VitArgs a{};
    a.em = make_emission(pobs, obs, sym, mu, sigma, Bt, M, ignore_outliers);
    a.N = N; a.K = K; a.offsets = offsets; a.A = A; a.pi = pi; a.backptr = backptr; a.path = nullptr;
    if (N <= 32 || N > 104) return 2;
#define VIT(EMK) \
    if (N <= 64) emu::launch(grid, 64, [&] { k_viterbi_regs<EMK, 64>(a); }); \
    else emu::launch(grid, 128, [&] { k_viterbi_regs<EMK, 104>(a); }); \
    return 0;
    switch (em_kind) {
        case EM_POBS: VIT(EM_POBS)
        case EM_GAUSS: VIT(EM_GAUSS)
        case EM_DISC: VIT(EM_DISC)
    }
    return 1;
}

// Viterbi with the matrix in shared memory and R trajectories per group (k_viterbi_multi, the default for 32 < N <= 104),
// shaped like launch_viterbi_regs_em: one group of sthr = 64 / 128 threads per block (the emulation has no named barriers)
extern "C" int panel_emu_viterbi_multi(int N, int em_kind, int grid, int K, const long long* offsets, const double* pobs,
                                       const double* obs, const int* sym, const double* mu, const double* sigma,
                                       const double* Bt, int M, int ignore_outliers, const double* A, const double* pi,
                                       unsigned char* backptr)
{
    VitArgs a{};
    a.em = make_emission(pobs, obs, sym, mu, sigma, Bt, M, ignore_outliers);
    a.N = N; a.K = K; a.offsets = offsets; a.A = A; a.pi = pi; a.backptr = backptr; a.path = nullptr;
    if (N <= 32 || N > 104) return 2;
    constexpr int R = VITERBI_MULTI_R;
    const int sthr = N <= 64 ? 64 : 128, NPS = (N + 1) & ~1, nsub = 1;
    emu::poison_dyn_smem(sizeof(double) * ((size_t)N * NPS + (size_t)nsub * (2 * (size_t)R * NPS + R + 2 * R)));
    switch (em_kind) {
        case EM_POBS: emu::launch(grid, nsub * sthr, [&] { k_viterbi_multi<EM_POBS, R>(a, NPS, sthr); }); return 0;
        case EM_GAUSS: emu::launch(grid, nsub * sthr, [&] { k_viterbi_multi<EM_GAUSS, R>(a, NPS, sthr); }); return 0;
        case EM_DISC: emu::launch(grid, nsub * sthr, [&] { k_viterbi_multi<EM_DISC, R>(a, NPS, sthr); }); return 0;
    }
    return 1;
}
extern "C" int panel_emu_viterbi_multi_r() { return VITERBI_MULTI_R; }

// Time-chunked Viterbi (N <= 32): chains with warm-up / exact starts; flagmap (rows): near-tie bits per row of the map
extern "C" int panel_emu_viterbi_chain(int N, int em_kind, int grid, const long long* row0, const int* len, const int* t0,
                                       const int* T, const int* list, int n_run, int warm, const int* warmv, int exact,
                                       const double* pobs, const double* obs, const int* sym, const double* mu,
                                       const double* sigma, const double* Bt, int M, int ignore_outliers, const double* A,
                                       const double* pi, unsigned char* backptr, double* hand_used, double* hand_end,
                                       unsigned* flagmap, double margin_min)
{
    VitChainArgs a{};
    a.ch = make_chains(row0, len, t0, T, list, n_run, warm, warmv, exact);
    a.em = make_emission(pobs, obs, sym, mu, sigma, Bt, M, ignore_outliers);
    a.N = N; a.A = A; a.pi = pi; a.backptr = backptr; a.hand_used = hand_used; a.hand_end = hand_end;
    a.flagmap = flagmap; a.margin_min = margin_min;
    switch (em_kind) {
        case EM_POBS: emu::launch(grid, PW * 32, [&] { k_viterbi_chain32<EM_POBS>(a); }); return 0;
        case EM_GAUSS: emu::launch(grid, PW * 32, [&] { k_viterbi_chain32<EM_GAUSS>(a); }); return 0;
        case EM_DISC: emu::launch(grid, PW * 32, [&] { k_viterbi_chain32<EM_DISC>(a); }); return 0;
    }
    return 1;
}

extern "C" int panel_emu_viterbi_path_flags(const unsigned* flagmap, const int* path, const long long* offsets, int K,
                                            long long rows)
{
    int counter = 0;
    emu::launch(2, 256, [&] { k_viterbi_path_flags(flagmap, path, offsets, K, rows, &counter); });
    return counter;
}
