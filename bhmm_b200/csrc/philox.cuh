// bhmm_b200/csrc/philox.cuh -- the library's counter-based random stream: Philox4x32-10 keyed by a 64-bit seed with a
// 128-bit counter (row, ctr), 53-bit uniforms and a Box-Muller normal from one block.  Used by the hidden-path sampler and
// the trajectory generator (sample_kernels.cu) and by the reversible transition-matrix sampler (tmatrix_kernels.cu);
// tests/generate_twin.py is its numpy restatement.
#pragma once
#include <stdint.h>

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

#ifdef PANEL_HOST_EMU
// the CPU emulation (tests/emu) has no cospi; its Gaussian draws are compared with a tolerance
inline double cospi(double x) { return cos(3.14159265358979323846 * x); }
#endif

// standard normal by Box-Muller on one block (seed, ctr, row): u1 in (0,1] from words 0-1, u2 in [0,1) from words 2-3
__device__ __forceinline__ double philox_normal(unsigned long long seed, unsigned long long ctr, long long row)
{
    uint32_t c0, c1, c2, c3;
    philox_block(seed, ctr, row, c0, c1, c2, c3);
    const double u1 = (double)(((((unsigned long long)c0 << 32) | c1) >> 11) + 1) * (1.0 / 9007199254740992.0);
    const double u2 = (double)((((unsigned long long)c2 << 32) | c3) >> 11) * (1.0 / 9007199254740992.0);
    return __dmul_rn(sqrt(-2.0 * log(u1)), cospi(2.0 * u2));
}

}  // namespace
