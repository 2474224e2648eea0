// tests/emu/cuda_fake.h -- the few device intrinsics warp_emu.h does not have yet, launch configuration and dynamic shared
// memory for hostified sources (hostify.py).  The fake CUDA runtime itself (cudaMalloc = malloc ...) is cuda_fake.cpp.
#pragma once
#include "warp_emu.h"

#undef __maxnreg__
#define __maxnreg__(...)

template <class T>
inline cudaError_t cudaFuncSetAttribute(T*, cudaFuncAttribute, int) { return cudaSuccess; }

namespace emu {
struct Cfg { int grid, block; size_t smem; };
inline Cfg cfg(int grid, int block, size_t smem = 0, cudaStream_t = 0) { return Cfg{grid, block, smem}; }
inline std::vector<double>& dyn_buf() { static std::vector<double> b; return b; }
inline double* dyn_smem() { return dyn_buf().data(); }
inline void launch(const Cfg& c, const std::function<void()>& body)
{
    dyn_buf().assign(c.smem / sizeof(double) + 2, 0.0);
    static const bool trace = getenv("EMU_TRACE") != nullptr;
    if (trace) fprintf(stderr, "emu launch: grid %d block %d smem %zu\n", c.grid, c.block, c.smem);
    launch(c.grid, c.block, body);
}
}  // namespace emu

inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { const unsigned long long o = *p; *p = o + v; return o; }
inline long long atomicAdd(long long* p, long long v) { const long long o = *p; *p = o + v; return o; }
inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v) { const unsigned long long o = *p; if (v > o) *p = v; return o; }
inline int atomicMax(int* p, int v) { const int o = *p; if (v > o) *p = v; return o; }
inline int atomicExch(int* p, int v) { const int o = *p; *p = v; return o; }
inline unsigned int __umulhi(unsigned int a, unsigned int b) { return (unsigned int)(((unsigned long long)a * b) >> 32); }
inline int __ffs(unsigned v) { return v ? __builtin_ctz(v) + 1 : 0; }
inline int __shfl_sync(unsigned, int v, int src)
{
    emu::Warp& w = emu::my_warp();
    w.si[emu::lane_id()] = v;
    emu::rendezvous(w.g);
    const int r = w.si[src & 31];
    emu::rendezvous(w.g);
    return r;
}
inline double __shfl_sync(unsigned, double v, int src)
{
    emu::Warp& w = emu::my_warp();
    w.sd[emu::lane_id()] = v;
    emu::rendezvous(w.g);
    const double r = w.sd[src & 31];
    emu::rendezvous(w.g);
    return r;
}
inline void __threadfence_block() {}
inline void __threadfence() {}

// the lane family (lane_kernels.cuh): constant-bank parameters, cache-hinted loads and stores, and its two warp collectives
#undef __grid_constant__
#define __grid_constant__
inline double __ldg(const double* p) { return *p; }
inline int __ldg(const int* p) { return *p; }
inline double2 __ldcs(const double2* p) { return *p; }
inline void __stcs(double2* p, double2 v) { *p = v; }
inline double __hiloint2double(int hi, int lo)
{
    const long long b = (long long)(((unsigned long long)(unsigned)hi << 32) | (unsigned)lo);
    double x;
    memcpy(&x, &b, 8);
    return x;
}
inline int __reduce_min_sync(unsigned, int v)
{
    emu::Warp& w = emu::my_warp();
    w.si[emu::lane_id()] = v;
    emu::rendezvous(w.g);
    int r = w.si[0];
    for (int i = 1; i < w.g.n; ++i) r = std::min(r, w.si[i]);
    emu::rendezvous(w.g);
    return r;
}
