// bhmm_b200/csrc/common.cuh -- shared definitions for the sm_100a HMM kernels.
//
// Vocabulary (follows the reference's domain, bhmm/hidden/api.py):
//   trajectory  one observation sequence of T frames
//   frame       one time step t of a trajectory; "row" = global frame index in the concatenated batch
//   chain       a contiguous range of frames of one trajectory that one team of threads walks
//               sequentially.  Long trajectories are cut into chains of `chunk` frames; a chain that
//               does not start at frame 0 is warmed up on the `warm` frames before it (the scaled
//               forward filter forgets its initial condition), and the hand-over is CERTIFIED
//               afterwards against the preceding chain's exact value (see certify.cu / DESIGN.md).
//   team        the threads that cooperate on one chain: thread j of a team owns hidden state j.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#define BHMM_OK 0
#define BHMM_ERR_INVALID 1
#define BHMM_ERR_NO_MEM 2      /* same value as _BHMM_ERR_NO_MEM, bhmm/hidden/impl_c/_hidden.h:5 */
#define BHMM_ERR_SAMPLE 3      /* _random_choice found no state (the reference calls exit(1), _hidden.c:299-304) */
#define BHMM_ERR_CUDA 4
#define BHMM_ERR_UNSUPPORTED 5
#define BHMM_ERR_NOT_CERTIFIED 6

// Emission source of a chain kernel.
//   EM_POBS  : p[t,j] read from a caller-supplied (T,N) table (the literal bhmm.hidden API)
//   EM_GAUSS : p[t,j] = N(o_t; mu_j, sigma_j)       (GaussianOutputModel.p_obs, _gaussian.c:5-21)
//   EM_DISC  : p[t,j] = B[j, o_t]                   (DiscreteOutputModel.p_obs, discrete.py:146-153)
enum { EM_POBS = 0, EM_GAUSS = 1, EM_DISC = 2 };

struct Emission {
    const double* pobs;     // EM_POBS : (rows, N) row-major
    const double* obs;      // EM_GAUSS: (rows)
    const int*    sym;      // EM_DISC : (rows) int32 symbols
    const double* mu;       // EM_GAUSS: (N)
    const double* sigma;    // EM_GAUSS: (N)
    const double* Bt;       // EM_DISC : (M, N) = B transposed, so one frame's N values are contiguous
    int M;
    int ignore_outliers;    // outlier rule of outputmodel.py:119-131 (rows that are all zero become all one)
};

// Chain table (struct of arrays, device memory).  Chains are ordered by (trajectory, start frame), so
// the chain that precedes chain c in time is c-1 whenever t0[c] > 0.
struct Chains {
    const long long* row0;  // global row of the chain's first frame
    const int* len;         // number of frames in the chain
    const int* t0;          // frame index (within its trajectory) of the chain's first frame
    const int* T;           // length of the trajectory the chain belongs to
    const int* list;        // optional indirection: run only chains list[0..n) (fix-up passes); may be NULL
    int n;                  // number of chains to run
    int warm;               // warm-up frames (used when warmv is NULL)
    const int* warmv;       // optional per-chain warm-up lengths, adapted by the certification (certify.cu)
    int exact;              // 1: fix-up pass, start from the recorded exact hand-over vector instead of warming up
    // optional per-chain starts of a time shard's E-step (engine.cu: border_setup), NULL elsewhere: chain c with gidx[c] >= 0
    // starts from the given border vector gvec + gidx[c] * N (forward: alpha at t0 - 1, backward: beta at t0 + len) instead
    // of a warm-up; gidx[c] == CHAIN_WARMS_UP marks a chain at the border of the owned range whose neighbour in the table is
    // not its neighbour in time, so that it keeps its warm-up in an exact pass too
    const int* gidx;
    const double* gvec;
};
constexpr int CHAIN_WARMS_UP = -2;

__device__ __forceinline__ bool chain_start_given(const Chains& ch, int c) { return ch.gidx != nullptr && ch.gidx[c] >= 0; }

// whether chain c starts from an exact vector (mode 2 of the chain kernels) rather than from pi or a warm-up
__device__ __forceinline__ bool chain_exact_start(const Chains& ch, int c)
{
    if (ch.gidx) {
        const int g = ch.gidx[c];
        return g >= 0 || (ch.exact && g != CHAIN_WARMS_UP);
    }
    return ch.exact != 0;
}

// Where an exact start of chain c is read: its given border start, else the end vector of its neighbour nb in hand_end
// (nb = c - 1 forward, c + 1 backward); rows of `stride` doubles.
__device__ __forceinline__ const double* chain_start_vec(const Chains& ch, const double* hand_end, int c, int nb, int stride)
{
    return chain_start_given(ch, c) ? ch.gvec + (long long)ch.gidx[c] * stride : hand_end + (long long)nb * stride;
}

__device__ __forceinline__ double gauss_pdf(double o, double mu, double sigma)
{
    // same expression tree as bhmm/output_models/impl_c/_gaussian.c:18-20
    const double norm = 1.0 / (sqrt(2.0 * 3.14159265358979323846) * sigma);
    const double z = (o - mu) / sigma;
    return norm * exp(-0.5 * z * z);
}

// Relative mismatch of two hand-over vectors, component-wise: |a-b| / max(|a|,|b|), 0 when both are 0.
// Component-wise RELATIVE agreement is what makes the certification rigorous: the normalised filter
// map is non-expansive in Hilbert's projective metric, so a relative error eps at the hand-over bounds
// the relative error of every later frame of the chain by (about) eps.
__device__ __forceinline__ double rel_mismatch(double a, double b)
{
    const double m = fmax(fabs(a), fabs(b));
    if (m == 0.0) return 0.0;
    const double d = fabs(a - b) / m;
    return (d == d) ? d : 1.0;   // NaN counts as a full mismatch
}

#define CUDA_TRY(expr)                                                        \
    do {                                                                      \
        cudaError_t e_ = (expr);                                              \
        if (e_ != cudaSuccess) { bhmm_set_error(BHMM_ERR_CUDA, cudaGetErrorString(e_)); return BHMM_ERR_CUDA; } \
    } while (0)

void bhmm_set_error(int code, const char* msg);
void bhmm_note_error(int code, const char* where);
