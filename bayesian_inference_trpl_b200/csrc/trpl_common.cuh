// trpl_common.cuh -- argument structs shared by host and device code, and small device helpers.
// Part of libtrpl_b200.so (see include/trpl_b200.h and trpl_kernels.cu for the overview).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <float.h>
#include <limits.h>
#include <stdio.h>

#include "trpl_b200.h"

namespace trpl {


constexpr unsigned FULL = 0xffffffffu;
constexpr int WARPS_PER_CTA = 4;      // warp kernel: one simulation per warp
constexpr int MIN_CTAS_PER_SM = 4;    // its __launch_bounds__ occupancy target (16 warps per SM)

// The solver's design choices (pivot scheme per kernel family, constant table, B-only last PCR stage)
// are fixed in the code; the measurements behind them are in profiles/r02_variants.txt.  The only
// build flag that selects other code is TRPL_DEBUG.
//
// -DTRPL_DEBUG=1: the sanitizer substitute (compute-sanitizer is closed on the pool this was developed on):
// device-side bounds checks on every ring slot, observation index and exchange-buffer row, and a canary
// word behind each warp's ring that is verified after every simulation.  A violation prints the site and
// traps, which surfaces as TRPL_ECUDA on the host.  tests: run the GPU suite with TRPL_LIB pointing at the
// debug build (tools/build_variants.py debug:-DTRPL_DEBUG=1; log in profiles/r02_debug_build_suite.txt).
#ifndef TRPL_DEBUG
#define TRPL_DEBUG 0
#endif
#if TRPL_DEBUG
#define TRPL_DASSERT(cond)                                                                      \
    do {                                                                                        \
        if (!(cond)) {                                                                          \
            printf("TRPL_DEBUG violation %s at %s:%d (block %d thread %d)\n", #cond, __FILE__, \
                   __LINE__, (int)blockIdx.x, (int)threadIdx.x);                                \
            __trap();                                                                           \
        }                                                                                       \
    } while (0)
#else
#define TRPL_DASSERT(cond) do { } while (0)
#endif
constexpr int RING_CANARY = TRPL_DEBUG ? 2 : 0;        // doubles appended to each warp's ring
constexpr unsigned long long CANARY_WORD = 0x5452504C43414E41ULL;   // "TRPLCANA"

struct ObsDev {
    int n;
    int pad_;
    const int *hi;
    const double *whi;
    const double *wlo;
    const double *val;
};

struct CurveDev {
    double scales[TRPL_NPAR];
    double init_mul;      // dx^3, or 1 when the profile is already in grid units
    double redim;         // dx^2 * dt                         (pvSimPCR.py:393)
    const double *init;   // [L]
    void *pl_out;         // row base for sample 0, or nullptr
    int t_last;           // last time index to integrate to (<= T)
    int pad_;
    ObsDev obs[TRPL_MAX_EXP];
};

struct KArgs {
    const double *x;
    long long ldx;
    long long S;
    long long pl_stride;
    double TOL;
    double *sse;                 // [E][C][S] or nullptr
    int *status;                 // [C][S] or nullptr
    long long *iters;            // [C][S] or nullptr
    unsigned long long *counter; // work-item counter (zeroed by the host)
    int mag_col;                 // < 0: no magnitude offset
    int C, E, L, plT, max_iter, max_order, flags, pl_dtype;
    int curve_order[TRPL_MAX_CURVES];   // curves sorted by decreasing work (longest first)
    CurveDev curves[TRPL_MAX_CURVES];
};

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double rcp64(double x)
{
    // MUFU.RCP64H seed (rel. error <= 1e-6, measured on B200 with tools/microbench.cu) followed by
    // one cubically convergent step r*(1 + e + e^2): max error 1 ulp (2.2e-16, measured over 2^24
    // operands in four magnitude ranges).  No slow path: operands here are normal, finite and far
    // from the exponent limits.
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    e = fma(e, e, e);
    return fma(r, e, r);
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

__device__ __forceinline__ double sel(bool c, double a, double b) { return c ? a : b; }


}  // namespace trpl
