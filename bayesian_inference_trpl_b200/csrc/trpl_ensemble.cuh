// trpl_ensemble.cuh -- the kernels of the ensemble sampler (include/trpl_b200_ensemble.h) and of its parallel
// tempering (include/trpl_b200_tempering.h): stretch-move proposals, the accept/reject step and the replica
// exchange between rungs.  One thread per walker (blockIdx.y = rung for the first two); a few thousand
// walkers per launch, so all three are latency-bound and cost next to nothing beside the solve between them
// (DESIGN.md §5b).
#pragma once
#include "trpl_aux_kernels.cuh"
#include "trpl_b200_tempering.h"

namespace trpl {

constexpr unsigned TAG_PROPOSE = 1, TAG_ACCEPT = 2, TAG_SWAP = TRPL_TAG_SWAP;   // counter word 3; trpl_random_grid uses 0

// The temperature ladder, passed by value (host array of the C ABI)
struct Ladder {
    int k;
    double t[TRPL_MAX_RUNGS];
};

// 53 random bits of two Philox words -> [0, 1)
__device__ __forceinline__ double unit53(unsigned hi, unsigned lo)
{
    return (double)((((unsigned long long)hi << 32) | lo) >> 11) * (1.0 / 9007199254740992.0);
}

// column j's source under the override flags (column 2 <- 3, 6 <- 5, 8 <- 7)
__device__ __forceinline__ int override_source(const GridArgs &ga, int j)
{
    if (ga.eq_mu && j == 2) return 3;
    if (ga.eq_s && j == 6) return 5;
    if (ga.eq_auger && j == 8) return 7;
    return j;
}

// Rung t = blockIdx.y: walkers x[(t n + i) ldx], complement rows t ncol .. of comp, column j of complement walker
// k at comp[j * ld_comp + k]; walker g = first + i of rung t draws from counter t W + g.
__global__ void trpl_stretch_propose_kernel(const double *x, long long n, long long ldx, unsigned long long first,
                                            unsigned long long W, const double *comp, long long ld_comp,
                                            long long nc, const GridArgs ga, int d, double a,
                                            unsigned long long seed, unsigned step, double *y, long long ldy,
                                            double *logq)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    const unsigned t = blockIdx.y;
    comp += (long long)t * ga.ncol * ld_comp;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long g = t * W + first + (unsigned long long)i;
        const long long row = t * n + i;
        unsigned r[4];
        philox4x32_10((unsigned)g, (unsigned)(g >> 32), step, TAG_PROPOSE, (unsigned)seed, (unsigned)(seed >> 32), r);
        const long long p = (long long)__umul64hi(((unsigned long long)r[0] << 32) | r[1], (unsigned long long)nc);
        const double u = unit53(r[2], r[3]);
        // explicit FMAs: the rounding of every step is fixed, so a host mirror can reproduce proposals exactly
        const double tz = fma(a - 1.0, u, 1.0);
        const double z = tz * tz / a;
        const double *xk = x + row * ldx;
        // pass 1: is the proposal inside the box (in prior coordinates; NaN counts as outside)?
        bool inside = true;
        for (int j = 0; j < ga.ncol; j++) {
            const double lo = ga.lo[j], hi = ga.hi[j];
            if (lo == hi || override_source(ga, j) != j) continue;
            const double xp = comp[j * ld_comp + p];
            double v;
            if (ga.do_log[j]) {
                const double tp = log10(xp);
                v = fma(z, log10(xk[j]) - tp, tp);
                inside = inside && v >= log10(lo) && v <= log10(hi);
            } else {
                v = fma(z, xk[j] - xp, xp);
                inside = inside && v >= lo && v <= hi;
            }
        }
        // pass 2: the row handed to the solver (the walker's own row when the proposal is out of the box)
        double *yk = y + row * ldy;
        for (int j = 0; j < ga.ncol; j++) {
            const int s = override_source(ga, j);
            double v = xk[s];
            if (inside && ga.lo[s] != ga.hi[s]) {
                const double xp = comp[s * ld_comp + p];
                if (ga.do_log[s]) {
                    const double tp = log10(xp);
                    v = exp10(fma(z, log10(xk[s]) - tp, tp));
                } else {
                    v = fma(z, xk[s] - xp, xp);
                }
            }
            yk[j] = v;
        }
        logq[row] = inside ? (double)(d - 1) * log(z) : -INFINITY;
    }
}

// Rung t = blockIdx.y at temperature lad.t[t]: rows, lnL and flags t n + i.
__global__ void trpl_stretch_accept_kernel(double *x, long long n, long long ldx, unsigned long long first,
                                           unsigned long long W, int ncol, double *lnl, const double *y,
                                           long long ldy, const double *lnl_y, const double *logq,
                                           const __grid_constant__ Ladder lad, unsigned long long seed,
                                           unsigned step, int *accepted)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    const unsigned t = blockIdx.y;
    const double temperature = lad.t[t];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long g = t * W + first + (unsigned long long)i;
        const long long row = t * n + i;
        const double lx_raw = lnl[row], ly_raw = lnl_y[row], q = logq[row];
        const double lx = (lx_raw == lx_raw) ? lx_raw : -INFINITY;     // not converged -> -inf
        const double ly = (ly_raw == ly_raw) ? ly_raw : -INFINITY;
        bool acc;
        if (q == -INFINITY || ly == -INFINITY) acc = false;            // out of the box, or an impossible proposal
        else if (lx == -INFINITY) acc = true;
        else {
            unsigned r[4];
            philox4x32_10((unsigned)g, (unsigned)(g >> 32), step, TAG_ACCEPT, (unsigned)seed, (unsigned)(seed >> 32), r);
            const double u = unit53(r[0], r[1]) + (1.0 / 9007199254740992.0);     // (0, 1]
            // a division, not a product with 1/T: rung 0 rounds like the untempered sampler, and T = inf gives 0
            acc = log(u) < q + (ly - lx) / temperature;
        }
        if (acc) {
            for (int j = 0; j < ncol; j++) x[row * ldx + j] = y[row * ldy + j];
            lnl[row] = ly_raw;
        }
        if (accepted) accepted[row] = acc ? 1 : 0;
    }
}

// Replica exchange of walker i between rungs t and t - 1, hottest pair first (include/trpl_b200_tempering.h).
__global__ void trpl_tempered_swap_kernel(double *x, long long n, long long ldx, unsigned long long first,
                                          unsigned long long W, int ncol, double *lnl,
                                          const __grid_constant__ Ladder lad, unsigned long long seed,
                                          unsigned step, int *swapped)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        for (int t = lad.k - 1; t >= 1; t--) {
            const long long hot = t * n + i, cold = hot - n;
            const double lh_raw = lnl[hot], lc_raw = lnl[cold];
            const double lh = (lh_raw == lh_raw) ? lh_raw : -INFINITY;
            const double lc = (lc_raw == lc_raw) ? lc_raw : -INFINITY;
            bool sw = false;
            if (lh != -INFINITY || lc != -INFINITY) {
                const double r = (1.0 / lad.t[t - 1] - 1.0 / lad.t[t]) * (lh - lc);
                if (r == INFINITY) sw = true;
                else if (r != -INFINITY) {                             // NaN r (+inf on both sides): no swap
                    const unsigned long long g = (unsigned long long)t * W + first + (unsigned long long)i;
                    unsigned q[4];
                    philox4x32_10((unsigned)g, (unsigned)(g >> 32), step, TAG_SWAP, (unsigned)seed,
                                  (unsigned)(seed >> 32), q);
                    sw = log(unit53(q[0], q[1]) + (1.0 / 9007199254740992.0)) < r;
                }
            }
            if (sw) {
                for (int j = 0; j < ncol; j++) {
                    const double v = x[hot * ldx + j];
                    x[hot * ldx + j] = x[cold * ldx + j];
                    x[cold * ldx + j] = v;
                }
                lnl[hot] = lc_raw;
                lnl[cold] = lh_raw;
            }
            if (swapped) swapped[cold] = sw ? 1 : 0;
        }
    }
}

}  // namespace trpl
