// trpl_ensemble.cuh -- the two kernels of the ensemble sampler (include/trpl_b200_ensemble.h): stretch-move
// proposals and the accept/reject step.  One thread per walker; a few thousand walkers per launch, so both
// are latency-bound and cost next to nothing beside the solve between them (DESIGN.md §5b).
#pragma once
#include "trpl_aux_kernels.cuh"

namespace trpl {

constexpr unsigned TAG_PROPOSE = 1, TAG_ACCEPT = 2;     // counter word 3; trpl_random_grid uses 0

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

// d_comp column-major: column j of complement walker k at comp[j * ld_comp + k]
__global__ void trpl_stretch_propose_kernel(const double *x, long long n, long long ldx, unsigned long long first,
                                            const double *comp, long long ld_comp, long long nc, const GridArgs ga,
                                            int d, double a, unsigned long long seed, unsigned step, double *y,
                                            long long ldy, double *logq)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long g = first + (unsigned long long)i;
        unsigned r[4];
        philox4x32_10((unsigned)g, (unsigned)(g >> 32), step, TAG_PROPOSE, (unsigned)seed, (unsigned)(seed >> 32), r);
        const long long p = (long long)__umul64hi(((unsigned long long)r[0] << 32) | r[1], (unsigned long long)nc);
        const double u = unit53(r[2], r[3]);
        // explicit FMAs: the rounding of every step is fixed, so a host mirror can reproduce proposals exactly
        const double t = fma(a - 1.0, u, 1.0);
        const double z = t * t / a;
        const double *xk = x + i * ldx;
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
        double *yk = y + i * ldy;
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
        logq[i] = inside ? (double)(d - 1) * log(z) : -INFINITY;
    }
}

__global__ void trpl_stretch_accept_kernel(double *x, long long n, long long ldx, unsigned long long first, int ncol,
                                           double *lnl, const double *y, long long ldy, const double *lnl_y,
                                           const double *logq, double temperature, unsigned long long seed,
                                           unsigned step, int *accepted)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long g = first + (unsigned long long)i;
        const double lx_raw = lnl[i], ly_raw = lnl_y[i], q = logq[i];
        const double lx = (lx_raw == lx_raw) ? lx_raw : -INFINITY;     // not converged -> -inf
        const double ly = (ly_raw == ly_raw) ? ly_raw : -INFINITY;
        bool acc;
        if (q == -INFINITY || ly == -INFINITY) acc = false;            // out of the box, or an impossible proposal
        else if (lx == -INFINITY) acc = true;
        else {
            unsigned r[4];
            philox4x32_10((unsigned)g, (unsigned)(g >> 32), step, TAG_ACCEPT, (unsigned)seed, (unsigned)(seed >> 32), r);
            const double u = unit53(r[0], r[1]) + (1.0 / 9007199254740992.0);     // (0, 1]
            acc = log(u) < q + (ly - lx) / temperature;
        }
        if (acc) {
            for (int j = 0; j < ncol; j++) x[i * ldx + j] = y[i * ldy + j];
            lnl[i] = ly_raw;
        }
        if (accepted) accepted[i] = acc ? 1 : 0;
    }
}

}  // namespace trpl
