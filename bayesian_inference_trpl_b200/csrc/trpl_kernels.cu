// trpl_kernels.cu -- sm_100a kernels + C ABI of libtrpl_b200.so (see include/trpl_b200.h).
//
// Files: trpl_solver.cuh (hot path), trpl_aux_kernels.cuh (small kernels), trpl_common.cuh (argument
// structs, helpers), this file (host side + C ABI).
//
// Hot path replaced: pvSimPCR.py:14-401 (tEvol/iterate/pcreduce/norm2 + pvSim host driver) and
// probs.py:20-85 (kernel_lnP, log_kernel), plus the glue bayeslib.simulate runs between them
// (bayeslib.py:150-196).  Written from scratch for B200; nothing here is a translation of the
// numba kernels:
//
//   * one WARP owns one (sample, curve) simulation for its whole time integration; lane p holds
//     M consecutive grid nodes (L = 128 -> M = 4) of N, P, E and the BDF history sums in
//     REGISTERS; the four older BDF levels live in a lane-private shared-memory ring (no
//     barriers anywhere -- the reference round-trips the state through global memory every
//     step and needs ~50 __syncthreads per Newton iteration);
//   * each tridiagonal system is solved by a register-local Thomas sweep over the M-1 interior rows
//     of every lane (spike vectors to the two interface unknowns) + a 32-lane parallel cyclic reduction
//     on the interface unknowns done with warp shuffles (at most 5 normalised stages, cut short once
//     the off-diagonals are negligible, instead of the reference's log2(L)-1 shared-memory stages
//     over all L rows); fine grids (L > 256) run one CTA per simulation and hand the 32*W interface
//     rows to one warp (two block barriers per solve);
//   * the stop rule of both species is reduced together with one 2-value butterfly, division-free;
//   * PL(t) is a warp reduction; 32 consecutive PL values are staged one per lane and then
//     consumed together: written with one coalesced store (trpl_solve_pl) and/or turned into
//     log10, time-interpolated onto the observation times and accumulated into the squared
//     log-residual sum (trpl_solve_loglik) -- PL never goes to HBM on the fused path;
//   * warps fetch work items from a global atomic counter (persistent CTAs), so a slowly
//     converging sample never idles a wave.
//
// All arithmetic is FP64 like the reference (pvSimPCR.py:11,113-125).  Divisions are replaced by
// a Newton-refined reciprocal (MUFU.RCP64H seed), accurate to <= 1 ulp; see DESIGN.md.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "trpl_common.cuh"
#include "trpl_solver.cuh"
#include "trpl_aux_kernels.cuh"

using namespace trpl;

namespace {

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
thread_local char g_cuda_err[256] = "";

int cuda_fail(cudaError_t e, const char *what)
{
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
    return TRPL_ECUDA;
}
#define CK(call)                                                   \
    do {                                                           \
        cudaError_t e_ = (call);                                   \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call);        \
    } while (0)
// propagates a TRPL_E* code of a host helper
#define TRY(call)                                                  \
    do {                                                           \
        if (int rc_ = (call)) return rc_;                          \
    } while (0)

// pvSimPCR.py:327-331 (same expression order; pow() is glibc's, as in CPython)
void make_scales(double length, double time, int L, int T, double *sc, double *dx_o, double *dt_o)
{
    const double dx = length / L, dt = time / T;
    const double dx3 = pow(dx, 3.0);
    const double dtdx = dt / dx, dtdx2 = dtdx / dx, dtdx6 = dt / pow(dx, 6.0);
    sc[0] = dx3; sc[1] = dx3; sc[2] = dtdx2; sc[3] = dtdx2; sc[4] = dtdx2 / dx;
    sc[5] = dtdx; sc[6] = dtdx; sc[7] = dtdx6; sc[8] = dtdx6;
    sc[9] = 1.0 / dt; sc[10] = 1.0 / dt; sc[11] = 1.0 / dx;
    *dx_o = dx; *dt_o = dt;
}

// stream-ordered device scratch, released on every exit path
struct Scratch {
    void *p = nullptr;
    cudaStream_t st;
    explicit Scratch(cudaStream_t s) : st(s) {}
    cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes, st); }
    ~Scratch() { if (p) cudaFreeAsync(p, st); }
    Scratch(const Scratch &) = delete;
    Scratch &operator=(const Scratch &) = delete;
};

// CUDA event, destroyed on every exit path
struct Event {
    cudaEvent_t e = nullptr;
    cudaError_t create() { return cudaEventCreate(&e); }
    ~Event() { if (e) cudaEventDestroy(e); }
    Event() = default;
    Event(const Event &) = delete;
    Event &operator=(const Event &) = delete;
};

// Grid of a grid-stride kernel over `work` items with `tb` threads per block: one item per thread, at most
// `per_sm` blocks per SM of `device`.  The reductions accumulate one partial sum per block, so their grouping
// (and last bits) follow this grid.
int stride_grid(int device, long long work, int tb, int per_sm, unsigned *grid)
{
    int nsm = 0;
    CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device));
    const long long want = (work + tb - 1) / tb, cap = (long long)nsm * per_sm;
    *grid = (unsigned)(want < cap ? want : cap);
    return TRPL_OK;
}

struct Cfg { int M; bool pad; int W; };      // W = warps per simulation (1: warp kernel, >1: CTA kernel)
int pick_cfg(int L, Cfg *cfg)
{
    if (L < 2) return TRPL_EINVAL;
    if (L <= 256) {
        // one warp per simulation, M nodes per lane; grids that do not fill 32*M nodes are padded
        int M = 1;
        while (32 * M < L) M <<= 1;
        cfg->M = M; cfg->pad = (L != 32 * M); cfg->W = 1;
        return TRPL_OK;
    }
    // fine grids: one CTA of W warps per simulation, 8 nodes per lane (fewer interface unknowns and
    // less solver work per node than 4: +25 % at L=1000, round 1).  pad = general padding (L % 8 != 0);
    // otherwise the unused lanes carry a dummy film (run_sim PADM = 1).
    if (L > 256 * 8) return TRPL_EUNSUPPORTED;
    int W = 2;
    while (32 * 8 * W < L) W <<= 1;
    cfg->M = 8; cfg->pad = (L % 8 != 0); cfg->W = W;
    return TRPL_OK;
}

typedef void (*kern_t)(const KArgs);
kern_t pick_kernel(const Cfg &c)
{
    if (c.W > 1) {
        switch (c.W) {
        case 2: return c.pad ? trpl_sim_cta_kernel<2, 8, 2> : trpl_sim_cta_kernel<2, 8, 1>;
        case 4: return c.pad ? trpl_sim_cta_kernel<4, 8, 2> : trpl_sim_cta_kernel<4, 8, 1>;
        default: return c.pad ? trpl_sim_cta_kernel<8, 8, 2> : trpl_sim_cta_kernel<8, 8, 1>;
        }
    }
    switch (c.M) {
    case 1: return c.pad ? trpl_sim_kernel<1, true> : trpl_sim_kernel<1, false>;
    case 2: return c.pad ? trpl_sim_kernel<2, true> : trpl_sim_kernel<2, false>;
    case 4: return c.pad ? trpl_sim_kernel<4, true> : trpl_sim_kernel<4, false>;
    default: return c.pad ? trpl_sim_kernel<8, true> : trpl_sim_kernel<8, false>;
    }
}

// threads per CTA, simulations per CTA and dynamic shared memory of a configuration
void cfg_shape(const Cfg &c, int *threads, int *sims_per_cta, size_t *smem)
{
    const size_t ring = (size_t)(4 * 3 * c.M * 32 + RING_CANARY) * sizeof(double);       // per warp
    if (c.W > 1) {
        *threads = c.W * 32;
        *sims_per_cta = 1;
        // + exchange buffer [2][2][32W], reduction scratch [2][W][4], interface-system planes [9][(32+16/W)W]
        *smem = c.W * ring + (size_t)(2 * 2 * 32 * c.W + 2 * c.W * 4 + 9 * (32 + 16 / c.W) * c.W) * sizeof(double);
    } else {
        *threads = WARPS_PER_CTA * 32;
        *sims_per_cta = WARPS_PER_CTA;
        *smem = WARPS_PER_CTA * ring;
    }
}

// Launch geometry of a configuration on `device`: kernel, threads and simulations per CTA, dynamic shared
// memory, resident CTAs per SM and SM count.
struct Geometry {
    kern_t k;
    int threads, sims_per_cta;
    size_t smem;
    int ctas_per_sm, sms;
};

int kernel_geometry(int device, const Cfg &cfg, Geometry *geo)
{
    kern_t k = pick_kernel(cfg);
    int threads, spc; size_t smem;
    cfg_shape(cfg, &threads, &spc, &smem);
    CK(cudaFuncSetAttribute((const void *)k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute((const void *)k, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    int nb = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, (const void *)k, threads, smem));
    if (nb < 1) return TRPL_EUNSUPPORTED;
    int nsm = 0;
    CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device));
    *geo = Geometry{k, threads, spc, smem, nb, nsm};
    return TRPL_OK;
}

// KArgs fields shared by both entry points: tolerance 10^-tol, BDF order clamped to 1..5 (out of range = 5)
void init_kargs(KArgs &ka, int L, int tol, int max_iter, int max_order)
{
    memset(&ka, 0, sizeof(ka));
    ka.TOL = pow(10.0, -(double)tol);
    ka.L = L;
    ka.max_iter = max_iter;
    ka.max_order = (max_order < 1 || max_order > 5) ? 5 : max_order;
}

// scales, initial-profile factor and PL re-dimensioning of one curve (pvSimPCR.py:327-331, :393)
void init_curve(CurveDev &cv, double length, double time, int L, int T, int flags, const double *d_init)
{
    double dx, dt;
    make_scales(length, time, L, T, cv.scales, &dx, &dt);
    cv.init_mul = (flags & TRPL_F_INIT_GRID_UNITS) ? 1.0 : cv.scales[0];
    cv.redim = pow(dx, 2.0) * dt;
    cv.init = d_init;
}

// Makes `device` current for the duration of one C-ABI call and restores the caller's device on every
// exit path (torch reads its current device from the runtime; a library must not change it).
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    int enter(int device)
    {
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
            cudaGetLastError();
            return TRPL_ENODEVICE;
        }
        CK(cudaGetDevice(&prev));
        if (prev != device) {
            CK(cudaSetDevice(device));
            switched = true;
        }
        return TRPL_OK;
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

// Runs `work` (returning a TRPL_* code) with `device` current, or returns why the device cannot be entered.
// Entry points validate their arguments before this and call it once, so every one has the same shape.
template <class F>
int on_device(int device, F &&work)
{
    DeviceGuard guard;
    TRY(guard.enter(device));
    return work();
}

int launch_sims(KArgs &ka, const Cfg &cfg, int device, cudaStream_t st)
{
    Geometry geo;
    int rc = kernel_geometry(device, cfg, &geo);
    if (rc) return rc;
    // longest-processing-time-first order of the curves (insertion sort, C <= 8)
    for (int c = 0; c < ka.C; c++) ka.curve_order[c] = c;
    for (int i = 1; i < ka.C; i++)
        for (int j = i; j > 0 && ka.curves[ka.curve_order[j]].t_last > ka.curves[ka.curve_order[j - 1]].t_last; j--) {
            const int t = ka.curve_order[j]; ka.curve_order[j] = ka.curve_order[j - 1]; ka.curve_order[j - 1] = t;
        }
    Scratch counter(st);
    CK(counter.alloc(sizeof(unsigned long long)));
    CK(cudaMemsetAsync(counter.p, 0, sizeof(unsigned long long), st));
    ka.counter = (unsigned long long *)counter.p;
    const unsigned long long items = (unsigned long long)ka.S * ka.C;
    unsigned long long want = (items + geo.sims_per_cta - 1) / geo.sims_per_cta;
    unsigned long long cap = (unsigned long long)geo.ctas_per_sm * geo.sms;
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    if (grid > 0) {
        geo.k<<<grid, geo.threads, geo.smem, st>>>(ka);
        CK(cudaGetLastError());
    }
    return TRPL_OK;
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int trpl_version(void) { return 200 + (TRPL_DEBUG ? 1 : 0); }   // odd = debug build (device-side checks)

const char *trpl_error_string(int code)
{
    switch (code) {
    case TRPL_OK: return "ok";
    case TRPL_EINVAL: return "invalid argument";
    case TRPL_EUNSUPPORTED: return "unsupported shape (need 2 <= L <= 2048, curves <= 8, observation files <= 4)";
    case TRPL_ECUDA: return "CUDA runtime error";
    case TRPL_ENODEVICE: return "no usable CUDA device";
    default: return "unknown error";
    }
}

const char *trpl_last_cuda_error(void) { return g_cuda_err; }

int trpl_resident_sims(int device, int L)
{
    Cfg cfg;
    TRY(pick_cfg(L, &cfg));
    return on_device(device, [&] {
        Geometry geo;
        TRY(kernel_geometry(device, cfg, &geo));
        return geo.ctas_per_sm * geo.sms * geo.sims_per_cta;
    });
}

int trpl_solve_pl(const double *d_matpar, int64_t S, int64_t ld_matpar, const double *d_init,
                  double length, double time, int L, int T, int plT, int tol, int max_iter,
                  int max_order, int flags, void *d_pl, int pl_dtype, int64_t pl_stride,
                  int32_t *d_status, int64_t *d_iters, int device, void *stream)
{
    if (!d_matpar || !d_init || !d_pl || S < 0 || ld_matpar < TRPL_NPAR || T < 1 || plT < 1 ||
        max_iter < 1 || !(length > 0) || !(time > 0) || pl_stride < T / plT + 1 ||
        (pl_dtype != TRPL_F64 && pl_dtype != TRPL_F32))
        return TRPL_EINVAL;
    Cfg cfg;
    TRY(pick_cfg(L, &cfg));
    return on_device(device, [&] {
        if (S == 0) return TRPL_OK;
        KArgs ka;
        init_kargs(ka, L, tol, max_iter, max_order);
        ka.x = d_matpar; ka.ldx = ld_matpar; ka.S = S; ka.pl_stride = pl_stride;
        ka.sse = nullptr; ka.status = d_status; ka.iters = (long long *)d_iters;
        ka.mag_col = -1; ka.C = 1; ka.E = 0; ka.plT = plT;
        ka.flags = (flags & TRPL_F_INIT_GRID_UNITS) | (pl_dtype == TRPL_F32 ? TRPL_F_EMULATE_F32 : 0);
        ka.pl_dtype = pl_dtype;
        CurveDev &cv = ka.curves[0];
        init_curve(cv, length, time, L, T, flags, d_init);
        cv.pl_out = d_pl;
        cv.t_last = T;
        return launch_sims(ka, cfg, device, (cudaStream_t)stream);
    });
}

int trpl_solve_loglik(const double *d_x, int64_t S, int64_t ldx, int mag_col,
                      const trpl_curve *curves, int C, int E, double time, int L, int T, int tol,
                      int max_iter, int max_order, int flags, double *d_sse, double *d_lnl,
                      int32_t *d_status, int64_t *d_iters, int device, void *stream)
{
    if (!d_x || !curves || !d_sse || !d_lnl || S < 0 || ldx < TRPL_NPAR || mag_col >= ldx ||
        T < 1 || max_iter < 1 || !(time > 0) || C < 1 || E < 1)
        return TRPL_EINVAL;
    if (C > TRPL_MAX_CURVES || E > TRPL_MAX_EXP) return TRPL_EUNSUPPORTED;
    Cfg cfg;
    TRY(pick_cfg(L, &cfg));
    return on_device(device, [&] {
        if (S == 0) return TRPL_OK;
        cudaStream_t st = (cudaStream_t)stream;

        KArgs ka;
        init_kargs(ka, L, tol, max_iter, max_order);
        ka.x = d_x; ka.ldx = ldx; ka.S = S; ka.pl_stride = 0;
        ka.sse = d_sse; ka.iters = (long long *)d_iters;
        ka.mag_col = mag_col; ka.C = C; ka.E = E; ka.plT = 1;
        ka.flags = flags; ka.pl_dtype = TRPL_F64;
        for (int c = 0; c < C; c++) {
            const trpl_curve &src = curves[c];
            if (!src.d_init || !(src.length > 0)) return TRPL_EINVAL;
            CurveDev &cv = ka.curves[c];
            init_curve(cv, src.length, time, L, T, flags, src.d_init);
            cv.pl_out = nullptr;
            cv.t_last = 0;
            for (int e = 0; e < E; e++) {
                const trpl_obs &o = src.obs[e];
                if (o.n < 0 || (o.n > 0 && (!o.d_hi || !o.d_whi || !o.d_wlo || !o.d_val)))
                    return TRPL_EINVAL;
                if (o.n > 0 && (o.hi_max < 1 || o.hi_max > T)) return TRPL_EINVAL;
                cv.obs[e].n = o.n; cv.obs[e].hi = o.d_hi; cv.obs[e].whi = o.d_whi;
                cv.obs[e].wlo = o.d_wlo; cv.obs[e].val = o.d_val;
                if (o.n > 0 && o.hi_max > cv.t_last) cv.t_last = o.hi_max;   // causal truncation
            }
        }
        Scratch status_cs(st);                     // allocated only after every argument was validated
        if (d_status) CK(status_cs.alloc(sizeof(int) * (size_t)C * S));
        ka.status = (int *)status_cs.p;
        TRY(launch_sims(ka, cfg, device, st));
        const int tb = 256;
        trpl_finish_kernel<<<(unsigned)((S + tb - 1) / tb), tb, 0, st>>>(d_sse, d_lnl, (const int *)status_cs.p,
                                                                          d_status, S, C, E);
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_log10_clamp(void *d_pl, int dtype, int64_t n, double min, int device, void *stream)
{
    if (!d_pl || n < 0 || (dtype != TRPL_F64 && dtype != TRPL_F32)) return TRPL_EINVAL;
    return on_device(device, [&] {
        if (n == 0) return TRPL_OK;
        cudaStream_t st = (cudaStream_t)stream;
        unsigned grid;
        TRY(stride_grid(device, n, 256, 16, &grid));
        if (dtype == TRPL_F64)
            trpl_log10_kernel<<<grid, 256, 0, st>>>((double *)d_pl, n, min);
        else
            trpl_log10_kernel<<<grid, 256, 0, st>>>((float *)d_pl, n, min);
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_lnp_accumulate(double *d_P, const double *d_pl, int64_t S, int64_t n, int64_t ld,
                        const double *d_values, const double *d_mag, int device, void *stream)
{
    if (!d_P || !d_pl || !d_values || !d_mag || S < 0 || n < 0 || ld < n) return TRPL_EINVAL;
    return on_device(device, [&] {
        if (S == 0) return TRPL_OK;
        unsigned grid;
        TRY(stride_grid(device, S * 32, 256, 8, &grid));    // one warp per sample
        trpl_lnp_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_P, d_pl, S, n, ld, d_values, d_mag);
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_obs_prepare(const double *times, int32_t n, double time, int T, int32_t *hi, double *whi,
                     double *wlo)
{
    if (!times || !hi || !whi || !wlo || n < 0 || T < 1 || !(time > 0)) return TRPL_EINVAL;
    // numpy.linspace(0, time, T+1): x_i = i*step with step = time/T, and x_T = time exactly
    const double step = time / T;
    int maxhi = 0;
    double prev = -INFINITY;
    for (int32_t i = 0; i < n; i++) {
        const double t = times[i];
        if (!(t >= 0.0) || !(t <= time) || t < prev) return TRPL_EINVAL;
        prev = t;
        // searchsorted(side='left'): first index k with x_k >= t
        long long k = (long long)floor(t / step);
        if (k < 0) k = 0;
        if (k > T) k = T;
        auto xk = [&](long long q) { return q >= T ? time : (double)q * step; };
        while (k > 0 && xk(k - 1) >= t) k--;
        while (k < T && xk(k) < t) k++;
        if (k < 1) k = 1;
        if (k > T) k = T;
        hi[i] = (int32_t)k;
        const double x_lo = xk(k - 1), x_hi = xk(k);
        whi[i] = (t - x_lo) / (x_hi - x_lo);
        wlo[i] = (x_hi - t) / (x_hi - x_lo);
        if (k > maxhi) maxhi = (int)k;
    }
    return maxhi;
}

int trpl_lse_partial(const double *d_x, int64_t n, double *d_out2, int device, void *stream)
{
    if (!d_x || !d_out2 || n < 0) return TRPL_EINVAL;
    return on_device(device, [&] {
        cudaStream_t st = (cudaStream_t)stream;
        trpl_lse_init_kernel<<<1, 1, 0, st>>>(d_out2);
        if (n > 0) {
            unsigned grid;
            TRY(stride_grid(device, n, 256, 8, &grid));
            trpl_lse_max_kernel<<<grid, 256, 0, st>>>(d_x, n, d_out2);
            trpl_lse_sum_kernel<<<grid, 256, 0, st>>>(d_x, n, d_out2);
        }
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_random_grid(double *d_x, int64_t S, int64_t ldx, const double *minx, const double *maxx,
                     const int32_t *do_log, int ncol, int override_flags, uint64_t seed,
                     uint64_t first_sample, int device, void *stream)
{
    if (!d_x || !minx || !maxx || !do_log || S < 0 || ncol < 1 || ncol > 16 || ldx < ncol) return TRPL_EINVAL;
    return on_device(device, [&] {
        if (S == 0) return TRPL_OK;
        GridArgs ga;
        memset(&ga, 0, sizeof(ga));
        for (int j = 0; j < ncol; j++) {
            if (!(minx[j] <= maxx[j]) || (do_log[j] && minx[j] != maxx[j] && !(minx[j] > 0))) return TRPL_EINVAL;
            ga.lo[j] = minx[j]; ga.hi[j] = maxx[j]; ga.do_log[j] = do_log[j];
        }
        ga.ncol = ncol;
        ga.eq_mu = (override_flags & 1) && ncol > 3;
        ga.eq_s = (override_flags & 2) && ncol > 6;
        ga.eq_auger = (override_flags & 4) && ncol > 8;
        unsigned grid;
        TRY(stride_grid(device, S * ncol, 256, 16, &grid));
        trpl_random_grid_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_x, S, ldx, ga, seed, first_sample);
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_posterior_weights(const double *d_lnp, int64_t n, double lse, double *d_w, int device, void *stream)
{
    if (!d_lnp || !d_w || n < 0) return TRPL_EINVAL;
    return on_device(device, [&] {
        if (n == 0) return TRPL_OK;
        unsigned grid;
        TRY(stride_grid(device, n, 256, 16, &grid));
        trpl_weights_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_lnp, n, lse, d_w);
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_weighted_hist(const double *d_x, int64_t n, int64_t ldx, int colx, int coly, const double *d_w,
                       double lox, double hix, int nbx, double loy, double hiy, int nby, double *d_hist,
                       int device, void *stream)
{
    if (!d_x || !d_hist || n < 0 || colx < 0 || colx >= ldx || coly >= ldx || nbx < 1 || !(hix > lox))
        return TRPL_EINVAL;
    if (coly >= 0 && (nby < 1 || !(hiy > loy))) return TRPL_EINVAL;
    const long long nb = (long long)nbx * (coly >= 0 ? nby : 1);
    if (nb > 8192) return TRPL_EUNSUPPORTED;
    return on_device(device, [&] {
        if (n == 0) return TRPL_OK;
        unsigned grid;
        TRY(stride_grid(device, n, 256, 4, &grid));
        const size_t smem = (size_t)nb * sizeof(double);
        CK(cudaFuncSetAttribute((const void *)trpl_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
        trpl_hist_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(d_x, ldx, colx, coly, d_w, n, lox, hix,
                                                                    nbx, loy, hiy, nby, d_hist);
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_weighted_moments(const double *d_x, int64_t n, int64_t ldx, int ncol, const double *d_w,
                          double *d_out, int device, void *stream)
{
    if (!d_x || !d_w || !d_out || n < 0 || ncol < 1 || ncol > 15 || ldx < ncol) return TRPL_EINVAL;
    return on_device(device, [&] {
        if (n == 0) return TRPL_OK;
        cudaStream_t st = (cudaStream_t)stream;
        unsigned grid;
        if (ncol == 13 || ncol == 12) {
            TRY(stride_grid(device, n, 128, 2, &grid));
            if (ncol == 13)
                trpl_moments_kernel_fixed<13><<<grid, 128, 0, st>>>(d_x, ldx, d_w, n, d_out);
            else
                trpl_moments_kernel_fixed<12><<<grid, 128, 0, st>>>(d_x, ldx, d_w, n, d_out);
        } else {
            TRY(stride_grid(device, n, 256, 8, &grid));
            const size_t smem = (size_t)(1 + ncol + ncol * ncol) * sizeof(double);
            trpl_moments_kernel<<<grid, 256, smem, st>>>(d_x, ldx, ncol, d_w, n, d_out);
        }
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_selftest_rcp(const double *d_x, double *d_y, int64_t n, int device, void *stream)
{
    if (!d_x || !d_y || n < 0) return TRPL_EINVAL;
    return on_device(device, [&] {
        if (n == 0) return TRPL_OK;
        long long blocks = (n + 255) / 256;
        if (blocks > 4096) blocks = 4096;
        trpl_rcp_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(d_x, d_y, n);
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_bench_dfma(int device, int iters, double *tflops, double *ms)
{
    if (!tflops || iters < 1) return TRPL_EINVAL;
    return on_device(device, [&] {
        int nsm = 0;
        CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device));
        Scratch out(0);                            // legacy default stream, where the kernels run
        CK(out.alloc(sizeof(double)));
        const int tb = 256, blocks = nsm * 8;
        Event e0, e1;
        CK(e0.create());
        CK(e1.create());
        trpl_dfma_kernel<<<blocks, tb>>>((double *)out.p, iters / 4 + 1, 1.0);   // warm-up
        CK(cudaEventRecord(e0.e));
        trpl_dfma_kernel<<<blocks, tb>>>((double *)out.p, iters, 1.0);
        CK(cudaEventRecord(e1.e));
        CK(cudaEventSynchronize(e1.e));
        float t = 0.f;
        CK(cudaEventElapsedTime(&t, e0.e, e1.e));
        const double flop = 2.0 * 8 * 16 * (double)iters * tb * (double)blocks;
        *tflops = flop / (t * 1e-3) / 1e12;
        if (ms) *ms = t;
        return TRPL_OK;
    });
}

}  // extern "C"
