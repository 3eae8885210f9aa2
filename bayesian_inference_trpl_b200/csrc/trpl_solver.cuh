// trpl_solver.cuh -- the forward-model + fused-likelihood kernels (the hot path):
// Comm<W> (lane communication policy), tridiag_solve (partition_sweep, warp_solve, cta_solve), Ring,
// run_sim, trpl_sim_kernel<M,PAD>, trpl_sim_cta_kernel<W,M,PADM>.  Replaces pvSimPCR.py:14-293 and
// bayeslib.py:150-196.  Comment lines tagged "[sec:" + a section name + "]" delimit the sections that
// profiles/sass_budget.py attributes SASS instructions to.
#pragma once
#include <type_traits>

#include "trpl_common.cuh"

namespace trpl {

// BDF1..5 coefficients (a0; a1..a5) of pvSimPCR.py:241-250, one row per order
__constant__ double c_bdf[5][6] = {
    {1.0, -1.0, 0.0, 0.0, 0.0, 0.0},
    {1.5, -2.0, 0.5, 0.0, 0.0, 0.0},
    {11.0 / 6, -3.0, 1.5, -1.0 / 3, 0.0, 0.0},
    {25.0 / 12, -4.0, 3.0, -4.0 / 3, 0.25, 0.0},
    {137.0 / 60, -5.0, 5.0, -10.0 / 3, 1.25, -0.2}};

// ---------------------------------------------------------------------------------------------
// Communication among the lanes that share one simulation.  W = warps per simulation.
//   W == 1: warp shuffles / votes only (the production path for L <= 256).
//   W  > 1: one CTA of W warps per simulation (fine grids, L up to 32*M*W).  Generic exchanges (a few per
//           time step) travel through a ping-pong buffer in shared memory, one __syncthreads each; the
//           tridiagonal solves use their own planes and two barriers per solve (tridiag_solve); the
//           stop rule rides on those barriers.  Every thread of the CTA executes the same sequence.
// g = index of this lane among the 32*W lanes of the simulation.
// ---------------------------------------------------------------------------------------------
template <int W>
struct Comm {
    int g;            // lane index within the simulation
    double *xb;       // W > 1: exchange buffer [2][XB_K][G] doubles
    double *red;      // W > 1: reduction scratch [2][W][4] doubles
    int phase;        // ping-pong selector of xb
    int rphase;       // ping-pong selector of red
    double *sb;       // W > 1: interface-system planes [9][SB_STRIDE * W] doubles (tridiag_solve)
    int solver;       // W > 1: warp that solves the next interface system (rotates after every solve)
    // Row r of the 32*W interface rows lives at slot(r): rows are dealt round-robin into W blocks of
    // 32 (+ padding), so that the solver warp, which takes W CONSECUTIVE rows per lane, and the
    // owning lanes, which touch one row each, both access shared memory without bank conflicts.
    static constexpr int XB_K = 2;
    static constexpr int SB_STRIDE = 32 + (W > 1 ? 16 / W : 0);
    static constexpr int SB_PLANE = SB_STRIDE * W;
    static __device__ __forceinline__ int slot(const int r) { return (r % W) * SB_STRIDE + r / W; }

    // W > 1: `buf` holds xb, red and sb back to back; the solver role starts at warp `solver0`
    __device__ __forceinline__ explicit Comm(const int g_, double *buf = nullptr, const int solver0 = 0)
        : g(g_), xb(buf), red(W > 1 ? buf + 2 * XB_K * 32 * W : nullptr), phase(0), rphase(0),
          sb(W > 1 ? red + 2 * W * 4 : nullptr), solver(solver0) {}

    // K values from lane g-dm (-> vm) and lane g+dp (-> vp); out-of-range sources return the
    // caller's own value (always multiplied by an exact zero downstream).  For W > 1 the barrier
    // of the exchange also OR-reduces `busy` over the simulation (BAR.RED.OR) and returns it, so a
    // block-wide vote costs no barrier of its own; W == 1 returns true.
    template <int K, bool WANT_M, bool WANT_P>
    __device__ __forceinline__ bool xchg(const double (&v)[K], const int dm, const int dp,
                                         double (&vm)[K], double (&vp)[K], const bool busy = true)
    {
        if constexpr (W == 1) {
#pragma unroll
            for (int k = 0; k < K; k++) {
                if (WANT_M) vm[k] = __shfl_up_sync(FULL, v[k], dm);
                if (WANT_P) vp[k] = __shfl_down_sync(FULL, v[k], dp);
            }
            return true;
        } else {
            constexpr int G = 32 * W;
            static_assert(K <= XB_K || W == 1, "exchange buffer too small");
            double *buf = xb + phase * (XB_K * G);
#pragma unroll
            for (int k = 0; k < K; k++) buf[k * G + g] = v[k];
            const bool any_busy = __syncthreads_or(busy) != 0;
            const int im = (g - dm >= 0) ? g - dm : g;
            const int ip = (g + dp < G) ? g + dp : g;
            TRPL_DASSERT(g >= 0 && g < G && im >= 0 && im < G && ip >= 0 && ip < G);
#pragma unroll
            for (int k = 0; k < K; k++) {
                if (WANT_M) vm[k] = buf[k * G + im];
                if (WANT_P) vp[k] = buf[k * G + ip];
            }
            phase ^= 1;
            return any_busy;
        }
    }
    __device__ __forceinline__ double from_prev(const double v)     // value of lane g-1
    {
        double a[1] = {v}, m[1], p_[1];
        xchg<1, true, false>(a, 1, 1, m, p_);
        return m[0];
    }
    __device__ __forceinline__ double from_next(const double v)     // value of lane g+1
    {
        double a[1] = {v}, m[1], p_[1];
        xchg<1, false, true>(a, 1, 1, m, p_);
        return p_[0];
    }
    __device__ __forceinline__ double sum(double v)                 // total over the simulation
    {
        v = warp_sum(v);
        if constexpr (W > 1) {
            double *r = red + rphase * (W * 4);
            if ((threadIdx.x & 31) == 0) r[(threadIdx.x >> 5) * 4] = v;
            __syncthreads();
            v = 0.0;
#pragma unroll
            for (int w = 0; w < W; w++) v += r[w * 4];
            rphase ^= 1;
        }
        return v;
    }
    // stop rule errN < TOL and errP < TOL (pvSimPCR.py:213-216) with err = sum|res| / sum|b|, evaluated
    // division-free as z = sum(|res| - TOL*|b|) < 0 for both species (one 2-value butterfly).
    // W > 1: stop_post() leaves the warp totals in shared memory, the block barriers of the tridiagonal
    // solve that follows publish them, stop_collect() adds them up -- no barrier of its own.
    __device__ __forceinline__ double stop_butterfly(const double zN, const double zP)
    {
        const int lane = threadIdx.x & 31;
        const bool hi16 = (lane & 16) != 0;
        double k = hi16 ? zP : zN;
        const double sd = hi16 ? zN : zP;
        k += __shfl_xor_sync(FULL, sd, 16);
        k += __shfl_xor_sync(FULL, k, 8);
        k += __shfl_xor_sync(FULL, k, 4);
        k += __shfl_xor_sync(FULL, k, 2);
        k += __shfl_xor_sync(FULL, k, 1);
        return k;                 // lanes 0-15: zN of this warp, lanes 16-31: zP
    }
    __device__ __forceinline__ void stop_rule(const double zN, const double zP, bool &converged,
                                              bool &nonfinite)
    {
        static_assert(W == 1, "multi-warp simulations use stop_post / stop_collect");
        const double k = stop_butterfly(zN, zP);
        converged = __all_sync(FULL, k < 0.0);
        nonfinite = __any_sync(FULL, !(fabs(k) <= DBL_MAX));
    }
    __device__ __forceinline__ void stop_post(const double zN, const double zP)
    {
        const int lane = threadIdx.x & 31;
        const double k = stop_butterfly(zN, zP);
        double *r = red + rphase * (W * 4);
        if ((lane & 15) == 0) r[(threadIdx.x >> 5) * 4 + (lane >> 4)] = k;
    }
    __device__ __forceinline__ void stop_collect(bool &converged, bool &nonfinite)
    {
        const int lane = threadIdx.x & 31;
        const double *r = red + rphase * (W * 4);
        double k = 0.0;
#pragma unroll
        for (int w = 0; w < W; w++) k += r[w * 4 + (lane >> 4)];
        rphase ^= 1;
        converged = __all_sync(FULL, k < 0.0);
        nonfinite = __any_sync(FULL, !(fabs(k) <= DBL_MAX));
    }
};

// one normalised PCR stage: row i absorbs rows i-rf (vm) and i+rf (vp); {L,U,B} with unit diagonal
__device__ __forceinline__ void pcr_stage(double &Lr, double &Ur, double &Br, const double (&vm)[3],
                                          const double (&vp)[3])
{
    const double Lm = vm[0], Um = vm[1], Bm = vm[2];
    const double Lp = vp[0], Up = vp[1], Bp = vp[2];
    const double D = fma(-Lp, Ur, fma(-Um, Lr, 1.0));
    const double B = fma(-Bp, Ur, fma(-Bm, Lr, Br));
    const double Ln = -Lm * Lr;
    const double Un = -Up * Ur;
    const double inv = rcp64(D);
    Br = B * inv;
    Lr = Ln * inv;
    Ur = Un * inv;
}

// Tridiagonal solve, M rows per lane (row n = M*g + j):  l[j] x[n-1] + d[j] x[n] + u[j] x[n+1] = b[j].
// Rows outside the physical system must be identity rows (l=u=0, d=1).  l of the first row
// and u of the last physical row must be 0.  Every lane first eliminates its M-1 interior rows
// (partition_sweep), which leaves one interface row per lane; the two kernel families then solve the
// interface system in their own way (warp_solve, cta_solve).  Both return the new value of the previous
// lane's last node (needed by the callers anyway) and store the new value of the NEXT lane's first node
// in xr.
//
// Pivots of the sweep, chosen per kernel family (each measured better on its own kernel,
// profiles/r02_variants.txt): the warp kernel uses the Thomas recurrence (3 multiplies fewer, but M-1
// reciprocals in series); the CTA kernel, whose simulations run 2 warps per scheduler and so expose
// dependent chains, uses reciprocals of the leading minors, which are independent of each other.

// [sec:partition] interior rows 0..M-2 of a lane (M > 1):  x_j = y_j - v_j * s_left - w_j * s_own
template <int M, bool MINOR_PIVOTS>
__device__ __forceinline__ void partition_sweep(const double (&l)[M], const double (&d)[M],
                                                const double (&u)[M], const double (&b)[M],
                                                double (&y)[M - 1], double (&v)[M - 1], double (&w)[M - 1])
{
    double c[M - 1];
    if constexpr (MINOR_PIVOTS) {
        // Pivot reciprocals from the leading principal minors m_{j+1} = d_j m_j - l_j u_{j-1} m_{j-1}
        // (1/pivot_j = m_j / m_{j+1}): independent reciprocals, 3 more multiplies per solve.
        double ip[M - 1];
        {
            double mm[M];                 // mm[j] = m_{j+1}
            mm[0] = d[0];
            if constexpr (M > 2) mm[1] = fma(d[1], d[0], -(l[1] * u[0]));
#pragma unroll
            for (int j = 2; j < M - 1; j++) mm[j] = fma(d[j], mm[j - 1], -((l[j] * u[j - 1]) * mm[j - 2]));
            ip[0] = rcp64(mm[0]);
#pragma unroll
            for (int j = 1; j < M - 1; j++) ip[j] = mm[j - 1] * rcp64(mm[j]);
        }
        c[0] = u[0] * ip[0];
        y[0] = b[0] * ip[0];
        v[0] = l[0] * ip[0];
#pragma unroll
        for (int j = 1; j < M - 1; j++) {
            c[j] = u[j] * ip[j];
            y[j] = fma(-l[j], y[j - 1], b[j]) * ip[j];
            v[j] = (-l[j] * v[j - 1]) * ip[j];
        }
    } else {
        // Thomas forward sweep: pivot_j = d_j - l_j c_{j-1}
        {
            const double ip0 = rcp64(d[0]);
            c[0] = u[0] * ip0;
            y[0] = b[0] * ip0;
            v[0] = l[0] * ip0;
        }
#pragma unroll
        for (int j = 1; j < M - 1; j++) {
            const double ipj = rcp64(fma(-l[j], c[j - 1], d[j]));
            c[j] = u[j] * ipj;
            y[j] = fma(-l[j], y[j - 1], b[j]) * ipj;
            v[j] = (-l[j] * v[j - 1]) * ipj;
        }
    }
    w[M - 2] = c[M - 2];
#pragma unroll
    for (int j = M - 3; j >= 0; j--) {
        y[j] = fma(-c[j], y[j + 1], y[j]);
        v[j] = fma(-c[j], v[j + 1], v[j]);
        w[j] = -c[j] * w[j + 1];
    }
}

// One warp, 32 interface rows (one per lane): parallel cyclic reduction with warp shuffles, then
// back-substitution.  Used by the warp kernel and by the solver warp of the CTA kernel.
template <int M, bool MINOR_PIVOTS>
__device__ __forceinline__ double warp_solve(const double (&l)[M], const double (&d)[M], const double (&u)[M],
                                             const double (&b)[M], double (&x)[M], Comm<1> &cm, double &xr)
{
    double Lr, Dr, Ur, Br;
    double y[M > 1 ? M - 1 : 1], v[M > 1 ? M - 1 : 1], w[M > 1 ? M - 1 : 1];
    if constexpr (M > 1) {
        partition_sweep<M, MINOR_PIVOTS>(l, d, u, b, y, v, w);
        // interface row (local M-1) couples s_left, s_own and the next lane's first interior row
        double mine[3] = {y[0], v[0], w[0]}, nm[3], nx[3];
        cm.xchg<3, false, true>(mine, 1, 1, nm, nx);
        const double y0n = nx[0], v0n = nx[1], w0n = nx[2];
        const double lr = l[M - 1], ur = u[M - 1];
        Lr = -lr * v[M - 2];
        Dr = fma(-ur, v0n, fma(-lr, w[M - 2], d[M - 1]));
        Ur = -ur * w0n;
        Br = fma(-ur, y0n, fma(-lr, y[M - 2], b[M - 1]));
    } else {
        Lr = l[0]; Dr = d[0]; Ur = u[0]; Br = b[0];
    }
    // [sec:normalise] parallel cyclic reduction over the 32 interface unknowns, unit diagonal
    {
        double inv = rcp64(Dr);
        Lr *= inv; Ur *= inv; Br *= inv;
    }
    // [sec:pcr]
    // off-diagonals below 2^-PCR_LAST_EXP: the stage degenerates to a B-only update.  At 35 that is exact
    // (see below); a 2^-27 threshold measured 1.3 % faster but is not bit-identical (profiles/r02_variants.txt).
    constexpr int PCR_LAST_EXP = 35;
#pragma unroll
    for (int rf = 1; rf < 32; rf <<= 1) {
        // Off-diagonals shrink quadratically per stage.  Let m = max |L|,|U| over the simulation:
        //   m < 2^-70: the remaining stages cannot change D = 1 or B in the last bit: stop;
        //   m < 2^-35: this is the last stage, and in it D = 1 - O(m^2) rounds to exactly 1 and the new
        //              off-diagonals are < 2^-70, so only B needs updating (bit-identical to a full
        //              stage followed by the stop above): one third of the exchange, 2 FMAs.
        // (Not tested before the first three stages: a coupling that small after two stages means
        // an initial one below 2^-9, i.e. practically no transport; those cases just run 3 stages.)
        const int hl = __double2hiint(Lr) & 0x7fffffff, hu = __double2hiint(Ur) & 0x7fffffff;
        const int hm = max(hl, hu);
        const bool busy = (rf < 8) || (hm >= ((1023 - PCR_LAST_EXP) << 20));
        if (rf >= 8 && !__any_sync(FULL, busy)) {
            if (__any_sync(FULL, hm >= ((1023 - 70) << 20))) {
                double mine[1] = {Br}, vm[1], vp[1];
                cm.xchg<1, true, true>(mine, rf, rf, vm, vp);
                Br = fma(-vp[0], Ur, fma(-vm[0], Lr, Br));
            }
            break;
        }
        double mine[3] = {Lr, Ur, Br}, vm[3], vp[3];
        cm.xchg<3, true, true>(mine, rf, rf, vm, vp);
        pcr_stage(Lr, Ur, Br, vm, vp);
    }
    // [sec:backsubst]
    x[M - 1] = Br;
    const double sl = cm.from_prev(Br);
    if constexpr (M > 1) {
#pragma unroll
        for (int j = 0; j < M - 1; j++) x[j] = fma(-w[j], Br, fma(-v[j], sl, y[j]));
    }
    xr = cm.from_next(x[0]);
    return sl;
}

// [sec:partition] One CTA of W warps, 32*W interface rows.  They are handed to ONE warp through shared
// memory, which holds W of them per lane and solves them with warp_solve (a second partition level +
// shuffle PCR): two block barriers per solve instead of one per PCR stage over 32*W unknowns.  The
// solver role rotates over the warps from solve to solve: warp k of every CTA sits on scheduler k, so a
// fixed solver warp would load one scheduler of the SM with the serial part of all resident CTAs (+46 %
// time per iteration, measured).  The neighbour values the caller needs (previous lane's last node,
// next lane's first node) are rebuilt from the interface solution, so no further exchange follows.
template <int M, int W>
__device__ __forceinline__ double cta_solve(const double (&l)[M], const double (&d)[M], const double (&u)[M],
                                            const double (&b)[M], double (&x)[M], Comm<W> &cm, double &xr)
{
    static_assert(W > 1 && M > 1, "multi-warp simulations keep at least 2 nodes per lane");
    double y[M - 1], v[M - 1], w[M - 1];
    partition_sweep<M, true>(l, d, u, b, y, v, w);
    // Shared-memory planes (rows at Comm::slot): 0-6 = input of the solver warp, written by every
    // lane before barrier 1 and read by the solver warp only; 7-8 = output (interface solution z, and
    // the next lane's first node xr), written by the solver warp before barrier 2 and read by every lane
    // after it.  Inputs and outputs never share a plane, so one buffer is enough: the next solve's
    // inputs are written after barrier 2 of this one, its outputs after its own barrier 1.
    constexpr int G = 32 * W, PL_ = Comm<W>::SB_PLANE, ST_ = Comm<W>::SB_STRIDE;
    const int g = cm.g;
    double *sb = cm.sb;
    const int me = Comm<W>::slot(g);
    TRPL_DASSERT(me >= 0 && me < PL_ && g < G);
    const double lr = l[M - 1];
    sb[0 * PL_ + me] = y[0];
    sb[1 * PL_ + me] = v[0];
    sb[2 * PL_ + me] = w[0];
    sb[3 * PL_ + me] = -lr * v[M - 2];                      // this lane's share of its interface row
    sb[4 * PL_ + me] = fma(-lr, w[M - 2], d[M - 1]);
    sb[5 * PL_ + me] = fma(-lr, y[M - 2], b[M - 1]);
    sb[6 * PL_ + me] = u[M - 1];
    __syncthreads();
    if ((g >> 5) == cm.solver) {
        const int sl_ = g & 31;                            // solver lane: rows W*sl_ .. W*sl_+W-1
        double L2[W], D2[W], U2[W], B2[W], Z[W];
#pragma unroll
        for (int k = 0; k < W; k++) {
            const int r = W * sl_ + k;                     // slot(r) = k * ST_ + sl_
            const int here = k * ST_ + sl_;
            const int next = (k + 1 < W) ? here + ST_ : ((sl_ < 31) ? sl_ + 1 : here);
            const double ur = (r < G - 1) ? sb[6 * PL_ + here] : 0.0;
            L2[k] = sb[3 * PL_ + here];
            D2[k] = fma(-ur, sb[1 * PL_ + next], sb[4 * PL_ + here]);
            U2[k] = -ur * sb[2 * PL_ + next];
            B2[k] = fma(-ur, sb[0 * PL_ + next], sb[5 * PL_ + here]);
        }
        Comm<1> c1(sl_);
        double znext;                                      // first row of the next lane
        warp_solve<W, true>(L2, D2, U2, B2, Z, c1, znext);
#pragma unroll
        for (int k = 0; k < W; k++) {
            const int here = k * ST_ + sl_;
            const int next = (k + 1 < W) ? here + ST_ : ((sl_ < 31) ? sl_ + 1 : here);
            const double zn = (k + 1 < W) ? Z[k + 1] : znext;
            sb[7 * PL_ + here] = Z[k];
            sb[8 * PL_ + here] = fma(-sb[2 * PL_ + next], zn, fma(-sb[1 * PL_ + next], Z[k], sb[0 * PL_ + next]));
        }
    }
    __syncthreads();
    cm.solver = (cm.solver + 1) & (W - 1);     // the role rotates: every scheduler gets its share of the serial part
    const double z = sb[7 * PL_ + me];
    const double zl = (g > 0) ? sb[7 * PL_ + Comm<W>::slot(g - 1)] : 0.0;
    xr = (g < G - 1) ? sb[8 * PL_ + me] : 0.0;
    x[M - 1] = z;
#pragma unroll
    for (int j = 0; j < M - 1; j++) x[j] = fma(-w[j], z, fma(-v[j], zl, y[j]));
    return zl;
}

template <int M, int W>
__device__ __forceinline__ double tridiag_solve(const double (&l)[M], const double (&d)[M],
                                                const double (&u)[M], const double (&b)[M],
                                                double (&x)[M], Comm<W> &cm, double &xr)
{
    if constexpr (W == 1) return warp_solve<M, false>(l, d, u, b, x, cm, xr);
    else return cta_solve<M, W>(l, d, u, b, x, cm, xr);
}

// [sec:none]
// lane-private ring of the 4 older BDF levels: [slot 0..3][field N,P,E][M doubles per lane]
template <int M>
struct Ring {
    double *base;   // warp base + lane offset
    // element (slot, field, j): chunks of 2 doubles per lane keep 16-byte accesses conflict-free
    __device__ __forceinline__ void load(int slot, int field, double (&h)[M]) const
    {
        TRPL_DASSERT(slot >= 0 && slot < 4 && field >= 0 && field < 3);
        if constexpr (M == 1) {
            h[0] = base[(slot * 3 + field) * 32];
        } else {
#pragma unroll
            for (int q = 0; q < M / 2; q++) {
                const double2 t = *reinterpret_cast<const double2 *>(
                    base + ((slot * 3 + field) * (M / 2) + q) * 64);
                h[2 * q] = t.x;
                h[2 * q + 1] = t.y;
            }
        }
    }
    __device__ __forceinline__ void store(int slot, int field, const double (&h)[M]) const
    {
        TRPL_DASSERT(slot >= 0 && slot < 4 && field >= 0 && field < 3);
        if constexpr (M == 1) {
            base[(slot * 3 + field) * 32] = h[0];
        } else {
#pragma unroll
            for (int q = 0; q < M / 2; q++)
                *reinterpret_cast<double2 *>(base + ((slot * 3 + field) * (M / 2) + q) * 64) =
                    make_double2(h[2 * q], h[2 * q + 1]);
        }
    }
};

struct WarpScratch {      // per-warp shared scratch touched once every 32 PL samples
    double sse[TRPL_MAX_EXP];
    int pos[TRPL_MAX_EXP];
};

// ---------------------------------------------------------------------------------------------
// one (sample, curve) simulation, executed by W warps (W == 1: one warp; W > 1: one CTA)
// ---------------------------------------------------------------------------------------------
// PADM = how a grid that does not fill the 32*W*M node slots is handled:
//   0  exact fit (L == 32*W*M);
//   1  L is a multiple of M: the lanes beyond the last physical one carry an independent dummy film at
//      equilibrium (N0, P0, E = 0, no excitation, no surface recombination, zero-flux ends).  It is
//      cut off from the physical system exactly like the two film surfaces are (one missing-neighbour
//      edge), it is left out of the residual norms and of PL, and it costs no per-row selects;
//   2  any L: nodes beyond L-1 are identity rows (selects on every row).
template <int M, int PADM, int W>
__device__ __forceinline__ void run_sim(const KArgs &a, const int c, const long long s,
                                        double *ring_warp, WarpScratch *ws, const int lane,
                                        Comm<W> &cm)
{
    constexpr int G = 32 * W;
    const int g = cm.g;                         // lane index within the simulation
    const bool io_warp = (W == 1) || (g < 32);  // the warp that stages, stores and scores PL
    const CurveDev &cv = a.curves[c];
    const int L = a.L;
    const int flags = a.flags;
    const bool emu32 = (flags & TRPL_F_EMULATE_F32) != 0;

    // ---- parameters: non-dimensionalise (pvSimPCR.py:327-331), one column per lane, then broadcast
    // Every per-simulation constant, raw or derived, is computed once, parked in one lane of `ctab`
    // and read back with a constant-lane shuffle: ptxas proves such a value warp-uniform and can
    // hold it in a uniform register; a derived constant it could recompute (tauP*N0P0 ...) would be
    // rematerialised inside the Newton loop as a product of two uniform values, which forces one of
    // them into a vector register for all of its uses (3-register DFMAs, +50 % issue time each).
    double ctab;
    {
        double raw = 0.0;
        if (lane < TRPL_NPAR) raw = a.x[s * a.ldx + lane] * cv.scales[lane];
        const double rN0 = __shfl_sync(FULL, raw, 0), rP0 = __shfl_sync(FULL, raw, 1);
        const double rDN = __shfl_sync(FULL, raw, 2), rDP = __shfl_sync(FULL, raw, 3);
        const double rtN = __shfl_sync(FULL, raw, 9), rtP = __shfl_sync(FULL, raw, 10);
        const double rLam = __shfl_sync(FULL, raw, 11);
        const double n0p0 = rN0 * rP0;
        ctab = raw;                                   // lanes 0..11: the scaled parameters
        ctab = (lane == 12) ? n0p0 : ctab;
        ctab = (lane == 13) ? 0.5 * rDN : ctab;
        ctab = (lane == 14) ? 0.5 * rDP : ctab;
        ctab = (lane == 15) ? rtP * n0p0 : ctab;
        ctab = (lane == 16) ? rtN * n0p0 : ctab;
        ctab = (lane == 17) ? rLam * rDP : ctab;
        ctab = (lane == 18) ? rLam * rDN : ctab;
        ctab = (lane == 19) ? 0.5 * (rLam * rDP) : ctab;
        ctab = (lane == 20) ? 0.5 * (rLam * rDN) : ctab;
        ctab = (lane == 21) ? -(double)L * n0p0 : ctab;
    }
    const double DN = __shfl_sync(FULL, ctab, 2), DP = __shfl_sync(FULL, ctab, 3);
    const double rate = __shfl_sync(FULL, ctab, 4);
    const double sr0 = __shfl_sync(FULL, ctab, 5), srL = __shfl_sync(FULL, ctab, 6);
    const double CN = __shfl_sync(FULL, ctab, 7), CP = __shfl_sync(FULL, ctab, 8);
    const double tauN = __shfl_sync(FULL, ctab, 9), tauP = __shfl_sync(FULL, ctab, 10);
    const double N0 = __shfl_sync(FULL, ctab, 0), P0 = __shfl_sync(FULL, ctab, 1);
    const double N0P0 = __shfl_sync(FULL, ctab, 12);
    const double hDN = __shfl_sync(FULL, ctab, 13), hDP = __shfl_sync(FULL, ctab, 14);
    const double tauP_N0P0 = __shfl_sync(FULL, ctab, 15), tauN_N0P0 = __shfl_sync(FULL, ctab, 16);
    const double LamDP = __shfl_sync(FULL, ctab, 17), LamDN = __shfl_sync(FULL, ctab, 18);
    const double hLamDP = __shfl_sync(FULL, ctab, 19), hLamDN = __shfl_sync(FULL, ctab, 20);
    const double mLN0P0 = __shfl_sync(FULL, ctab, 21);   // pvSimPCR.py:278
    const double TOL = a.TOL;
    const double mag = (a.mag_col >= 0) ? a.x[s * a.ldx + a.mag_col] : 0.0;

    // ---- geometry of this lane
    const int last_lane = (L - 1) / M;         // lane owning node L-1 ...
    constexpr bool PAD = (PADM == 2);
    const int jl = PAD ? (L - 1) % M : M - 1;  // ... at local index jl (M-1 unless PADM == 2)
    const bool dummy = (PADM == 1) && (g > last_lane);   // lane of the dummy film
    bool ev[M + 1];                            // edge m = M*g + j is an interior edge (1..L-1)
#pragma unroll
    for (int j = 0; j <= M; j++) {
        const int m = M * g + j;
        // exact-fit grids (L == M*G): only edge 0 (first lane) and edge L (last lane) are
        // boundaries, so the selects on the inner edges fold away at compile time
        ev[j] = PAD ? ((m >= 1) && (m <= L - 1))
                    : (j == 0 ? (g != 0 && !(PADM == 1 && g == last_lane + 1))
                              : (j == M ? (g != G - 1 && !(PADM == 1 && g == last_lane)) : true));
    }
    bool nv[M];                                // node n = M*g + j exists
#pragma unroll
    for (int j = 0; j < M; j++) nv[j] = PAD ? (M * g + j < L) : true;
    // surface rows: lane 0 applies the front surface to j=0, last_lane the back surface to j=jl
    const bool is_first = (g == 0), is_last = (g == last_lane);
    const double srf = is_first ? sr0 : (is_last ? srL : 0.0);

    // ---- initial state (pvSimPCR.py:339-362): N = N0 + dN, P = P0 + dN, E = 0
    double N[M], P[M], E[M];
#pragma unroll
    for (int j = 0; j < M; j++) {
        const int n = M * g + j;
        double dn = 0.0;
        if (n < L) dn = cv.init[n] * cv.init_mul;
        N[j] = nv[j] ? N0 + dn : 0.0;
        P[j] = nv[j] ? P0 + dn : 0.0;
        E[j] = 0.0;
    }
    Ring<M> ring;
    ring.base = ring_warp + ((M == 1) ? lane : 2 * lane);
    {
        double z[M];
#pragma unroll
        for (int j = 0; j < M; j++) z[j] = 0.0;
#pragma unroll
        for (int sl = 0; sl < 4; sl++)
#pragma unroll
            for (int f = 0; f < 3; f++) ring.store(sl, f, z);
    }
    if (io_warp && lane < TRPL_MAX_EXP) {
        ws->sse[lane] = 0.0;
        ws->pos[lane] = 0;
    }
    __syncwarp();

    // neighbour values carried across iterations and steps
    double Nl, Nr, Pl, Pr;
    {
        double mine[2] = {N[M - 1], P[M - 1]}, vm[2], vp[2];
        cm.template xchg<2, true, false>(mine, 1, 1, vm, vp);
        Nl = vm[0]; Pl = vm[1];
        double mine2[2] = {N[0], P[0]};
        cm.template xchg<2, false, true>(mine2, 1, 1, vm, vp);
        Nr = vp[0]; Pr = vp[1];
    }
    double En = 0.0;   // E on edge M*g + M (owned by the next lane)

    const int t_last = cv.t_last;
    const int plT = a.plT;
    const int n_pl = t_last / plT + 1;
    double keep = 0.0;          // PL sample staged in this lane
    double lp_carry = 0.0;      // log PL of the sample preceding the current block of 32
    double pl0 = 1.0;           // PL(t=0) for self-normalisation

    // PL sample i of this simulation into the caller's buffer (f32 or f64)
    auto store_pl = [&](const int i, const double v) {
        if (a.pl_dtype == TRPL_F32)
            reinterpret_cast<float *>(cv.pl_out)[s * a.pl_stride + i] = (float)v;
        else
            reinterpret_cast<double *>(cv.pl_out)[s * a.pl_stride + i] = v;
    };
    // consume a block of `cnt` staged PL samples starting at index idx0
    // [sec:step-flush]
    auto flush = [&](const int idx0, const int cnt) {
        double val;
        if (emu32) {
            float f = (float)keep;             // value rounded on store into the f32 buffer
            f = f / (float)cv.redim;           // plI_main /= dx**2*dt in float32
            val = (double)f;
        } else {
            val = keep / cv.redim;
        }
        if (cv.pl_out != nullptr && lane < cnt) store_pl(idx0 + lane, val);
        if (a.E == 0) return;
        if (flags & TRPL_F_SELF_NORMALIZE) {
            if (idx0 == 0) pl0 = __shfl_sync(FULL, val, 0);
            val = emu32 ? (double)((float)val / (float)pl0) : val / pl0;
        }
        double lp = val;
        if (flags & TRPL_F_LOG_PL) {
            if (emu32) {
                float f = (float)val;
                if ((double)f < DBL_MIN) f = 0.0f;   // (float)sys.float_info.min == 0  (probs.py:72-73)
                lp = (double)log10f(f);
            } else {
                lp = log10(val < DBL_MIN ? DBL_MIN : val);
            }
        }
        for (int e = 0; e < a.E; e++) {
            const ObsDev &ob = cv.obs[e];
            int pos = ws->pos[e];
            double acc = 0.0;
            for (;;) {
                const int i = pos + lane;
                const int h = (i < ob.n) ? ob.hi[i] : INT_MAX;
                const bool mine = h < idx0 + cnt;
                const unsigned bm = __ballot_sync(FULL, mine);
                if (bm == 0u) break;
                TRPL_DASSERT(pos >= 0 && pos <= ob.n);
                TRPL_DASSERT(!mine || (h - idx0 >= 0 && h - idx0 < cnt && h >= 1));
                const int shi = mine ? h - idx0 : 0;       // 0..cnt-1
                const int slo = shi - 1;                   // -1..cnt-2
                const double y_hi = __shfl_sync(FULL, lp, shi & 31);
                double y_lo = __shfl_sync(FULL, lp, slo & 31);
                if (slo < 0) y_lo = lp_carry;
                double sq = 0.0;
                if (mine) {
                    // scipy interp1d._call_linear: w_hi*y_hi + w_lo*y_lo, no contraction.  An
                    // observation exactly on a grid point has a zero weight on the other neighbour: take
                    // the value itself (the reference's on-grid bypass reads plI directly,
                    // bayeslib.py:173-183), so that 0 * -inf (PL <= 0 under the f32 clamp) is not NaN.
                    const double wh = ob.whi[i], wl = ob.wlo[i];
                    const double yi = (wl == 0.0) ? y_hi : (wh == 0.0) ? y_lo
                                                  : __dadd_rn(__dmul_rn(wh, y_hi), __dmul_rn(wl, y_lo));
                    double err = yi + mag;                  // probs.py:33-38
                    err -= ob.val[i];
                    sq = err * err;
                }
                acc += warp_sum(sq);
                const int took = __popc(bm);
                pos += took;
                if (took < 32) break;
            }
            if (lane == 0) {
                ws->pos[e] = pos;
                ws->sse[e] += acc;
            }
        }
        lp_carry = __shfl_sync(FULL, lp, cnt - 1);
        __syncwarp();
    };

    // Newton system of one species with the other one frozen (pvSimPCR.py:147-216): l, d, u, b of X and
    // the stop-rule partial sum z = sum(|residual| - TOL*|b|) of the current iterate (err < TOL <=> z < 0).
    // `species` is std::true_type for the N system (X = N, Y = P) and std::false_type for the P system
    // (X = P, Y = N); every product of N and P keeps its N-first operand order.
    // -ds = X*(B + CP*P + CN*N) + C_X*np + srh: the factor B + CP*P + CN*N is shared with the rhs, and no
    // product of two per-simulation constants appears inside the loop (see ctab above).  The SRH
    // numerator (for N: P*tp - tauP*np) is evaluated as the equal tauN*P^2 + tauP*N0P0 (one product
    // fewer, no cancellation).
    // [sec:assembly]
    auto assemble = [&](auto species, const double a0, const double (&bX)[M], const double Xl, const double Xr,
                        const double En, double (&l)[M], double (&d)[M], double (&u)[M], double (&b)[M]) {
        constexpr bool IS_N = decltype(species)::value;
        const double (&X)[M] = IS_N ? N : P;
        const double (&Y)[M] = IS_N ? P : N;
        const double tX = IS_N ? tauP : tauN, tY = IS_N ? tauN : tauP;
        const double tX_N0P0 = IS_N ? tauP_N0P0 : tauN_N0P0;
        const double CX = IS_N ? CN : CP, CY = IS_N ? CP : CN;
        double nds_[M];
#pragma unroll
        for (int j = 0; j < M; j++) {
            const double Xj = X[j], Yj = Y[j];
            const double yt = Yj * tY;
            const double tp = fma(Xj, tX, yt);
            const double npp = IS_N ? fma(Xj, Yj, -N0P0) : fma(Yj, Xj, -N0P0);
            const double r = rcp64(tp);
            const double qr = fma(yt, Yj, tX_N0P0) * r;
            const double hr = fma(CY, Yj, CX * Xj) + rate;
            const double nds = fma(Yj, hr, fma(CX, npp, qr * r));               // = -ds
            nds_[j] = nds;
            b[j] = fma(nds, Xj, -fma(hr + r, npp, bX[j]));
        }
        // transport rows.  The diagonal takes exactly the rounded off-diagonals of the two
        // neighbouring rows (d_j = a0 - u_{j-1} - l_{j+1} - ds, pvSimPCR.py:159): the column sums of
        // the transport part vanish in floating point, i.e. the step conserves carriers to the
        // last bit -- a diagonal rebuilt from E differences does not, and that noise ends up in
        // PL = rate*(sum N*P - L*N0*P0) once the excess has decayed (measured: stiff-regime agreement
        // with the CPU restatement 96.9 % -> 94.9 %, profiles/r02_variants.txt).
        {
            const double D = IS_N ? DN : DP;
            const double hDu = IS_N ? -hDN : hDP;    // D/2 with the sign of the field term in u
            const double cu0 = sel(ev[0], fma(hDu, E[0], -D), 0.0);      // u of the previous lane's last row
            const double clM = sel(ev[M], fma(-hDu, En, -D), 0.0);         // l of the next lane's first row
#pragma unroll
            for (int j = 0; j < M; j++) {
                const double Ep = (j < M - 1) ? E[j + 1] : En;
                l[j] = fma(-hDu, E[j], -D);                                      // N: DN*(+E/2 - 1), P: DP*(-E/2 - 1)
                u[j] = fma(hDu, Ep, -D);                                        // N: DN*(-E/2 - 1), P: DP*(+E/2 - 1)
                if (PAD) {
                    l[j] = sel(nv[j] && ev[j], l[j], 0.0);
                    u[j] = sel(nv[j] && ev[j + 1], u[j], 0.0);
                }
            }
            if (!PAD) {
                l[0] = sel(ev[0], l[0], 0.0);
                u[M - 1] = sel(ev[M], u[M - 1], 0.0);
            }
#pragma unroll
            for (int j = 0; j < M; j++)
                d[j] = ((a0 - ((j == 0) ? cu0 : u[j - 1])) - ((j == M - 1) ? clM : l[j + 1])) + nds_[j];
        }
        // [sec:surface] surface recombination rows (pvSimPCR.py:164-170) + missing-neighbour fix
        {
            double Nb = N[M - 1], Pb = P[M - 1];        // back-surface node of this lane
            if (PAD) {
#pragma unroll
                for (int j = 0; j < M - 1; j++) { Nb = (j == jl) ? N[j] : Nb; Pb = (j == jl) ? P[j] : Pb; }
            }
            const double Ns = is_first ? N[0] : Nb;
            const double Ps = is_first ? P[0] : Pb;
            const double Xs = IS_N ? Ns : Ps, Ys = IS_N ? Ps : Ns;
            const double rs = rcp64(Ns + Ps);
            const double srs = srf * rs;
            const double nd = fma(Ys, Ys, N0P0) * (srs * rs);                   // = -ds0
            const double db = fma(-nd, Xs, fma(Ns, Ps, -N0P0) * srs);
            if (PAD) {
#pragma unroll
                for (int j = 0; j < M; j++) {
                    const bool at = (is_first && j == 0) || (is_last && j == jl);
                    d[j] += at ? nd : 0.0;
                    b[j] -= at ? db : 0.0;
                }
            } else {
                d[0] += is_first ? nd : 0.0;
                b[0] -= is_first ? db : 0.0;
                d[M - 1] += is_last ? nd : 0.0;
                b[M - 1] -= is_last ? db : 0.0;
            }
        }
        if (PAD) {
#pragma unroll
            for (int j = 0; j < M; j++) {
                d[j] = sel(nv[j], d[j], 1.0);
                b[j] = sel(nv[j], b[j], 0.0);
            }
        }
        // [sec:residual] L1 residual of the current iterate         (pvSimPCR.py:172, :14-40)
        double z = 0.0;
#pragma unroll
        for (int j = 0; j < M; j++) {
            const double xm = (j == 0) ? Xl : X[j - 1];
            const double xp = (j == M - 1) ? Xr : X[j + 1];
            const double res = fma(l[j], xm, fma(d[j], X[j], fma(u[j], xp, -b[j])));
            z = fma(-TOL, fabs(b[j]), z + fabs(res));
        }
        if (PADM == 1) z = dummy ? 0.0 : z;
        return z;
    };

    // =========================================================================================
    // time loop (pvSimPCR.py:237-293): t = 0 .. t_last, PL(t) emitted from the state at time t
    // =========================================================================================
    // [sec:step]
    // time-loop state.  The declaration order matters to ptxas: other orders change the register
    // assignment of the fine-grid kernel (+5 three-register DFMAs, profiles/r03_refactor_sass_budget.txt).
    bool failed = false;
    int t_next_pl = 0;
    int t;
    int pl_idx = 0;             // index of the next PL sample
    int status = 0;
    long long iters_total = 0;
    for (t = 0; t <= t_last; t++) {
        // [sec:step-PL] ---- PL(t) = rate * (sum_n N*P - L*N0*P0)             (pvSimPCR.py:276-281)
        bool emitted = false;
        if (t == t_next_pl) {
            emitted = true;
            double part = 0.0;
#pragma unroll
            for (int j = 0; j < M; j++) part = fma(N[j], P[j], part);
            if (PADM == 1) part = dummy ? 0.0 : part;
            const double tot = cm.sum(part);
            const double plraw = rate * (tot + mLN0P0);
            if (lane == (pl_idx & 31)) keep = plraw;
            t_next_pl += plT;
            pl_idx++;
        }

        // [sec:step-bdf] ---- BDF coefficients, order ramp 1..5              (pvSimPCR.py:241-250)
        // (looked up every step on purpose: as step-local values read from the constant bank with a uniform
        // index they stay in uniform registers; hoisted out of the loop they become loop-carried vector
        // registers and 29 more DFMAs per iteration turn into the 3-cycle three-register kind.  A table
        // lookup costs 6 uniform loads; the five-way select it replaces cost 57 moves per step.)
        int order = t + 1;
        if (order > 5) order = 5;
        if (order > a.max_order) order = a.max_order;
        const double a0 = c_bdf[order - 1][0], a1 = c_bdf[order - 1][1], a2 = c_bdf[order - 1][2];
        const double a3 = c_bdf[order - 1][3], a4 = c_bdf[order - 1][4], a5 = c_bdf[order - 1][5];
        // [sec:step-history] ---- history sums bU = a1 U(t) + ... + a5 U(t-4) (pvSimPCR.py:133-135)
        double bN[M], bP[M], bE[M];
#pragma unroll
        for (int j = 0; j < M; j++) {
            bN[j] = a1 * N[j];
            bP[j] = a1 * P[j];
            bE[j] = a1 * E[j];
        }
        {
            const double ac[4] = {a2, a3, a4, a5};
#pragma unroll
            for (int i = 1; i <= 4; i++) {
                const int slot = (t - i) & 3;
                double h[M];
                ring.load(slot, 0, h);
#pragma unroll
                for (int j = 0; j < M; j++) bN[j] = fma(ac[i - 1], h[j], bN[j]);
                ring.load(slot, 1, h);
#pragma unroll
                for (int j = 0; j < M; j++) bP[j] = fma(ac[i - 1], h[j], bP[j]);
                ring.load(slot, 2, h);
#pragma unroll
                for (int j = 0; j < M; j++) bE[j] = fma(ac[i - 1], h[j], bE[j]);
            }
            const int slot = t & 3;    // level t replaces level t-4
            ring.store(slot, 0, N);
            ring.store(slot, 1, P);
            ring.store(slot, 2, E);
        }
        double bEn = 0.0;              // history sum of the next lane's first edge (W > 1 only)
        if constexpr (W > 1) bEn = cm.from_next(bE[0]);

        // [sec:loop] ---- Newton / Gauss-Seidel iteration                   (pvSimPCR.py:147-216)
        int it = 0;
        bool nonfinite = false;
        for (;;) {
            double l[M], d[M], u[M], b[M];
            bool converged_now = false, nonfinite_now = false;
            // [sec:N] ======== N system (P, E frozen) ========
            const double zN = assemble(std::true_type(), a0, bN, Nl, Nr, En, l, d, u, b);
            // [sec:N-solve]
            Nl = tridiag_solve<M, W>(l, d, u, b, N, cm, Nr);
            // [sec:P] ======== P system (new N) ========
            const double zP = assemble(std::false_type(), a0, bP, Pl, Pr, En, l, d, u, b);
            // [sec:stop-rule] ---- stop decision for THIS iteration (pvSimPCR.py:213-216): both L1
            // residuals are known here, before the P solve; reducing them now lets the shuffle
            // chain overlap the solve.
            if constexpr (W == 1) cm.stop_rule(zN, zP, converged_now, nonfinite_now);
            else cm.stop_post(zN, zP);
            // [sec:P-solve]
            Pl = tridiag_solve<M, W>(l, d, u, b, P, cm, Pr);
            if constexpr (W > 1) cm.stop_collect(converged_now, nonfinite_now);

            // [sec:E-update] ======== E update on interior edges             (pvSimPCR.py:205-209)
#pragma unroll
            for (int j = 0; j < M; j++) {
                const double Nm = (j == 0) ? Nl : N[j - 1];
                const double Pm = (j == 0) ? Pl : P[j - 1];
                const double den = fma(hLamDP, P[j] + Pm, fma(hLamDN, N[j] + Nm, a0));
                const double num = fma(LamDP, P[j] - Pm, fma(-LamDN, N[j] - Nm, -bE[j]));
                E[j] = sel(ev[j], num * rcp64(den), 0.0);
            }
            if constexpr (W == 1) {
                En = sel(ev[M], cm.from_next(E[0]), 0.0);      // no edge beyond the back surface
            } else {
                // the next lane's first edge from values this lane already holds (bit-identical to what
                // the owner computes): saves a block barrier per iteration
                const double den = fma(hLamDP, Pr + P[M - 1], fma(hLamDN, Nr + N[M - 1], a0));
                const double num = fma(LamDP, Pr - P[M - 1], fma(-LamDN, Nr - N[M - 1], -bEn));
                En = sel(ev[M], num * rcp64(den), 0.0);
            }

            // [sec:loop] ======== stop rule (pvSimPCR.py:213-216): decided by the flags computed before the P solve
            it++;
            if (nonfinite_now) { nonfinite = true; break; }
            if (converged_now) break;
            if (it >= a.max_iter) break;
        }
        // [sec:step]
        iters_total += it;
        if (nonfinite || it >= a.max_iter) {                 // pvSimPCR.py:269-274
            status |= nonfinite ? TRPL_ST_NONFINITE : TRPL_ST_NOCONV;
            failed = true;
            // the reference stops before emitting PL(t): un-count the sample staged for this step
            if (emitted) pl_idx--;
            break;
        }
        if (io_warp && emitted && (pl_idx & 31) == 0) flush(pl_idx - 32, 32);
    }

    // [sec:tail] ---- partially filled block; after a failure everything from pl_idx on is NaN
    if (io_warp && (pl_idx & 31)) flush(pl_idx & ~31, pl_idx & 31);
    if (io_warp && failed && cv.pl_out != nullptr) {
        const double qnan = __longlong_as_double(0x7ff8000000000000LL);
        for (int i = pl_idx + lane; i < n_pl; i += 32) store_pl(i, qnan);
    }

    // ---- results
    __syncwarp();
    if (io_warp && lane == 0) {
        const long long cs = (long long)c * a.S + s;
        if (a.status) a.status[cs] = status;
        if (a.iters) a.iters[cs] = iters_total;
    }
    if (io_warp && a.sse != nullptr && lane < a.E) {
        double v = ws->sse[lane];
        if (failed && ws->pos[lane] < cv.obs[lane].n) v = __longlong_as_double(0x7ff8000000000000LL);
        a.sse[((long long)lane * a.C + c) * a.S + s] = v;
    }
    __syncwarp();
}

// [sec:kernel]
template <int M, bool PAD>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, MIN_CTAS_PER_SM)
trpl_sim_kernel(const __grid_constant__ KArgs a)
{
    extern __shared__ __align__(16) double smem[];
    __shared__ WarpScratch scratch[WARPS_PER_CTA];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *ring_warp = smem + (size_t)warp * (4 * 3 * M * 32 + RING_CANARY);
    if (TRPL_DEBUG && lane == 0) reinterpret_cast<unsigned long long *>(ring_warp + 4 * 3 * M * 32)[0] = CANARY_WORD;
    const unsigned long long total = (unsigned long long)a.S * (unsigned long long)a.C;
    Comm<1> cm(lane);
    for (;;) {
        unsigned long long item = 0;
        if (lane == 0) item = atomicAdd(a.counter, 1ULL);
        item = __shfl_sync(FULL, item, 0);
        if (item >= total) break;
        // items are issued curve-major, longest curve first, so short ones fill the tail of the launch
        const int c = a.curve_order[(int)(item / (unsigned long long)a.S)];
        const long long s = (long long)(item % (unsigned long long)a.S);
        run_sim<M, PAD ? 2 : 0, 1>(a, c, s, ring_warp, &scratch[warp], lane, cm);
        if (TRPL_DEBUG) TRPL_DASSERT(reinterpret_cast<unsigned long long *>(ring_warp + 4 * 3 * M * 32)[0] == CANARY_WORD);
    }
}

// Fine grids: one CTA of W warps per simulation, M nodes per lane (L <= 32*M*W); PADM as in run_sim
// (1: L % M == 0, 2: any L).
template <int W, int M, int PADM>
__global__ void __launch_bounds__(W * 32, 1)
trpl_sim_cta_kernel(const __grid_constant__ KArgs a)
{
    extern __shared__ __align__(16) double smem[];
    __shared__ WarpScratch scratch;
    __shared__ unsigned long long next_item;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *ring_warp = smem + (size_t)warp * (4 * 3 * M * 32 + RING_CANARY);
    if (TRPL_DEBUG && lane == 0) reinterpret_cast<unsigned long long *>(ring_warp + 4 * 3 * M * 32)[0] = CANARY_WORD;
    Comm<W> cm(threadIdx.x, smem + (size_t)W * (4 * 3 * M * 32 + RING_CANARY), blockIdx.x & (W - 1));
    const unsigned long long total = (unsigned long long)a.S * (unsigned long long)a.C;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) next_item = atomicAdd(a.counter, 1ULL);
        __syncthreads();
        const unsigned long long item = next_item;
        if (item >= total) break;
        const int c = a.curve_order[(int)(item / (unsigned long long)a.S)];
        const long long s = (long long)(item % (unsigned long long)a.S);
        run_sim<M, PADM, W>(a, c, s, ring_warp, &scratch, lane, cm);
        if (TRPL_DEBUG) TRPL_DASSERT(reinterpret_cast<unsigned long long *>(ring_warp + 4 * 3 * M * 32)[0] == CANARY_WORD);
    }
}


}  // namespace trpl
