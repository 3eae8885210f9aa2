/*
 * trpl_b200_ensemble.h -- the affine-invariant ensemble sampler (stretch move, Goodman & Weare 2010,
 * in the two-half form of emcee, Foreman-Mackey et al. 2013) on the device: proposals and the
 * accept/reject step around trpl_solve_loglik.  Part of libtrpl_b200.so; conventions of trpl_b200.h
 * (d_* are device pointers, host arrays are only read during the call, calls are asynchronous on
 * `stream` of `device`, the return value is 0 or a negative TRPL_E* code, arguments are validated
 * before the device is entered).
 *
 * Ensemble: n_walkers = W walkers (W even), half A = walkers [0, W/2), half B = [W/2, W).  One step
 * moves A against the complement B, then B against the updated A.  A call handles n walkers of ONE
 * half, global indices [first_walker, first_walker + n), so a rank passes its shard of the half.
 *
 * Coordinates: moves happen in the prior's coordinates, log10(x) for do_log columns and x otherwise;
 * the prior is uniform on the box [minx, maxx] there.  Fixed columns (minx == maxx) keep their value;
 * override_flags (bit 0: column 2 <- 3, bit 1: 6 <- 5, bit 2: 8 <- 7, as trpl_random_grid) copy the
 * source column after the move.  d = number of remaining (free) columns.
 *
 * Randomness: Philox4x32-10 with key = seed and counter (walker lo, walker hi, step, tag): tag 1 gives
 * the partner and z, tag 2 the accept uniform (trpl_random_grid uses tag 0).  A chain is therefore a
 * pure function of (seed, initial walkers, likelihood), whatever the sharding.
 */
#ifndef TRPL_B200_ENSEMBLE_H
#define TRPL_B200_ENSEMBLE_H

#include <stdint.h>

#include "trpl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Proposals of the n walkers d_x[n][ldx] (engine units).  d_comp holds the complement half, column
 * j of its walker k at d_comp[j*ld_comp + k] (X transposed, the layout trpl_allgather_rows returns).
 * For walker g = first_walker + i: partner p uniform in [0, W/2), z = ((a-1)u + 1)^2 / a, y = x_p +
 * z (x_g - x_p) in prior coordinates, written to d_y[i][ldy] in engine units with d_logq[i] =
 * (d-1) ln z.  A proposal outside the box is never written: d_y gets the walker's own row and
 * d_logq = -inf, so it can go to the solver unchanged and is rejected.  W must be even and >= 2 max(d, 1),
 * and a > 1.                                                                                     */
int trpl_stretch_propose(const double *d_x, int64_t n, int64_t ldx, int64_t first_walker, int64_t n_walkers,
                         const double *d_comp, int64_t ld_comp, const double *minx, const double *maxx,
                         const int32_t *do_log, int ncol, int override_flags, double a, uint64_t seed,
                         uint32_t step, double *d_y, int64_t ldy, double *d_logq, int device, void *stream);

/* Accept/reject of the proposals of trpl_stretch_propose given their log-likelihoods d_lnl_y[n].
 * Target: log pi = lnL / temperature inside the box.  NaN lnL counts as -inf; a -inf proposal (or
 * d_logq = -inf) never replaces a walker, a finite one always replaces a -inf walker; otherwise accept
 * iff ln u < logq + (lnL_y - lnL_x) / temperature with u in (0, 1].  Accepted walkers get the first
 * ncol columns of their proposal in d_x and its lnL in d_lnl (both in place); d_accepted[i] (may be
 * NULL) is 1 for an accepted proposal, else 0.                                                   */
int trpl_stretch_accept(double *d_x, int64_t n, int64_t ldx, int64_t first_walker, int64_t n_walkers, int ncol,
                        double *d_lnl, const double *d_y, int64_t ldy, const double *d_lnl_y,
                        const double *d_logq, double temperature, uint64_t seed, uint32_t step,
                        int32_t *d_accepted, int device, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TRPL_B200_ENSEMBLE_H */
