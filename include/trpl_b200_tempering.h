/*
 * trpl_b200_tempering.h -- parallel tempering of the ensemble sampler (trpl_b200_ensemble.h) on the device:
 * K copies ("rungs") of the ensemble sample lnL / T_t on a temperature ladder T_0 < T_1 < ... < T_{K-1},
 * and neighbouring rungs exchange walkers.  Part of libtrpl_b200.so; conventions of trpl_b200.h (d_* are
 * device pointers, host arrays are only read during the call, calls are asynchronous on `stream` of
 * `device`, the return value is 0 or a negative TRPL_E* code, arguments are validated before the device
 * is entered).
 *
 * Layout: every rung holds an ensemble of W = n_walkers walkers with the halves of trpl_b200_ensemble.h.
 * A call handles the same n walkers of ONE half, global indices [first_walker, first_walker + n) inside
 * the rung, in every rung: walker i of rung t is row t*n + i of d_x (row stride ldx), and its lnL,
 * proposal, log q and flags are entry t*n + i of their arrays.
 *
 * Ladder: `temperatures` is a host array of n_rungs entries, strictly increasing, with T_0 > 0; only the
 * last entry may be +inf (that rung samples the prior).  1 <= n_rungs <= TRPL_MAX_RUNGS.
 *
 * Randomness: Philox4x32-10 with key = seed and counter (G lo, G hi, step, tag), G = t*W + g for walker g
 * of rung t.  Rung 0 therefore draws exactly what trpl_stretch_propose / trpl_stretch_accept draw (tags 1
 * and 2); swaps use tag 3.
 */
#ifndef TRPL_B200_TEMPERING_H
#define TRPL_B200_TEMPERING_H

#include <stdint.h>

#include "trpl_b200.h"

#define TRPL_MAX_RUNGS 64
#define TRPL_TAG_SWAP 3

#ifdef __cplusplus
extern "C" {
#endif

/* trpl_stretch_propose for every rung: rung t's walkers (rows t*n .. t*n + n - 1 of d_x) move against rung
 * t's complement, the ncol rows t*ncol .. t*ncol + ncol - 1 of d_comp [n_rungs*ncol][ld_comp] (the layout
 * one trpl_allgather_rows of the other half's [n_rungs*ncol, n_other] transpose returns).  d_y and d_logq
 * get n_rungs*n entries.  With n_rungs = 1 this is trpl_stretch_propose, bit for bit.               */
int trpl_tempered_propose(const double *d_x, int64_t n, int64_t ldx, int64_t first_walker, int64_t n_walkers,
                          int n_rungs, const double *d_comp, int64_t ld_comp, const double *minx,
                          const double *maxx, const int32_t *do_log, int ncol, int override_flags, double a,
                          uint64_t seed, uint32_t step, double *d_y, int64_t ldy, double *d_logq, int device,
                          void *stream);

/* trpl_stretch_accept for every rung, rung t at temperature T_t: accept iff
 * ln u < logq + (lnL_y - lnL_x) / T_t, with the NaN / -inf rules of trpl_stretch_accept.  At T = +inf an
 * in-box proposal is accepted with probability min(1, z^(d-1)).  With n_rungs = 1 this is
 * trpl_stretch_accept at temperature T_0, bit for bit.                                            */
int trpl_tempered_accept(double *d_x, int64_t n, int64_t ldx, int64_t first_walker, int64_t n_walkers,
                         int n_rungs, const double *temperatures, int ncol, double *d_lnl, const double *d_y,
                         int64_t ldy, const double *d_lnl_y, const double *d_logq, uint64_t seed, uint32_t step,
                         int32_t *d_accepted, int device, void *stream);

/* Replica exchange between neighbouring rungs, in place.  Walker i of rung t pairs with walker i of rung
 * t - 1, for t = n_rungs - 1 down to 1 (the hottest pair first, so a state can fall several rungs in one
 * call).  With beta = 1 / T (0 at +inf) and NaN lnL counted as -inf: no swap if both lnL are -inf;
 * otherwise r = (beta_{t-1} - beta_t) (lnL_t - lnL_{t-1}), swap if r = +inf, not if r = -inf, else iff
 * ln u < r with u in (0, 1] from counter (t*W + g, step, TRPL_TAG_SWAP).  A swap exchanges the first
 * ncol columns and the raw lnL of the two rows.  d_swapped[(t-1)*n + i] (may be NULL, n_rungs - 1
 * entries per walker) is 1 for a swap, else 0.                                                     */
int trpl_tempered_swap(double *d_x, int64_t n, int64_t ldx, int64_t first_walker, int64_t n_walkers, int n_rungs,
                       const double *temperatures, int ncol, double *d_lnl, uint64_t seed, uint32_t step,
                       int32_t *d_swapped, int device, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TRPL_B200_TEMPERING_H */
