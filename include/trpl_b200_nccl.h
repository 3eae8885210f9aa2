/*
 * trpl_b200_nccl.h -- C ABI of libtrpl_b200_nccl.so: the multi-GPU exchange at the end of a run
 * (merge the per-rank likelihood tables, normalise the posterior over all ranks' samples) over NCCL,
 * for hosts that bind the C ABI directly and have no torch.distributed (INTEGRATION.md, route C).
 * A companion of libtrpl_b200.so: it is linked with libnccl.so.2, the core library is not.
 *
 * Conventions of trpl_b200.h: pointers named d_* are DEVICE pointers; stream-ordered calls are
 * asynchronous on `stream` (a cudaStream_t passed as void*, NULL = legacy default stream) of the
 * communicator's device and never synchronise the host; the return value is 0 or a negative
 * TRPL_E* code, and arguments are validated before the device is entered.
 *
 * One process per GPU, one communicator per process.  Samples are sharded by columns, contiguously
 * and balanced: rank r owns columns [lo, hi) with base = n_total / nranks, rem = n_total % nranks,
 * lo = r*base + min(r, rem), hi = lo + base + (r < rem)   (distributed.shard_bounds).
 *
 * Reference interfaces replaced (paths relative to this repository):
 *   trpl_allgather_rows      distributed.gather_rows                          distributed.py:17-29
 *   trpl_logsumexp_nccl      distributed.global_logsumexp                     distributed.py:32-44
 *   trpl_allreduce_sum_nccl  distributed.merge_block_cyclic, posterior._allreduce_sum
 *   trpl_posterior_weights_dev  trpl_posterior_weights with a device-resident lse per row
 */
#ifndef TRPL_B200_NCCL_H
#define TRPL_B200_NCCL_H

#include <stdint.h>

#include "trpl_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define TRPL_NCCL_ID_BYTES 128  /* size of the unique id rank 0 hands to every rank            */

/* error codes beyond those of trpl_b200.h (TRPL_EINVAL, TRPL_ECUDA, TRPL_ENODEVICE are reused) */
#define TRPL_ENCCL      -5      /* NCCL error (see trpl_nccl_last_error)                        */
#define TRPL_ETIMEDOUT  -6      /* the communicator did not become ready in time; it is aborted */

typedef struct trpl_comm trpl_comm;   /* opaque: NCCL communicator, rank, nranks, device */

/* Runtime NCCL version code (ncclGetVersion, e.g. 22703 for 2.27.3), or a negative code.     */
int trpl_nccl_version(void);

/* Thread-local text of the last NCCL or CUDA failure of this library.                         */
const char *trpl_nccl_last_error(void);

/* Writes TRPL_NCCL_ID_BYTES bytes to the host buffer id_out.  Called on rank 0 only; every rank
 * then passes the same bytes to trpl_nccl_comm_init.                                          */
int trpl_nccl_unique_id(void *id_out);

/* Joins the communicator of `nranks` ranks on CUDA device `device`.  The call returns once every
 * rank has joined, or after timeout_ms (> 0) with TRPL_ETIMEDOUT, having aborted its part, so a
 * rank that never arrives cannot hang the others forever.  Later calls that must wait for peers
 * to set up a connection use the same limit.                                                  */
int trpl_nccl_comm_init(const void *id, int nranks, int rank, int device, int timeout_ms,
                        trpl_comm **out);

/* Flushes and releases the communicator; NULL is a no-op.                                      */
int trpl_nccl_comm_destroy(trpl_comm *c);

int trpl_nccl_rank_info(const trpl_comm *c, int *rank, int *nranks, int *device);

/* d_all[rows][n_total] on every rank from every rank's d_local[rows][ld_local] holding its n_local
 * columns of the shard rule above (TRPL_EINVAL when n_local disagrees with it).  d_local may be
 * NULL when n_local is 0.  For a sample matrix X[S][ncol], pass X transposed ([ncol][S]).      */
int trpl_allgather_rows(trpl_comm *c, const double *d_local, int64_t rows, int64_t ld_local,
                        int64_t n_local, int64_t n_total, double *d_all, void *stream);

/* d_lse[r] = log sum_i exp(x[r][i]) over ALL ranks' columns of row r, with this rank's
 * d_x[rows][ld] holding n_local columns.  NaN entries are skipped and -inf entries weigh 0, as in
 * trpl_lse_partial; a row with no finite entry on any rank gives -inf.                         */
int trpl_logsumexp_nccl(trpl_comm *c, const double *d_x, int64_t rows, int64_t ld, int64_t n_local,
                        double *d_lse, void *stream);

/* d_w[r][i] = exp(d_lnp[r][i] - d_lse[r]) for i < n, both [rows][ld]; NaN -> 0, and a row with
 * d_lse[r] = -inf is all 0.  Bit-identical to trpl_posterior_weights for the same lse value.
 * Needs no communicator.                                                                        */
int trpl_posterior_weights_dev(const double *d_lnp, int64_t rows, int64_t ld, int64_t n,
                               const double *d_lse, double *d_w, int device, void *stream);

/* In-place sum of d_buf[n] over all ranks (block-cyclic likelihood tables, histogram and
 * moment sums).                                                                                 */
int trpl_allreduce_sum_nccl(trpl_comm *c, double *d_buf, int64_t n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TRPL_B200_NCCL_H */
