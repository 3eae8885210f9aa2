// trpl_nccl.cu -- C ABI of libtrpl_b200_nccl.so (see include/trpl_b200_nccl.h): the end-of-run exchange
// of a multi-GPU run over NCCL, for hosts without torch.distributed.  Linked with -lnccl; the core library
// libtrpl_b200.so is not.
//
// Replaces distributed.gather_rows / global_logsumexp / merge_block_cyclic and posterior._allreduce_sum.
// The shard-local log-sum-exp pass is the one trpl_lse_partial runs (same kernels from trpl_aux_kernels.cuh,
// same grid), and the lse stays on the device up to the weights: nothing here synchronises the host with
// the stream.
//
// Communicators are created non-blocking (ncclConfig_t::blocking = 0), so that joining and any later call
// that has to wait for peers (lazy connection set-up) can be given up after the communicator's timeout
// instead of hanging the process when a rank never arrives.
#include <string.h>

#include <chrono>
#include <new>
#include <thread>

#include <nccl.h>

#include "trpl_b200_nccl.h"
#include "trpl_common.cuh"
#include "trpl_aux_kernels.cuh"
#include "trpl_host.cuh"

static_assert(sizeof(ncclUniqueId) == TRPL_NCCL_ID_BYTES, "TRPL_NCCL_ID_BYTES must match ncclUniqueId");

struct trpl_comm {
    ncclComm_t comm;        // nullptr once aborted after a timeout
    int rank, nranks, device, timeout_ms;
};

using namespace trpl;

namespace {

// ---- global log-sum-exp around the shard-local (max, sum) pairs part[rows][2] ---------------------------
__global__ void trpl_lse_split_kernel(const double *part, long long rows, double *gmax)
{
    const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (r < rows) gmax[r] = part[2 * r];
}
// s[r] = local sum rescaled to the global maximum; a rank without a finite entry in row r adds 0
// (distributed.global_logsumexp)
__global__ void trpl_lse_rescale_kernel(const double *part, const double *gmax, long long rows, double *s)
{
    const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const double m = part[2 * r];
    s[r] = isfinite(m) ? part[2 * r + 1] * exp(m - gmax[r]) : 0.0;
}
// lse[r] = gmax[r] + log(sum over ranks); -inf + log(0) = -inf for a row with no finite entry anywhere
__global__ void trpl_lse_finalize_kernel(const double *gmax, long long rows, double *lse)
{
    const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (r < rows) lse[r] = gmax[r] + log(lse[r]);
}

// Rows of weights with a device-resident lse per row.  A row whose lse is -inf has no finite entry on any
// rank, so all its weights are 0 (exp(-inf - -inf) would be NaN).
__global__ void trpl_weights_rows_kernel(const double *lnp, long long rows, long long ld, long long n,
                                         const double *lse, double *w)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < rows * n; i += stride) {
        const long long r = i / n, j = i - r * n;
        const double l = lse[r];
        w[r * ld + j] = (l == -INFINITY) ? 0.0 : posterior_weight(lnp[r * ld + j], l);
    }
}

// ---- host side -------------------------------------------------------------------------------------------
// g_cuda_err (trpl_host.cuh) holds the text of the last NCCL failure too: trpl_nccl_last_error returns it.
int nccl_fail(ncclResult_t r, ncclComm_t comm, const char *what)
{
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s (%s)", what, ncclGetErrorString(r), ncclGetLastError(comm));
    return TRPL_ENCCL;
}

// Waits until the host-side part of a call on a non-blocking communicator is done (r == ncclInProgress
// until then), for at most timeout_ms.  Does not wait for the stream.
int nccl_settle(ncclComm_t comm, ncclResult_t r, int timeout_ms, const char *what)
{
    using clk = std::chrono::steady_clock;
    const auto deadline = clk::now() + std::chrono::milliseconds(timeout_ms);
    while (r == ncclInProgress) {
        if (clk::now() > deadline) {
            snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: not ready after %d ms", what, timeout_ms);
            return TRPL_ETIMEDOUT;
        }
        std::this_thread::sleep_for(std::chrono::microseconds(200));
        const ncclResult_t q = ncclCommGetAsyncError(comm, &r);
        if (q != ncclSuccess) r = q;
    }
    return r == ncclSuccess ? TRPL_OK : nccl_fail(r, comm, what);
}

// nccl_settle for a call on c; a timeout aborts the communicator (its peers are gone or stuck)
int settle(trpl_comm *c, ncclResult_t r, const char *what)
{
    const int rc = nccl_settle(c->comm, r, c->timeout_ms, what);
    if (rc == TRPL_ETIMEDOUT) {
        ncclCommAbort(c->comm);
        c->comm = nullptr;
    }
    return rc;
}

int aborted()
{
    snprintf(g_cuda_err, sizeof(g_cuda_err), "the communicator was aborted after a timeout");
    return TRPL_ENCCL;
}

// distributed.shard_bounds
void shard_bounds(int64_t n, int rank, int nranks, int64_t *lo, int64_t *hi)
{
    const int64_t base = n / nranks, rem = n % nranks;
    *lo = rank * base + (rank < rem ? rank : rem);
    *hi = *lo + base + (rank < rem ? 1 : 0);
}

unsigned small_grid(long long rows) { return (unsigned)((rows + 255) / 256); }

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int trpl_nccl_version(void)
{
    int v = 0;
    const ncclResult_t r = ncclGetVersion(&v);
    return r == ncclSuccess ? v : nccl_fail(r, nullptr, "ncclGetVersion");
}

const char *trpl_nccl_last_error(void) { return g_cuda_err; }

int trpl_nccl_unique_id(void *id_out)
{
    if (!id_out) return TRPL_EINVAL;
    ncclUniqueId id;
    const ncclResult_t r = ncclGetUniqueId(&id);
    if (r != ncclSuccess) return nccl_fail(r, nullptr, "ncclGetUniqueId");
    memcpy(id_out, &id, sizeof(id));
    return TRPL_OK;
}

int trpl_nccl_comm_init(const void *id, int nranks, int rank, int device, int timeout_ms, trpl_comm **out)
{
    if (!id || !out || nranks < 1 || rank < 0 || rank >= nranks || timeout_ms <= 0) return TRPL_EINVAL;
    *out = nullptr;
    return on_device(device, [&] {
        ncclUniqueId uid;
        memcpy(&uid, id, sizeof(uid));
        ncclConfig_t cfg = NCCL_CONFIG_INITIALIZER;
        cfg.blocking = 0;
        ncclComm_t comm = nullptr;
        const ncclResult_t r = ncclCommInitRankConfig(&comm, nranks, uid, rank, &cfg);
        if (r != ncclSuccess && r != ncclInProgress) {
            const int rc = nccl_fail(r, comm, "ncclCommInitRankConfig");
            if (comm) ncclCommAbort(comm);
            return rc;
        }
        const int rc = nccl_settle(comm, r, timeout_ms, "ncclCommInitRankConfig");
        if (rc) {
            ncclCommAbort(comm);
            return rc;
        }
        trpl_comm *c = new (std::nothrow) trpl_comm{comm, rank, nranks, device, timeout_ms};
        if (!c) {
            ncclCommAbort(comm);
            return cuda_fail(cudaErrorMemoryAllocation, "trpl_nccl_comm_init");
        }
        *out = c;
        return TRPL_OK;
    });
}

int trpl_nccl_comm_destroy(trpl_comm *c)
{
    if (!c) return TRPL_OK;
    const int rc = on_device(c->device, [&] {
        if (!c->comm) return TRPL_OK;
        const int rc = nccl_settle(c->comm, ncclCommFinalize(c->comm), c->timeout_ms, "ncclCommFinalize");
        if (rc) {
            ncclCommAbort(c->comm);
            return rc;
        }
        const ncclResult_t r = ncclCommDestroy(c->comm);
        return r == ncclSuccess ? TRPL_OK : nccl_fail(r, nullptr, "ncclCommDestroy");
    });
    delete c;
    return rc;
}

int trpl_nccl_rank_info(const trpl_comm *c, int *rank, int *nranks, int *device)
{
    if (!c || !rank || !nranks || !device) return TRPL_EINVAL;
    *rank = c->rank;
    *nranks = c->nranks;
    *device = c->device;
    return TRPL_OK;
}

int trpl_allgather_rows(trpl_comm *c, const double *d_local, int64_t rows, int64_t ld_local, int64_t n_local,
                        int64_t n_total, double *d_all, void *stream)
{
    if (!c || !d_all || rows < 1 || n_total < 0 || n_local < 0 || ld_local < n_local || (n_local > 0 && !d_local))
        return TRPL_EINVAL;
    int64_t lo, hi;
    shard_bounds(n_total, c->rank, c->nranks, &lo, &hi);
    if (n_local != hi - lo) return TRPL_EINVAL;
    return on_device(c->device, [&] {
        if (!c->comm) return aborted();
        cudaStream_t st = (cudaStream_t)stream;
        // every rank broadcasts each of its rows straight into place in d_all; one group, so NCCL fuses them
        ncclResult_t first = ncclGroupStart();
        for (int r = 0; r < c->nranks && first == ncclSuccess; r++) {
            int64_t rlo, rhi;
            shard_bounds(n_total, r, c->nranks, &rlo, &rhi);
            if (rhi == rlo) continue;
            for (int64_t i = 0; i < rows && first == ncclSuccess; i++) {
                double *dst = d_all + i * n_total + rlo;
                const double *src = (r == c->rank) ? d_local + i * ld_local : dst;
                first = ncclBroadcast(src, dst, (size_t)(rhi - rlo), ncclDouble, r, c->comm, st);
            }
        }
        const ncclResult_t end = ncclGroupEnd();        // always closes the group
        if (first != ncclSuccess) return nccl_fail(first, c->comm, "ncclBroadcast");
        return settle(c, end, "trpl_allgather_rows");
    });
}

int trpl_logsumexp_nccl(trpl_comm *c, const double *d_x, int64_t rows, int64_t ld, int64_t n_local,
                        double *d_lse, void *stream)
{
    if (!c || !d_lse || rows < 1 || n_local < 0 || ld < n_local || (n_local > 0 && !d_x)) return TRPL_EINVAL;
    return on_device(c->device, [&] {
        if (!c->comm) return aborted();
        cudaStream_t st = (cudaStream_t)stream;
        Scratch scratch(st);                         // part [rows][2], gmax [rows]
        CK(scratch.alloc(sizeof(double) * 3 * (size_t)rows));
        double *part = (double *)scratch.p, *gmax = part + 2 * rows;
        // shard-local (max, sum exp(x - max)) of every row: the pass and grid of trpl_lse_partial
        unsigned grid = 0;
        if (n_local > 0) TRY(stride_grid(c->device, n_local, 256, 8, &grid));
        for (int64_t r = 0; r < rows; r++) {
            trpl_lse_init_kernel<<<1, 1, 0, st>>>(part + 2 * r);
            if (n_local > 0) {
                trpl_lse_max_kernel<<<grid, 256, 0, st>>>(d_x + r * ld, n_local, part + 2 * r);
                trpl_lse_sum_kernel<<<grid, 256, 0, st>>>(d_x + r * ld, n_local, part + 2 * r);
            }
        }
        trpl_lse_split_kernel<<<small_grid(rows), 256, 0, st>>>(part, rows, gmax);
        CK(cudaGetLastError());
        TRY(settle(c, ncclAllReduce(gmax, gmax, (size_t)rows, ncclDouble, ncclMax, c->comm, st), "ncclAllReduce(max)"));
        trpl_lse_rescale_kernel<<<small_grid(rows), 256, 0, st>>>(part, gmax, rows, d_lse);
        CK(cudaGetLastError());
        TRY(settle(c, ncclAllReduce(d_lse, d_lse, (size_t)rows, ncclDouble, ncclSum, c->comm, st), "ncclAllReduce(sum)"));
        trpl_lse_finalize_kernel<<<small_grid(rows), 256, 0, st>>>(gmax, rows, d_lse);
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_posterior_weights_dev(const double *d_lnp, int64_t rows, int64_t ld, int64_t n, const double *d_lse,
                               double *d_w, int device, void *stream)
{
    if (!d_lnp || !d_lse || !d_w || rows < 1 || n < 0 || ld < n) return TRPL_EINVAL;
    return on_device(device, [&] {
        if (n == 0) return TRPL_OK;
        unsigned grid;
        TRY(stride_grid(device, rows * n, 256, 16, &grid));
        trpl_weights_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_lnp, rows, ld, n, d_lse, d_w);
        CK(cudaGetLastError());
        return TRPL_OK;
    });
}

int trpl_allreduce_sum_nccl(trpl_comm *c, double *d_buf, int64_t n, void *stream)
{
    if (!c || !d_buf || n < 0) return TRPL_EINVAL;
    return on_device(c->device, [&] {
        if (!c->comm) return aborted();
        if (n == 0) return TRPL_OK;
        return settle(c, ncclAllReduce(d_buf, d_buf, (size_t)n, ncclDouble, ncclSum, c->comm, (cudaStream_t)stream),
                      "ncclAllReduce(sum)");
    });
}

}  // extern "C"
