// trpl_aux_kernels.cuh -- the small kernels around the solver: curve reduction, probs.fastlog /
// probs.prob drop-ins, log-sum-exp pieces, device-side sampling, posterior products, DFMA
// micro-benchmark.  All HBM-bound or trivial.
#pragma once
#include "trpl_common.cuh"

namespace trpl {

// lnl[e][s] -= sum_c sse[e][c][s] (curves in order), status[s] = OR_c status[c][s]
__global__ void trpl_finish_kernel(const double *sse, double *lnl, const int *status_cs,
                                   int *status_s, long long S, int C, int E)
{
    const long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (s >= S) return;
    for (int e = 0; e < E; e++) {
        double p = lnl[e * S + s];
        for (int c = 0; c < C; c++) p -= sse[((long long)e * C + c) * S + s];
        lnl[e * S + s] = p;
    }
    if (status_s) {
        int st = 0;
        for (int c = 0; c < C; c++) st |= status_cs[(long long)c * S + s];
        status_s[s] = st;
    }
}

// ---- probs.fastlog / log_kernel (probs.py:64-85) ---------------------------------------------
// Clamp and log of one element.  float32 follows the reference's float32 buffer: compare in double, clamp
// to (float)min, log10f.
__device__ __forceinline__ double clamp_min(double v, double mn) { return v < mn ? mn : v; }
__device__ __forceinline__ float clamp_min(float v, double mn) { return (double)v < mn ? (float)mn : v; }
__device__ __forceinline__ double log10_of(double v) { return log10(v); }
__device__ __forceinline__ float log10_of(float v) { return log10f(v); }
// HBM-bound streaming kernel: 4 independent loads in flight per thread (memory-level parallelism).  All four
// are clamped before the first log: clamping each just before its log costs the float64 kernel 3 registers.
template <class T>
__global__ void trpl_log10_kernel(T *x, long long n, double mn)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n; i += 4 * stride) {
        const T v0 = clamp_min(x[i], mn), v1 = clamp_min(x[i + stride], mn);
        const T v2 = clamp_min(x[i + 2 * stride], mn), v3 = clamp_min(x[i + 3 * stride], mn);
        x[i] = log10_of(v0); x[i + stride] = log10_of(v1); x[i + 2 * stride] = log10_of(v2); x[i + 3 * stride] = log10_of(v3);
    }
    for (; i < n; i += stride) x[i] = log10_of(clamp_min(x[i], mn));
}

// ---- probs.prob / kernel_lnP (probs.py:20-62): one warp per sample, coalesced row reads -------
__global__ void trpl_lnp_kernel(double *P, const double *pl, long long S, long long n, long long ld,
                                const double *values, const double *mag)
{
    const int lane = threadIdx.x & 31;
    const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long j = warp; j < S; j += nwarps) {
        const double m = mag[j];
        const double *row = pl + j * ld;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
        long long i = lane;
        for (; i + 96 < n; i += 128) {
            const double r0 = row[i], r1 = row[i + 32], r2 = row[i + 64], r3 = row[i + 96];
            const double e0 = (r0 + m) - values[i], e1 = (r1 + m) - values[i + 32];
            const double e2 = (r2 + m) - values[i + 64], e3 = (r3 + m) - values[i + 96];
            a0 = fma(e0, e0, a0); a1 = fma(e1, e1, a1); a2 = fma(e2, e2, a2); a3 = fma(e3, e3, a3);
        }
        for (; i < n; i += 32) {
            const double e = (row[i] + m) - values[i];
            a0 = fma(e, e, a0);
        }
        const double acc = warp_sum((a0 + a1) + (a2 + a3));
        if (lane == 0) P[j] += (0.0 - acc);
    }
}

// ---- shard-local log-sum-exp pieces (Visualization/utils.py:157-166) --------------------------
// Block reduction of one value per thread: xor butterfly 16 -> 1 in every warp, the warp partials through
// shared memory, then a butterfly over them in warp 0.  Thread 0 holds the block's result.
template <class Op>
__device__ __forceinline__ double block_reduce(double v, double identity, Op op)
{
    __shared__ double sh[32];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v = op(v, __shfl_xor_sync(FULL, v, o));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        v = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : identity;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) v = op(v, __shfl_xor_sync(FULL, v, o));
    }
    return v;
}
__global__ void trpl_lse_max_kernel(const double *x, long long n, double *out)
{
    double m = -INFINITY;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        const double v = x[i];
        if (v == v && v > m) m = v;
    }
    m = block_reduce(m, -INFINITY, [](double a, double b) { return fmax(a, b); });
    if (threadIdx.x == 0) {
        // atomic max on doubles via ordered-integer trick
        unsigned long long *addr = reinterpret_cast<unsigned long long *>(out);
        unsigned long long old = *addr, assumed;
        do {
            assumed = old;
            if (__longlong_as_double((long long)assumed) >= m) break;
            old = atomicCAS(addr, assumed, (unsigned long long)__double_as_longlong(m));
        } while (assumed != old);
    }
}
__global__ void trpl_lse_sum_kernel(const double *x, long long n, double *out)
{
    const double mx = out[0];
    double acc = 0.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        const double v = x[i];
        if (v == v && v > -INFINITY) acc += exp(v - mx);   // -inf entries weigh 0 (also when every entry is -inf)
    }
    acc = block_reduce(acc, 0.0, [](double a, double b) { return a + b; });
    if (threadIdx.x == 0) atomicAdd(out + 1, acc);
}
__global__ void trpl_lse_init_kernel(double *out)
{
    out[0] = -INFINITY;
    out[1] = 0.0;
}

// ---- sample generation on the device (bayeslib.random_grid / make_grid, bayeslib.py:18-76) -----
// Counter-based Philox4x32-10: sample s, column j uses counter (s_lo, s_hi, j, 0) and key (seed_lo,
// seed_hi); u = 53 random bits / 2^53.  Same bounds / log / override semantics as the reference.
__device__ __forceinline__ void philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3,
                                              unsigned k0, unsigned k1, unsigned (&out)[4])
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

struct GridArgs {
    double lo[16], hi[16];
    int do_log[16];
    int ncol, eq_mu, eq_s, eq_auger;
};

__global__ void trpl_random_grid_kernel(double *x, long long S, long long ldx, const GridArgs ga,
                                        unsigned long long seed, unsigned long long first)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long total = S * ga.ncol;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long s = i / ga.ncol;
        const int j = (int)(i - s * ga.ncol);
        int src = j;                                   // override_equal_*: copy the draw of another column
        if (ga.eq_mu && j == 2) src = 3;
        if (ga.eq_s && j == 6) src = 5;
        if (ga.eq_auger && j == 8) src = 7;
        const unsigned long long id = first + (unsigned long long)s;
        unsigned r[4];
        philox4x32_10((unsigned)id, (unsigned)(id >> 32), (unsigned)src, 0u, (unsigned)seed,
                      (unsigned)(seed >> 32), r);
        const unsigned long long bits = (((unsigned long long)r[0] << 32) | r[1]) >> 11;
        const double u = (double)bits * (1.0 / 9007199254740992.0);
        const double lo = ga.lo[src], hi = ga.hi[src];
        double v;
        if (lo == hi) v = lo;
        else if (ga.do_log[src]) {
            const double a = log10(lo), b = log10(hi);
            v = exp10(a + (b - a) * u);
        } else v = lo + (hi - lo) * u;
        x[s * ldx + j] = v;
    }
}

// ---- posterior products (Visualization/utils.py:157-285) -------------------------------------
__global__ void trpl_weights_kernel(const double *lnp, long long n, double lse, double *w)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        const double v = lnp[i];
        w[i] = (v == v) ? exp(v - lse) : 0.0;
    }
}

// numpy.histogram bin of v over nb uniform bins on [lo, hi] (right edge inclusive), or -1
__device__ __forceinline__ int hist_bin(double v, double lo, double hi, int nb)
{
    if (!(v >= lo) || !(v <= hi)) return -1;
    int b = (int)((v - lo) / (hi - lo) * nb);
    if (b >= nb) b = nb - 1;
    // guard the edges against rounding of the scaled position (numpy does the same correction)
    const double e0 = lo + (hi - lo) * b / nb, e1 = lo + (hi - lo) * (b + 1) / nb;
    if (v < e0 && b > 0) b--;
    else if (v >= e1 && b < nb - 1) b++;
    return b;
}

__global__ void trpl_hist_kernel(const double *x, long long ldx, int colx, int coly, const double *w,
                                 long long n, double lox, double hix, int nbx, double loy, double hiy,
                                 int nby, double *hist)
{
    extern __shared__ double sh[];
    const int nb = nbx * (coly >= 0 ? nby : 1);
    for (int i = threadIdx.x; i < nb; i += blockDim.x) sh[i] = 0.0;
    __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        const int bx = hist_bin(x[i * ldx + colx], lox, hix, nbx);
        int b = bx;
        if (coly >= 0) {
            const int by = hist_bin(x[i * ldx + coly], loy, hiy, nby);
            b = (bx < 0 || by < 0) ? -1 : bx * nby + by;
        }
        if (b >= 0) atomicAdd(&sh[b], w ? w[i] : 1.0);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nb; i += blockDim.x)
        if (sh[i] != 0.0) atomicAdd(&hist[i], sh[i]);
}

// out[0] = sum w, out[1+j] = sum w x_j, out[1+ncol+j*ncol+k] = sum w x_j x_k
// One thread per sample row (coalescing comes from the 32 rows of a warp being adjacent in
// memory and ncol <= 15 columns being read in order); accumulators live in shared memory per
// warp and are reduced with shuffles -> few atomics.
__global__ void trpl_moments_kernel(const double *x, long long ldx, int ncol, const double *w,
                                    long long n, double *out)
{
    const int nacc = 1 + ncol + ncol * ncol;
    extern __shared__ double acc_sh[];          // [nacc] per block
    for (int i = threadIdx.x; i < nacc; i += blockDim.x) acc_sh[i] = 0.0;
    __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    double sw = 0.0, sx[15], sxx[15];           // per thread: sum w, sum w x_j, and ONE row of x x^T at a time
#pragma unroll
    for (int j = 0; j < 15; j++) { sx[j] = 0.0; sxx[j] = 0.0; }
    // pass structure: for each j0, accumulate sum w x_j0 x_k for all k (re-reading the row from L1/L2)
    for (int j0 = -1; j0 < ncol; j0++) {
#pragma unroll
        for (int k = 0; k < 15; k++) sxx[k] = 0.0;
        for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
            const double ww = w[i];
            const double *row = x + i * ldx;
            if (j0 < 0) {
                sw += ww;
#pragma unroll
                for (int k = 0; k < 15; k++) if (k < ncol) sx[k] = fma(ww, row[k], sx[k]);
            } else {
                const double wx = ww * row[j0];
#pragma unroll
                for (int k = 0; k < 15; k++) if (k < ncol) sxx[k] = fma(wx, row[k], sxx[k]);
            }
        }
        if (j0 < 0) {
            sw = warp_sum(sw);
            if ((threadIdx.x & 31) == 0) atomicAdd(&acc_sh[0], sw);
#pragma unroll
            for (int k = 0; k < 15; k++) if (k < ncol) {
                const double t = warp_sum(sx[k]);
                if ((threadIdx.x & 31) == 0) atomicAdd(&acc_sh[1 + k], t);
            }
        } else {
#pragma unroll
            for (int k = 0; k < 15; k++) if (k < ncol) {
                const double t = warp_sum(sxx[k]);
                if ((threadIdx.x & 31) == 0) atomicAdd(&acc_sh[1 + ncol + j0 * ncol + k], t);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nacc; i += blockDim.x)
        if (acc_sh[i] != 0.0) atomicAdd(&out[i], acc_sh[i]);
}

// Single-pass variant for the usual sample matrix (NC columns known at compile time): one thread per
// row, sum w / sum w x_j / upper triangle of sum w x_j x_k in registers, one warp reduction at the end.
template <int NC>
__global__ void __launch_bounds__(128, 2)
trpl_moments_kernel_fixed(const double *x, long long ldx, const double *w, long long n, double *out)
{
    constexpr int NT = NC * (NC + 1) / 2;
    double sw = 0.0, sx[NC], sxx[NT];
#pragma unroll
    for (int j = 0; j < NC; j++) sx[j] = 0.0;
#pragma unroll
    for (int j = 0; j < NT; j++) sxx[j] = 0.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) {
        const double ww = w[i];
        double r[NC];
#pragma unroll
        for (int j = 0; j < NC; j++) r[j] = x[i * ldx + j];
        sw += ww;
        int q = 0;
#pragma unroll
        for (int j = 0; j < NC; j++) {
            const double wx = ww * r[j];
            sx[j] += wx;
#pragma unroll
            for (int k = j; k < NC; k++) { sxx[q] = fma(wx, r[k], sxx[q]); q++; }
        }
    }
    const bool lead = (threadIdx.x & 31) == 0;
    sw = warp_sum(sw);
    if (lead && sw != 0.0) atomicAdd(&out[0], sw);
    int q = 0;
#pragma unroll
    for (int j = 0; j < NC; j++) {
        const double t = warp_sum(sx[j]);
        if (lead && t != 0.0) atomicAdd(&out[1 + j], t);
#pragma unroll
        for (int k = j; k < NC; k++) {
            const double u = warp_sum(sxx[q++]);
            if (lead && u != 0.0) {
                atomicAdd(&out[1 + NC + j * NC + k], u);
                if (k != j) atomicAdd(&out[1 + NC + k * NC + j], u);
            }
        }
    }
}

// ---- self-test of the solver's reciprocal (trpl_common.cuh: rcp64) -----------------------------
__global__ void trpl_rcp_kernel(const double *x, double *y, long long n)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += stride) y[i] = rcp64(x[i]);
}

// ---- FP64 FMA pipe microbenchmark ------------------------------------------------------------
__global__ void trpl_dfma_kernel(double *out, int iters, double seed)
{
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5,
           a6 = a0 + 6, a7 = a0 + 7;
    const double m = 0.999999, c = 1e-7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    const double r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == 12345.678) out[0] = r;   // never true; keeps the chain alive
}


}  // namespace trpl
