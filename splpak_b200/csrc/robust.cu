// robust.cu -- the kernels of the iteratively reweighted (Huber / bisquare) fit, splpak_b200_fit_robust_device.
//
// One reweighting of the loop in capi.cu (fit_robust_impl), after the residual pass s(x_i) of the current coefficients:
//   1. spl_robust_key_kernel      r_i = w_i (y_i - s(x_i)) -> key_i = bit pattern of |r_i| as uint64 (monotone for
//                                 non-negative doubles); w_i <= 0 -> ROBUST_KEY_NONE, above every |r_i|
//   2. radix select of the k-th smallest key, k = ceil(m / 2), m the points with w_i > 0, ROBUST_PASSES passes of
//      spl_robust_hist_kernel    histogram of one ROBUST_DIGIT-bit digit of the keys that match the prefix chosen so far
//                                (CTA-private shared-memory counts, merged into global uint64 counts)
//      spl_robust_select_kernel  one CTA: the digit holding rank k, (prefix, k) updated in device memory; after the last
//                                pass sigma = MAD / 0.6744897501960817 with MAD = the selected key read as a double
//      A multi-GPU fit all-reduces the integer histogram between the two kernels of each pass: exact, so every rank
//      selects the same key.  The host never waits inside the selection.
//   3. spl_robust_weight_kernel  u_i from |r_i| / (c sigma), row weights w_i sqrt(u_i) (and u_i), per-CTA partial sums
//                                of u_i and an integer count of the rejected points (w_i > 0, u_i = 0);
//      spl_robust_stats_kernel   the partial sums added in CTA order: bit-identical from call to call
//   4. spl_robust_change_kernel  max |c - c_prev| and max |c| over the ncol coefficients (order-independent maxima)
//
// Every index over the points is a long long and every loop is grid-stride, so n is bounded by memory, not by 2^31.
// The CTA-private counters are 32-bit: spl_robust_hist_launch sizes the grid so that no CTA visits 2^31 keys.
#include <string.h>

#include "common.cuh"

#define ROBUST_DIGIT 13                                  // bits per selection pass: 8192 counters = 32 KB of shared memory
#define ROBUST_BINS (1 << ROBUST_DIGIT)
#define ROBUST_PASSES 5                                  // 13 + 13 + 13 + 13 + 12 = 64 bits
#define ROBUST_KEY_NONE 0xffffffffffffffffULL            // points with w <= 0: above every |r| (+inf and NaN included)
#define ROBUST_NT 1024
#define MAD_SCALE 0.6744897501960817                     // Phi^-1(3/4): MAD / MAD_SCALE estimates sigma of Gaussian noise

// select state (uint64 words): [0] prefix, [1] rank k still to find inside the prefix, [2] m, [3] sigma (double bits)
#define RS_PREFIX 0
#define RS_K 1
#define RS_M 2
#define RS_SIGMA 3

struct RobustShape {
    int shift, width;
};
// pass p reads bits [shift, shift + width) of the key; the passes go from the top bits down
static __host__ __device__ inline RobustShape robust_pass_shape(int pass) {
    const int hi = 64 - ROBUST_DIGIT * pass;
    const int shift = hi - ROBUST_DIGIT > 0 ? hi - ROBUST_DIGIT : 0;
    return RobustShape{shift, hi - shift};
}

__global__ void __launch_bounds__(256)
spl_robust_key_kernel(const real_t *__restrict__ y, const real_t *__restrict__ w, int weighted,
                      const real_t *__restrict__ s, long long n, unsigned long long *__restrict__ key) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double wv = weighted ? (double)w[i] : 1.0;
        const double r = wv * ((double)y[i] - (double)s[i]);
        key[i] = wv > 0.0 ? (unsigned long long)__double_as_longlong(fabs(r)) : ROBUST_KEY_NONE;
    }
}

// Counts of the digit of pass `pass` among the keys whose bits above it equal the prefix in state[RS_PREFIX].
__global__ void __launch_bounds__(ROBUST_NT)
spl_robust_hist_kernel(const unsigned long long *__restrict__ key, long long n, int pass,
                       const unsigned long long *__restrict__ state, unsigned long long *__restrict__ hist) {
    __shared__ unsigned s_hist[ROBUST_BINS];
    const RobustShape sh = robust_pass_shape(pass);
    const int top = sh.shift + sh.width;
    const unsigned long long hmask = top >= 64 ? 0ULL : ~0ULL << top;
    const unsigned long long prefix = state[RS_PREFIX] & hmask;
    const unsigned long long dmask = (1ULL << sh.width) - 1ULL;
    for (int e = threadIdx.x; e < ROBUST_BINS; e += blockDim.x) s_hist[e] = 0u;
    __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long k = __ldcs(key + i);
        if ((k & hmask) == prefix) atomicAdd(s_hist + ((k >> sh.shift) & dmask), 1u);
    }
    __syncthreads();
    for (int e = threadIdx.x; e < ROBUST_BINS; e += blockDim.x) {
        const unsigned c = s_hist[e];
        if (c) atomicAdd(hist + e, (unsigned long long)c);
    }
}

// One CTA of ROBUST_NT threads, 8 counters each: the digit d with  sum_{e<d} hist[e] < k <= sum_{e<=d} hist[e].
// Clears the histogram for the next pass.
__global__ void __launch_bounds__(ROBUST_NT)
spl_robust_select_kernel(unsigned long long *__restrict__ hist, int pass, unsigned long long *__restrict__ state) {
    constexpr int PER = ROBUST_BINS / ROBUST_NT;
    __shared__ unsigned long long s_warp[ROBUST_NT / 32];
    __shared__ unsigned long long s_k;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const RobustShape sh = robust_pass_shape(pass);
    const int nb = 1 << sh.width;
    unsigned long long v[PER], sum = 0;
#pragma unroll
    for (int q = 0; q < PER; ++q) {
        const int e = tid * PER + q;
        v[q] = e < nb ? hist[e] : 0ULL;
        sum += v[q];
    }
    if (pass == 0) {
        // m: every key below the sentinel's digit (the first digit of ROBUST_KEY_NONE is the last bin), k = ceil(m / 2)
        unsigned long long mine = 0;
#pragma unroll
        for (int q = 0; q < PER; ++q) mine += (tid * PER + q < nb - 1) ? v[q] : 0ULL;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
        if (lane == 0) s_warp[warp] = mine;
        __syncthreads();
        if (tid == 0) {
            unsigned long long m = 0;
            for (int k = 0; k < ROBUST_NT / 32; ++k) m += s_warp[k];
            state[RS_M] = m;
            state[RS_K] = (m + 1) / 2;
            state[RS_PREFIX] = 0ULL;
        }
        __syncthreads();
    }
    // exclusive scan of the per-thread sums (fixed order)
    unsigned long long incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    if (tid == 0) s_k = state[RS_K];
    __syncthreads();
    unsigned long long before = incl - sum;
    for (int k = 0; k < warp; ++k) before += s_warp[k];
    const unsigned long long k = s_k;
    // the thread whose range holds rank k (k >= 1; m = 0 leaves k = 0 and the prefix at 0: MAD = 0)
    if (k >= 1 && before < k && k <= before + sum) {
        unsigned long long run = before;
        for (int q = 0; q < PER; ++q) {
            if (k <= run + v[q]) {
                const unsigned long long d = (unsigned long long)(tid * PER + q);
                state[RS_PREFIX] |= d << sh.shift;
                state[RS_K] = k - run;
                break;
            }
            run += v[q];
        }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < PER; ++q) hist[tid * PER + q] = 0ULL;
    if (pass == ROBUST_PASSES - 1 && tid == 0) {
        const double mad = state[RS_M] ? __longlong_as_double((long long)state[RS_PREFIX]) : 0.0;
        state[RS_SIGMA] = (unsigned long long)__double_as_longlong(mad / MAD_SCALE);
    }
}

// u from a = |r| (the key) and cs = c sigma: Huber min(1, 1/|t|), bisquare (1 - t^2)^2 for |t| < 1, t = a / cs.
// sigma == nullptr: u = 1 for every point with w > 0 (the weights of the unweighted first fit).
__global__ void __launch_bounds__(256)
spl_robust_weight_kernel(const unsigned long long *__restrict__ key, const real_t *__restrict__ w, int weighted,
                         long long n, int psi, double c, const unsigned long long *__restrict__ state,
                         real_t *__restrict__ rw, real_t *__restrict__ u_out, double *__restrict__ part,
                         unsigned long long *__restrict__ nzero) {
    const bool unit = state == nullptr;
    const double cs = unit ? 0.0 : c * __longlong_as_double((long long)state[RS_SIGMA]);
    double su = 0.0;
    unsigned long long nz = 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long k = key[i];
        const double wv = weighted ? (double)w[i] : 1.0;
        double u = 0.0;
        if (k != ROBUST_KEY_NONE) {
            if (unit) {
                u = 1.0;
            } else {
                const double t = __longlong_as_double((long long)k) / cs;
                if (psi == SPLPAK_ROBUST_HUBER) {
                    u = fmin(1.0, 1.0 / t);
                } else if (t < 1.0) {
                    const double v = 1.0 - t * t;
                    u = v * v;
                }
            }
            if (u == 0.0) ++nz;
        }
        rw[i] = (real_t)(wv * sqrt(u));
        if (u_out) u_out[i] = (real_t)u;
        su += u;
    }
    __shared__ double s_su[8];
    __shared__ unsigned long long s_nz[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        su += __shfl_xor_sync(0xffffffffu, su, o);
        nz += __shfl_xor_sync(0xffffffffu, nz, o);
    }
    if ((threadIdx.x & 31) == 0) {
        s_su[threadIdx.x >> 5] = su;
        s_nz[threadIdx.x >> 5] = nz;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        unsigned long long z = 0;
        for (int k = 0; k < (int)(blockDim.x >> 5); ++k) {
            t += s_su[k];
            z += s_nz[k];
        }
        part[blockIdx.x] = t;
        if (z) atomicAdd(nzero, z);
    }
}

// stats[0] = sum u (the CTA partials in CTA order), stats[1] = the rejected count as a double
__global__ void spl_robust_stats_kernel(const double *__restrict__ part, int nparts,
                                        const unsigned long long *__restrict__ nzero, double *__restrict__ stats) {
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int k = 0; k < nparts; ++k) s += part[k];
        stats[0] = s;
        stats[1] = (double)*nzero;
    }
}

// out2 = {max |c - c_prev|, max |c|}
__global__ void __launch_bounds__(ROBUST_NT)
spl_robust_change_kernel(const double *__restrict__ c, const double *__restrict__ cprev, long long n,
                         double *__restrict__ out2) {
    __shared__ double s_d[ROBUST_NT / 32], s_c[ROBUST_NT / 32];
    double md = 0.0, mc = 0.0;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
        md = fmax(md, fabs(c[i] - cprev[i]));
        mc = fmax(mc, fabs(c[i]));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        md = fmax(md, __shfl_xor_sync(0xffffffffu, md, o));
        mc = fmax(mc, __shfl_xor_sync(0xffffffffu, mc, o));
    }
    if ((threadIdx.x & 31) == 0) {
        s_d[threadIdx.x >> 5] = md;
        s_c[threadIdx.x >> 5] = mc;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 0; k < ROBUST_NT / 32; ++k) {
            md = fmax(md, s_d[k]);
            mc = fmax(mc, s_c[k]);
        }
        out2[0] = md;
        out2[1] = mc;
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int robust_weight_grid(long long n, int nsm) {
    const long long nb = (n + 255) / 256, cap = (long long)nsm * 8;
    return (int)(nb < cap ? (nb < 1 ? 1 : nb) : cap);
}

void spl_robust_scratch_free(RobustScratch &rs);

// Scratch of one call: keys, spline values and row weights of the n points, the selection's histogram and state, the
// weight kernel's partial sums, [previous coefficients | {max|dc|, max|c|} | {sum u, rejected} | totals | partials].
int spl_robust_scratch_init(RobustScratch &rs, long long n, long long ncol, int nsm) {
    memset(&rs, 0, sizeof(rs));
    rs.n = n;
    rs.nparts = robust_weight_grid(n, nsm);
    bool ok = cudaMalloc((void **)&rs.key, sizeof(unsigned long long) * (size_t)n) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&rs.s, sizeof(real_t) * (size_t)n) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&rs.rw, sizeof(real_t) * (size_t)n) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&rs.hist, sizeof(unsigned long long) * (ROBUST_BINS + 8)) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&rs.small, sizeof(double) * (size_t)(rs.nparts + ncol + 8)) == cudaSuccess;
    if (!ok) {
        cudaGetLastError();
        spl_robust_scratch_free(rs);
        return SPLPAK_ERR_ALLOC;
    }
    rs.state = rs.hist + ROBUST_BINS;
    rs.nzero = rs.state + 4;
    rs.cprev = rs.small;
    rs.change = rs.cprev + ncol;
    rs.stats = rs.change + 2;
    rs.tot0 = rs.stats + 2;
    rs.part = rs.tot0 + 2;
    SPL_CUDA_TRY(cudaMemset(rs.hist, 0, sizeof(unsigned long long) * (ROBUST_BINS + 8)));
    return SPLPAK_OK;
}

void spl_robust_scratch_free(RobustScratch &rs) {
    if (rs.key) cudaFree(rs.key);
    if (rs.s) cudaFree(rs.s);
    if (rs.rw) cudaFree(rs.rw);
    if (rs.hist) cudaFree(rs.hist);
    if (rs.small) cudaFree(rs.small);
    memset(&rs, 0, sizeof(rs));
}

int spl_robust_key_launch(const RobustScratch &rs, const real_t *d_y, const real_t *d_w, int weighted, cudaStream_t st,
                          int nsm) {
    spl_robust_key_kernel<<<robust_weight_grid(rs.n, nsm), 256, 0, st>>>(d_y, d_w, weighted, rs.s, rs.n, rs.key);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

int spl_robust_passes() { return ROBUST_PASSES; }
long long spl_robust_bins() { return ROBUST_BINS; }

int spl_robust_hist_launch(const RobustScratch &rs, int pass, cudaStream_t st, int nsm) {
    const long long nb = (rs.n + ROBUST_NT - 1) / ROBUST_NT;
    long long grid = (long long)nsm * 2;
    if (grid > nb) grid = nb < 1 ? 1 : nb;
    // no CTA may count 2^31 keys into one 32-bit shared counter
    const long long need = (rs.n >> 31) + 1;
    if (grid < need) grid = need;
    spl_robust_hist_kernel<<<(unsigned)grid, ROBUST_NT, 0, st>>>(rs.key, rs.n, pass, rs.state, rs.hist);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

int spl_robust_select_launch(const RobustScratch &rs, int pass, cudaStream_t st) {
    spl_robust_select_kernel<<<1, ROBUST_NT, 0, st>>>(rs.hist, pass, rs.state);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// unit != 0: u = 1 for every point with w > 0 (keys must still mark w <= 0)
int spl_robust_weight_launch(const RobustScratch &rs, const real_t *d_w, int weighted, int psi, double c, int unit,
                             real_t *d_u, cudaStream_t st, int nsm) {
    SPL_CUDA_TRY(cudaMemsetAsync(rs.nzero, 0, sizeof(unsigned long long), st));
    spl_robust_weight_kernel<<<rs.nparts, 256, 0, st>>>(rs.key, d_w, weighted, rs.n, psi, c, unit ? nullptr : rs.state,
                                                        rs.rw, d_u, rs.part, rs.nzero);
    spl_robust_stats_kernel<<<1, 32, 0, st>>>(rs.part, rs.nparts, rs.nzero, rs.stats);
    g_spl_launches += 2;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

int spl_robust_change_launch(const RobustScratch &rs, const double *d_c, long long ncol, cudaStream_t st) {
    spl_robust_change_kernel<<<1, ROBUST_NT, 0, st>>>(d_c, rs.cprev, ncol, rs.change);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}
