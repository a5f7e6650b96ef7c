// glm.cu -- the kernels of the penalized IRLS fit of Poisson, binomial and Gamma responses, splpak_b200_fit_glm_device.
//
// One evaluation of the loop in capi.cu (fit_glm_impl), after the residual pass s(x_i) of the current coefficients:
//   spl_glm_work_kernel<FAM, START>  eta_i = s(x_i) + o_i (START: eta_i = g(mu0_i), the offset ignored as glm.fit does),
//                                    mu_i, mu'_i, V(mu_i) with the clamps of R's make.link; the working response
//                                    z_i = eta_i - o_i + (y_i - mu_i) / mu'_i and row weight sqrt(W_i) = w_i mu'_i / sqrt(V)
//                                    of the next assembly (0 and 0 where w_i <= 0, y_i not read there), mu_i on request,
//                                    and per-CTA partial sums of the deviance D, of Pearson's X^2 and of
//                                    ywy = sum (sqrt(W_i) z_i)^2 (from z and the row weight as stored, so that in the
//                                    REAL32 library it is the sum of what the next assembly reads)
//   spl_glm_dev_kernel               the partial sums added in CTA order: bit-identical from call to call
// and, once before the first assembly, spl_glm_check_kernel: an integer count of the y_i outside the family's domain
// (or not finite) where w_i > 0, and m, the points with w_i > 0.  spl_glm_halve_kernel is the step halving
// c = (c + c_prev) / 2.
//
// Every index over the points is a long long and every loop is grid-stride, so n is bounded by memory, not by 2^31.
// Everything is FP64 inside the kernels (the REAL32 library reads and writes float).
#include <string.h>

#include "common.cuh"

#define GLM_EPS 2.220446049250313e-16                  // 2^-52, R's .Machine$double.eps
#define GLM_THRESH 30.0                                // logit_linkinv / logit_mu_eta of R's family.c
#define GLM_NT 256

// The link, the mean mu(eta) with its derivative mu'(eta) (one exp for both), the variance function and the unit
// deviance of each family (R's make.link, family.c and the dev.resids of poisson(), binomial() and Gamma());
// a = prior weight.
template <int FAM> struct GlmFamily;

template <> struct GlmFamily<SPLPAK_GLM_POISSON> {
    static __device__ bool valid(double y) { return y >= 0.0 && y < INFINITY; }
    static __device__ double start(double y, double) { return y + 0.1; }
    static __device__ double link(double mu) { return log(mu); }
    static __device__ void mean(double eta, double &mu, double &mue) { mu = mue = fmax(exp(eta), GLM_EPS); }
    static __device__ double variance(double mu) { return mu; }
    static __device__ double dev(double y, double mu, double a) {
        return 2.0 * a * (y > 0.0 ? y * log(y / mu) - (y - mu) : mu);
    }
};

template <> struct GlmFamily<SPLPAK_GLM_BINOMIAL> {
    static __device__ double ylogy(double y, double mu) { return y != 0.0 ? y * log(y / mu) : 0.0; }
    static __device__ bool valid(double y) { return y >= 0.0 && y <= 1.0; }
    static __device__ double start(double y, double a) { return (a * y + 0.5) / (a + 1.0); }
    static __device__ double link(double mu) { return log(mu / (1.0 - mu)); }
    static __device__ void mean(double eta, double &mu, double &mue) {
        const double e = exp(eta), ope = 1.0 + e;
        const double t = eta < -GLM_THRESH ? GLM_EPS : (eta > GLM_THRESH ? 1.0 / GLM_EPS : e);
        mu = t / (1.0 + t);
        mue = (eta > GLM_THRESH || eta < -GLM_THRESH) ? GLM_EPS : e / (ope * ope);
    }
    static __device__ double variance(double mu) { return mu * (1.0 - mu); }
    static __device__ double dev(double y, double mu, double a) {
        return 2.0 * a * (ylogy(y, mu) + ylogy(1.0 - y, 1.0 - mu));
    }
};

template <> struct GlmFamily<SPLPAK_GLM_GAMMA> {
    static __device__ bool valid(double y) { return y > 0.0 && y < INFINITY; }
    static __device__ double start(double y, double) { return y; }
    static __device__ double link(double mu) { return log(mu); }
    static __device__ void mean(double eta, double &mu, double &mue) { mu = mue = fmax(exp(eta), GLM_EPS); }
    static __device__ double variance(double mu) { return mu * mu; }
    static __device__ double dev(double y, double mu, double a) { return -2.0 * a * (log(y / mu) - (y - mu) / mu); }
};

// bad and m over the points; NaN fails every comparison of valid(), so it counts as outside the domain
template <int FAM>
__global__ void __launch_bounds__(GLM_NT)
spl_glm_check_kernel(const real_t *__restrict__ y, const real_t *__restrict__ w, int weighted, long long n,
                     unsigned long long *__restrict__ count) {
    unsigned long long bad = 0, m = 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (!((weighted ? (double)w[i] : 1.0) > 0.0)) continue;
        ++m;
        if (!GlmFamily<FAM>::valid((double)y[i])) ++bad;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
        m += __shfl_xor_sync(0xffffffffu, m, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (bad) atomicAdd(count, bad);
        if (m) atomicAdd(count + 1, m);
    }
}

template <int FAM, bool START>
__global__ void __launch_bounds__(GLM_NT)
spl_glm_work_kernel(const real_t *__restrict__ y, const real_t *__restrict__ w, int weighted,
                    const real_t *__restrict__ o, const real_t *__restrict__ s, long long n, real_t *__restrict__ z,
                    real_t *__restrict__ rw, real_t *__restrict__ mu_out, double *__restrict__ part) {
    typedef GlmFamily<FAM> F;
    double dsum = 0.0, xsum = 0.0, ysum = 0.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double wv = weighted ? (double)w[i] : 1.0;
        const double ov = o ? (double)o[i] : 0.0;
        double zi = 0.0, rwi = 0.0, mu = 0.0, mue;
        if (!START) F::mean((double)s[i] + ov, mu, mue);
        if (wv > 0.0) {
            const double yv = (double)y[i], a = wv * wv;
            double zbase;
            if (START) {
                const double eta = F::link(F::start(yv, a));
                zbase = eta - ov;
                F::mean(eta, mu, mue);
            } else {
                zbase = (double)s[i];
            }
            // 1 / sqrt(V) once: the row weight w mu' / sqrt(V) and Pearson's a (y - mu)^2 / V
            const double rs = rsqrt(F::variance(mu)), r = yv - mu, rr = r * rs;
            zi = zbase + r / mue;
            rwi = wv * mue * rs;
            dsum += F::dev(yv, mu, a);
            xsum += a * rr * rr;
        }
        const real_t zs = (real_t)zi, rws = (real_t)rwi;
        z[i] = zs;
        rw[i] = rws;
        if (mu_out) mu_out[i] = (real_t)mu;
        const double t = (double)rws * (double)zs;
        ysum = fma(t, t, ysum);
    }
    __shared__ double s_d[GLM_NT / 32], s_x[GLM_NT / 32], s_y[GLM_NT / 32];
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) {
        dsum += __shfl_xor_sync(0xffffffffu, dsum, k);
        xsum += __shfl_xor_sync(0xffffffffu, xsum, k);
        ysum += __shfl_xor_sync(0xffffffffu, ysum, k);
    }
    if ((threadIdx.x & 31) == 0) {
        s_d[threadIdx.x >> 5] = dsum;
        s_x[threadIdx.x >> 5] = xsum;
        s_y[threadIdx.x >> 5] = ysum;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double d = 0.0, x = 0.0, yy = 0.0;
        for (int k = 0; k < GLM_NT / 32; ++k) {
            d += s_d[k];
            x += s_x[k];
            yy += s_y[k];
        }
        part[3 * blockIdx.x] = d;
        part[3 * blockIdx.x + 1] = x;
        part[3 * blockIdx.x + 2] = yy;
    }
}

// dev = {D, X^2, ywy}: the CTA partials in CTA order
__global__ void spl_glm_dev_kernel(const double *__restrict__ part, int nparts, double *__restrict__ dev) {
    if (threadIdx.x == 0) {
        double d = 0.0, x = 0.0, yy = 0.0;
        for (int k = 0; k < nparts; ++k) {
            d += part[3 * k];
            x += part[3 * k + 1];
            yy += part[3 * k + 2];
        }
        dev[0] = d;
        dev[1] = x;
        dev[2] = yy;
    }
}

__global__ void spl_glm_halve_kernel(double *__restrict__ c, const double *__restrict__ cprev, long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        c[i] = 0.5 * (c[i] + cprev[i]);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int glm_grid(long long n, int nsm) {
    const long long nb = (n + GLM_NT - 1) / GLM_NT, cap = (long long)nsm * 8;
    return (int)(nb < cap ? (nb < 1 ? 1 : nb) : cap);
}

void spl_glm_scratch_free(GlmScratch &gs);

// Scratch of one call: s, z and row weights of the n points, the two counts, [cprev | cfin | dev(3) | tot0 | partials].
int spl_glm_scratch_init(GlmScratch &gs, long long n, long long ncol, int nsm) {
    memset(&gs, 0, sizeof(gs));
    gs.n = n;
    gs.nparts = glm_grid(n, nsm);
    bool ok = cudaMalloc((void **)&gs.s, sizeof(real_t) * (size_t)n) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&gs.z, sizeof(real_t) * (size_t)n) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&gs.rw, sizeof(real_t) * (size_t)n) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&gs.count, sizeof(unsigned long long) * 2) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&gs.small, sizeof(double) * (size_t)(2 * ncol + 5 + 3 * gs.nparts)) == cudaSuccess;
    if (!ok) {
        cudaGetLastError();
        spl_glm_scratch_free(gs);
        return SPLPAK_ERR_ALLOC;
    }
    gs.cprev = gs.small;
    gs.cfin = gs.cprev + ncol;
    gs.dev = gs.cfin + ncol;
    gs.tot0 = gs.dev + 3;
    gs.part = gs.tot0 + 2;
    return SPLPAK_OK;
}

void spl_glm_scratch_free(GlmScratch &gs) {
    if (gs.s) cudaFree(gs.s);
    if (gs.z) cudaFree(gs.z);
    if (gs.rw) cudaFree(gs.rw);
    if (gs.count) cudaFree(gs.count);
    if (gs.small) cudaFree(gs.small);
    memset(&gs, 0, sizeof(gs));
}

int spl_glm_check_launch(const GlmScratch &gs, int family, const real_t *d_y, const real_t *d_w, int weighted,
                         cudaStream_t st, int nsm) {
    SPL_CUDA_TRY(cudaMemsetAsync(gs.count, 0, sizeof(unsigned long long) * 2, st));
    const int grid = glm_grid(gs.n, nsm);
    if (family == SPLPAK_GLM_POISSON)
        spl_glm_check_kernel<SPLPAK_GLM_POISSON><<<grid, GLM_NT, 0, st>>>(d_y, d_w, weighted, gs.n, gs.count);
    else if (family == SPLPAK_GLM_BINOMIAL)
        spl_glm_check_kernel<SPLPAK_GLM_BINOMIAL><<<grid, GLM_NT, 0, st>>>(d_y, d_w, weighted, gs.n, gs.count);
    else
        spl_glm_check_kernel<SPLPAK_GLM_GAMMA><<<grid, GLM_NT, 0, st>>>(d_y, d_w, weighted, gs.n, gs.count);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

template <int FAM>
static void glm_work(const GlmScratch &gs, int start, const real_t *d_y, const real_t *d_w, int weighted,
                     const real_t *d_o, real_t *d_mu, cudaStream_t st) {
    if (start)
        spl_glm_work_kernel<FAM, true><<<gs.nparts, GLM_NT, 0, st>>>(d_y, d_w, weighted, d_o, gs.s, gs.n, gs.z, gs.rw,
                                                                    d_mu, gs.part);
    else
        spl_glm_work_kernel<FAM, false><<<gs.nparts, GLM_NT, 0, st>>>(d_y, d_w, weighted, d_o, gs.s, gs.n, gs.z, gs.rw,
                                                                     d_mu, gs.part);
}

// start != 0: the working quantities of mu0 (gs.s is not read); otherwise of s = gs.s.  {D, X^2, ywy} into gs.dev.
int spl_glm_work_launch(const GlmScratch &gs, int family, int start, const real_t *d_y, const real_t *d_w, int weighted,
                        const real_t *d_o, real_t *d_mu, cudaStream_t st) {
    if (family == SPLPAK_GLM_POISSON) glm_work<SPLPAK_GLM_POISSON>(gs, start, d_y, d_w, weighted, d_o, d_mu, st);
    else if (family == SPLPAK_GLM_BINOMIAL) glm_work<SPLPAK_GLM_BINOMIAL>(gs, start, d_y, d_w, weighted, d_o, d_mu, st);
    else glm_work<SPLPAK_GLM_GAMMA>(gs, start, d_y, d_w, weighted, d_o, d_mu, st);
    spl_glm_dev_kernel<<<1, 32, 0, st>>>(gs.part, gs.nparts, gs.dev);
    g_spl_launches += 2;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

int spl_glm_halve_launch(const GlmScratch &gs, double *d_c, long long ncol, cudaStream_t st) {
    spl_glm_halve_kernel<<<spl_div_up(ncol, 256), 256, 0, st>>>(d_c, gs.cprev, ncol);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}
