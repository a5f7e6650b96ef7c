// penalty.cu -- roughness penalty of the smoothing fit (splpak_b200_fit_set_smoothing; DESIGN §4.11).
//
// The streaming Cholesky fit with lambda > 0 solves (G + lambda R) c = g, where
//     c^T R c = integral over [xmin, xmax] of  sum_d (d2 s / dx_d^2)^2            (curvature)
//                                           [+ 2 sum_{i<j} (d2 s / dx_i dx_j)^2]  (thin plate)
// Every term is a product of 1-D integrals, R = sum_terms kron_d M_d^(k_d), with
//     M_d^(k)[i][j] = integral_{xmin_d}^{xmax_d} phi_i^(k) phi_j^(k) dx,    k_d in {0, 1, 2},
// phi_i the fit's own 1-D basis (spl_bas1, edge functions included).  M_d^(k) is symmetric and couples nodes at most 3
// apart, so R has exactly the structure of the orthant-stencil storage of G (common.cuh) and is added to S in place.
//
// Three kernels, no atomics: every output entry is one thread's sum in a fixed order, so the result is the same on every
// run and on every rank.
//   spl_penalty_gram_kernel      tables m_d^(k)[i][delta] = M_d^(k)[i][i + delta], delta = 0..3 (4-point Gauss-Legendre
//                                per cell, exact for the degree-6 products), layout below
//   spl_penalty_add_kernel       S[node, sten] += lambda R[node][node + delta]
//   spl_penalty_residual_kernel  g[i] -= lambda sum_j R[i][j] c[j] over the 7^ndim stencil neighbours (refinement)
// Table layout: dimension d starts at 12 * sum_{d' < d} nodes_d'; entry (k, i, delta) at + (k * nodes_d + i) * 4 + delta.
#include "basis.cuh"

// 4-point Gauss-Legendre rule on [-1, 1]
__constant__ double c_gl_t[4] = {-0.86113631159405257522, -0.33998104358485626480, 0.33998104358485626480,
                                 0.86113631159405257522};
__constant__ double c_gl_w[4] = {0.34785484513745385737, 0.65214515486254614263, 0.65214515486254614263,
                                 0.34785484513745385737};

// doubles the tables of a grid take (the caller allocates them)
long long spl_penalty_table_len(const GridParams &gp) {
    long long n = 0;
    for (int d = 0; d < gp.ndim; ++d) n += 12LL * gp.nodes[d];
    return n;
}

// One thread per table entry (d, k, i, delta): the <= 4 cells where both functions live, 4 Gauss points each, in order.
// A function counts at a point only inside the reference's index box there (spl_box), as for the data rows.
__global__ void __launch_bounds__(128)
spl_penalty_gram_kernel(const __grid_constant__ GridParams gp, double *__restrict__ tab, long long ntab) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ntab) return;
    int d = 0;
    long long r = e;
    while (d < gp.ndim - 1 && r >= 12LL * gp.nodes[d]) r -= 12LL * gp.nodes[d++];
    const int nod = gp.nodes[d];
    const int delta = (int)(r & 3);
    const int i = (int)((r >> 2) % nod);
    const int k = (int)((r >> 2) / nod);
    const int j = i + delta;
    double sum = 0.0;
    if (j < nod) {
        const double xmin = gp.xmin[d], dx = gp.dx[d], dxin = gp.dxin[d];
        const int c0 = max(j - 2, 0), c1 = min(i + 1, nod - 2);
        for (int c = c0; c <= c1; ++c) {
            double cs = 0.0;
            for (int q = 0; q < 4; ++q) {
                const double x = xmin + ((double)c + 0.5 + 0.5 * c_gl_t[q]) * dx;
                int ws, ibmn, ibmx;
                spl_box(x, xmin, dxin, nod, ws, ibmn, ibmx);
                if (i < ibmn || j > ibmx) continue;
                const double pi = spl_bas1(i, nod, k, x, xmin, dx, dxin);
                const double pj = spl_bas1(j, nod, k, x, xmin, dx, dxin);
                cs = fma(c_gl_w[q] * pi, pj, cs);
            }
            sum += cs;
        }
        sum *= 0.5 * dx;
    }
    tab[e] = sum;
}

// The 1-D factors of R[row][col] in dimension d for k = 0, 1, 2: lo = min(row_d, col_d), delta = |row_d - col_d|.
template <int NDIM>
__device__ __forceinline__ void spl_penalty_factors(const double *tab, const GridParams &gp, const int lo[NDIM],
                                                    const int delta[NDIM], double a[NDIM][3]) {
    int off = 0;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) {
#pragma unroll
        for (int k = 0; k < 3; ++k) a[d][k] = tab[off + (k * gp.nodes[d] + lo[d]) * 4 + delta[d]];
        off += 12 * gp.nodes[d];
    }
}

// sum over the terms of the penalty of the products of their 1-D factors, in a fixed order
template <int NDIM>
__device__ __forceinline__ double spl_penalty_entry(const double a[NDIM][3], int thin_plate) {
    double v = 0.0;
#pragma unroll
    for (int t = 0; t < NDIM; ++t) {             // curvature terms: (d2 s / dx_t^2)^2
        double p = 1.0;
#pragma unroll
        for (int d = 0; d < NDIM; ++d) p *= a[d][d == t ? 2 : 0];
        v += p;
    }
    if (thin_plate) {
#pragma unroll
        for (int t0 = 0; t0 < NDIM; ++t0)
#pragma unroll
            for (int t1 = t0 + 1; t1 < NDIM; ++t1) {   // mixed terms: 2 (d2 s / dx_t0 dx_t1)^2
                double p = 2.0;
#pragma unroll
                for (int d = 0; d < NDIM; ++d) p *= a[d][(d == t0 || d == t1) ? 1 : 0];
                v += p;
            }
    }
    return v;
}

// One thread per stencil entry (node, sten) of S; the tables in shared memory (SMEM) or read through L1.
template <int NDIM, bool SMEM>
__global__ void __launch_bounds__(256)
spl_penalty_add_kernel(const __grid_constant__ GridParams gp, const double *__restrict__ tab_g, int ntab, double lambda,
                       int thin_plate, double *__restrict__ S) {
    extern __shared__ double tab_s[];
    const double *tab = tab_g;
    if (SMEM) {
        for (int e = threadIdx.x; e < ntab; e += blockDim.x) tab_s[e] = tab_g[e];
        __syncthreads();
        tab = tab_s;
    }
    constexpr int NSTEN = spl_ipow(4, NDIM);
    const long long total = gp.ncol * NSTEN;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        long long node = e / NSTEN;
        int sten = (int)(e % NSTEN);
        int lo[NDIM], delta[NDIM];
        bool inside = true;
#pragma unroll
        for (int d = 0; d < NDIM; ++d) {
            lo[d] = (int)(node % gp.nodes[d]);
            node /= gp.nodes[d];
            delta[d] = sten & 3;
            sten >>= 2;
            inside = inside && lo[d] + delta[d] < gp.nodes[d];
        }
        if (!inside) continue;
        double a[NDIM][3];
        spl_penalty_factors<NDIM>(tab, gp, lo, delta, a);
        S[e] += lambda * spl_penalty_entry<NDIM>(a, thin_plate);
    }
}

// One thread per node i: g[i] -= lambda * sum_j R[i][j] c[j], the 7^ndim neighbours j in a fixed order.
template <int NDIM, bool SMEM>
__global__ void __launch_bounds__(256)
spl_penalty_residual_kernel(const __grid_constant__ GridParams gp, const double *__restrict__ tab_g, int ntab,
                            double lambda, int thin_plate, const double *__restrict__ coef, double *__restrict__ g) {
    extern __shared__ double tab_s[];
    const double *tab = tab_g;
    if (SMEM) {
        for (int e = threadIdx.x; e < ntab; e += blockDim.x) tab_s[e] = tab_g[e];
        __syncthreads();
        tab = tab_s;
    }
    constexpr int NOFF = spl_ipow(7, NDIM);
    for (long long node = (long long)blockIdx.x * blockDim.x + threadIdx.x; node < gp.ncol;
         node += (long long)gridDim.x * blockDim.x) {
        int in[NDIM];
        {
            long long k = node;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) {
                in[d] = (int)(k % gp.nodes[d]);
                k /= gp.nodes[d];
            }
        }
        double acc = 0.0;
        for (int o = 0; o < NOFF; ++o) {
            int oo = o;
            int lo[NDIM], delta[NDIM];
            long long col = 0, stride = 1;
            bool inside = true;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) {
                const int j = in[d] + oo % 7 - 3;
                oo /= 7;
                inside = inside && j >= 0 && j < gp.nodes[d];
                lo[d] = min(in[d], j);
                delta[d] = abs(j - in[d]);
                col += (long long)j * stride;
                stride *= gp.nodes[d];
            }
            if (!inside) continue;
            double a[NDIM][3];
            spl_penalty_factors<NDIM>(tab, gp, lo, delta, a);
            acc = fma(spl_penalty_entry<NDIM>(a, thin_plate), coef[col], acc);
        }
        g[node] -= lambda * acc;
    }
}

// tables up to 48 KB (no opt-in needed) are staged in shared memory; larger ones (more than 512 nodes summed over the
// dimensions) are read through L1
static bool penalty_smem(long long ntab) { return ntab * (long long)sizeof(double) <= 48 * 1024; }

template <int NDIM>
static void penalty_add_once(const GridParams &gp, const double *d_tab, int ntab, double lambda, int thin_plate,
                             double *d_S, cudaStream_t st, int nsm) {
    const long long total = gp.ncol * spl_ipow(4, NDIM);
    long long blocks = (total + 255) / 256;
    if (blocks > (long long)nsm * 8) blocks = (long long)nsm * 8;
    if (penalty_smem(ntab))
        spl_penalty_add_kernel<NDIM, true><<<(unsigned)blocks, 256, sizeof(double) * ntab, st>>>(gp, d_tab, ntab, lambda,
                                                                                                thin_plate, d_S);
    else
        spl_penalty_add_kernel<NDIM, false><<<(unsigned)blocks, 256, 0, st>>>(gp, d_tab, ntab, lambda, thin_plate, d_S);
    ++g_spl_launches;
}

template <int NDIM>
static void penalty_residual_once(const GridParams &gp, const double *d_tab, int ntab, double lambda, int thin_plate,
                                  const double *d_coef, double *d_g, cudaStream_t st, int nsm) {
    long long blocks = (gp.ncol + 255) / 256;
    if (blocks > (long long)nsm * 8) blocks = (long long)nsm * 8;
    if (penalty_smem(ntab))
        spl_penalty_residual_kernel<NDIM, true><<<(unsigned)blocks, 256, sizeof(double) * ntab, st>>>(
            gp, d_tab, ntab, lambda, thin_plate, d_coef, d_g);
    else
        spl_penalty_residual_kernel<NDIM, false><<<(unsigned)blocks, 256, 0, st>>>(gp, d_tab, ntab, lambda, thin_plate,
                                                                                 d_coef, d_g);
    ++g_spl_launches;
}

// tables, then S += lambda R.  penalty: SPLPAK_PENALTY_CURVATURE or SPLPAK_PENALTY_THIN_PLATE.
int spl_penalty_add_launch(const GridParams &gp, double lambda, int penalty, double *d_tab, double *d_S,
                           cudaStream_t st, int nsm) {
    const long long ntab = spl_penalty_table_len(gp);
    spl_penalty_gram_kernel<<<spl_div_up(ntab, 128), 128, 0, st>>>(gp, d_tab, ntab);
    ++g_spl_launches;
    const int tp = penalty == SPLPAK_PENALTY_THIN_PLATE;
    switch (gp.ndim) {
    case 1: penalty_add_once<1>(gp, d_tab, (int)ntab, lambda, tp, d_S, st, nsm); break;
    case 2: penalty_add_once<2>(gp, d_tab, (int)ntab, lambda, tp, d_S, st, nsm); break;
    case 3: penalty_add_once<3>(gp, d_tab, (int)ntab, lambda, tp, d_S, st, nsm); break;
    case 4: penalty_add_once<4>(gp, d_tab, (int)ntab, lambda, tp, d_S, st, nsm); break;
    default: return SPLPAK_ERR_NDIM;
    }
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// g -= lambda R c with the tables spl_penalty_add_launch left in d_tab
int spl_penalty_residual_launch(const GridParams &gp, double lambda, int penalty, const double *d_tab,
                                const double *d_coef, double *d_g, cudaStream_t st, int nsm) {
    const int ntab = (int)spl_penalty_table_len(gp);
    const int tp = penalty == SPLPAK_PENALTY_THIN_PLATE;
    switch (gp.ndim) {
    case 1: penalty_residual_once<1>(gp, d_tab, ntab, lambda, tp, d_coef, d_g, st, nsm); break;
    case 2: penalty_residual_once<2>(gp, d_tab, ntab, lambda, tp, d_coef, d_g, st, nsm); break;
    case 3: penalty_residual_once<3>(gp, d_tab, ntab, lambda, tp, d_coef, d_g, st, nsm); break;
    case 4: penalty_residual_once<4>(gp, d_tab, ntab, lambda, tp, d_coef, d_g, st, nsm); break;
    default: return SPLPAK_ERR_NDIM;
    }
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// rho = sum_i G0_ii / sum_i R_ii, the scale of the default lambda range of splpak_b200_fit_select_smoothing: one CTA,
// every thread a fixed set of nodes, a fixed-order reduction.  out2 = {sum G0_ii, sum R_ii}.
template <int NDIM>
__global__ void __launch_bounds__(1024)
spl_penalty_diag_kernel(const __grid_constant__ GridParams gp, const double *__restrict__ tab, int thin_plate,
                        const double *__restrict__ S, double *__restrict__ out2) {
    __shared__ double s_g[1024], s_r[1024];
    double sg = 0.0, sr = 0.0;
    for (long long node = threadIdx.x; node < gp.ncol; node += blockDim.x) {
        int lo[NDIM], delta[NDIM];
        long long k = node;
#pragma unroll
        for (int d = 0; d < NDIM; ++d) {
            lo[d] = (int)(k % gp.nodes[d]);
            k /= gp.nodes[d];
            delta[d] = 0;
        }
        double a[NDIM][3];
        spl_penalty_factors<NDIM>(tab, gp, lo, delta, a);
        sr += spl_penalty_entry<NDIM>(a, thin_plate);
        sg += S[node * gp.nsten];
    }
    s_g[threadIdx.x] = sg;
    s_r[threadIdx.x] = sr;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            s_g[threadIdx.x] += s_g[threadIdx.x + o];
            s_r[threadIdx.x] += s_r[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out2[0] = s_g[0];
        out2[1] = s_r[0];
    }
}

int spl_penalty_diag_launch(const GridParams &gp, int penalty, double *d_tab, const double *d_S, double *d_out2,
                            cudaStream_t st) {
    const long long ntab = spl_penalty_table_len(gp);
    spl_penalty_gram_kernel<<<spl_div_up(ntab, 128), 128, 0, st>>>(gp, d_tab, ntab);
    ++g_spl_launches;
    const int tp = penalty == SPLPAK_PENALTY_THIN_PLATE;
    switch (gp.ndim) {
    case 1: spl_penalty_diag_kernel<1><<<1, 1024, 0, st>>>(gp, d_tab, tp, d_S, d_out2); break;
    case 2: spl_penalty_diag_kernel<2><<<1, 1024, 0, st>>>(gp, d_tab, tp, d_S, d_out2); break;
    case 3: spl_penalty_diag_kernel<3><<<1, 1024, 0, st>>>(gp, d_tab, tp, d_S, d_out2); break;
    case 4: spl_penalty_diag_kernel<4><<<1, 1024, 0, st>>>(gp, d_tab, tp, d_S, d_out2); break;
    default: return SPLPAK_ERR_NDIM;
    }
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}
