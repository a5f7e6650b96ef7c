// variance.cu -- pointwise posterior variances of a smoothing fit (splpak_b200_fit_prepare_variance / _fit_variance;
// DESIGN §4.13).
//
// With Sigma = M^-1 (selinv.cu) and b_k(x) the row of basis values (or of their nderiv derivatives) at x,
//     q_k(x) = b_k(x)^T Sigma b_k(x),        Var[d^k s(x)] = sigma2 q_k(x).
// b_k(x) is non-zero only on the 4^ndim nodes of x's window and is a tensor product v_1 (x) ... (x) v_ndim, so
//     q = sum over p in {0..9}^ndim of  W_w[p] prod_d u_d[p_d],    u_d[{a, b}] = v_d[a] v_d[b]   (a <= b, spl_pair order)
// with W_w[p] the sum of Sigma(j(a), j(b)) over the 2^(#d with a_d != b_d) ordered node pairs of window w that map to p.
// Two nodes of one window are at most sum_d 3 stride_d = b (the half bandwidth) apart, so every entry lies in the band
// the selected inverse forms.  One table of 10^ndim doubles per window, windows in node order, p_1 fastest:
//   spl_variance_table_kernel  one thread per entry, a fixed-order sum of <= 2^ndim band entries (no atomics)
//   spl_variance_kernel        one query per group of G lanes: the lanes read consecutive table entries (coalesced),
//                              each keeps its own partial sums, a fixed xor-shuffle tree adds them (deterministic)
#include "basis.cuh"

#define VAR_THREADS 256

// Lanes per query.  The window's table is 10^ndim doubles; the group reads it as rows of L = 10^min(ndim, 2) entries
// (the p_1 / p_2 part), H = 10^(ndim - 2) rows.  1-D: 8 lanes cover the 10 entries (one 32-byte sector per load);
// 2-D: 16 lanes cover a 100-entry row in 7 loads of 128 bytes; 3-D / 4-D: the whole warp, 4 loads per 100-entry row,
// the per-query set-up (basis, pair products, shuffle tree) amortised over 10 or 100 rows.
template <int NDIM> struct VarCfg {
    static constexpr int G = NDIM == 1 ? 8 : NDIM == 2 ? 16 : 32;
    static constexpr int L = NDIM == 1 ? 10 : 100;
    static constexpr int H = NDIM <= 2 ? 1 : NDIM == 3 ? 10 : 100;
    static constexpr int E = L * H;                       // 10^ndim entries per window
    static constexpr int NLO = (L + G - 1) / G;           // row entries per lane
};

long long spl_variance_table_len(const GridParams &gp) {
    long long e = 1;
    for (int d = 0; d < gp.ndim; ++d) e *= 10;
    return gp.nwindows * e;
}

// ---- table build: W[w * 10^ndim + p] ----
template <int NDIM>
__global__ void __launch_bounds__(VAR_THREADS)
spl_variance_table_kernel(const GridParams gp, const double *__restrict__ AB, long long lda, double *__restrict__ W,
                          long long total) {
    constexpr int E = VarCfg<NDIM>::E;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
        long long w = t / E;
        int p = (int)(t - w * E);
        int lo[NDIM], hi[NDIM];
        long long base = 0, cs = 1, cstr[NDIM];
#pragma unroll
        for (int d = 0; d < NDIM; ++d) {
            const long long ws = w % gp.nwin[d];
            w /= gp.nwin[d];
            spl_pair(p % 10, lo[d], hi[d]);
            p /= 10;
            cstr[d] = cs;
            base += ws * cs;
            cs *= gp.nodes[d];
        }
        // ordered pairs (a, b) in mask order: bit d set swaps a_d and b_d (only where they differ)
        double sum = 0.0;
#pragma unroll
        for (int m = 0; m < (1 << NDIM); ++m) {
            bool ok = true;
            long long r = base, c = base;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) {
                const bool sw = (m >> d) & 1;
                ok = ok && !(sw && lo[d] == hi[d]);
                r += (sw ? hi[d] : lo[d]) * cstr[d];
                c += (sw ? lo[d] : hi[d]) * cstr[d];
            }
            if (ok) {
                const long long i = r > c ? r : c, j = r > c ? c : r;      // Sigma(i, j), i >= j, at AB[i + j lda]
                sum += AB[i + j * lda];
            }
        }
        W[t] = sum;
    }
}

// ---- queries ----
template <int NDIM>
__global__ void __launch_bounds__(VAR_THREADS, 3)
spl_variance_kernel(const GridParams gp, int4 nder, const real_t *__restrict__ X, int l1x, long long nq,
                    const double *__restrict__ W, real_t *__restrict__ out) {
    using C = VarCfg<NDIM>;
    constexpr int G = C::G, L = C::L, H = C::H, NLO = C::NLO, QPW = 32 / G;
    __shared__ double s_v[VAR_THREADS / G][16];            // v_d[k] of each group's query
    __shared__ double s_hi[VAR_THREADS / G][H];            // prod_{d >= 3} u_d[p_d] (1 for ndim <= 2)
    __shared__ int s_ws[VAR_THREADS / G][NDIM];           // the query's window, per dimension
    __shared__ int s_nan[VAR_THREADS / G][NDIM];          // its coordinate is NaN
    const int lane = threadIdx.x & 31, gl = lane & (G - 1), grp = threadIdx.x / G;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long qb = warp0 * QPW; qb < nq; qb += nwarps * QPW) {   // uniform per warp: every lane reaches the syncs
        const long long q = qb + (lane / G);
        const bool live = q < nq;
        // the 4 ndim window weights, one per lane: lane 4 d + k forms v_d[k] exactly as spl_window_weights does (the
        // same box, the same spl_bas1 of node ws + k, the same mask), so the values are bit-identical to bascmp's
        if (live && gl < 4 * NDIM) {
            const int d = gl >> 2, k = gl & 3;
            const double x = (double)X[q * l1x + d];
            const int nd = d == 0 ? nder.x : d == 1 ? nder.y : d == 2 ? nder.z : nder.w;
            int ws, ibmn, ibmx;
            spl_box(x, gp.xmin[d], gp.dxin[d], gp.nodes[d], ws, ibmn, ibmx);
            const int ib = ws + k;
            const double v = spl_bas1(ib, gp.nodes[d], nd, x, gp.xmin[d], gp.dx[d], gp.dxin[d]);
            s_v[grp][gl] = (ib >= ibmn && ib <= ibmx) ? v : 0.0;
            if (k == 0) {
                s_ws[grp][d] = ws;
                s_nan[grp][d] = x != x;
            }
        }
        __syncwarp();
        long long win = 0, wst = 1;
        int isn = 0;
#pragma unroll
        for (int d = 0; d < NDIM; ++d) {
            win += s_ws[grp][d] * wst;
            wst *= gp.nwin[d];
            isn |= s_nan[grp][d];
        }
        // the row weights of this lane, u_1[p_1] (1-D) or u_1[p_1] u_2[p_2], and the group's row factors
        double a[NLO];
#pragma unroll
        for (int k = 0; k < NLO; ++k) {
            const int e = gl + G * k;
            a[k] = 0.0;
            if (e < L) {
                int i, j;
                spl_pair(e % 10, i, j);
                double u = s_v[grp][i] * s_v[grp][j];
                if (NDIM >= 2) {
                    spl_pair(e / 10, i, j);
                    u = u * (s_v[grp][4 + i] * s_v[grp][4 + j]);
                }
                a[k] = u;
            }
        }
        if (NDIM >= 3) {
            for (int h = gl; h < H; h += G) {
                int i, j;
                spl_pair(h % 10, i, j);
                double u = s_v[grp][8 + i] * s_v[grp][8 + j];
                if (NDIM == 4) {
                    spl_pair(h / 10, i, j);
                    u = u * (s_v[grp][12 + i] * s_v[grp][12 + j]);
                }
                s_hi[grp][h] = u;
            }
        } else if (gl == 0) {
            s_hi[grp][0] = 1.0;
        }
        __syncwarp();
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        if (live) {
            const double *T = W + win * C::E + gl;
            // four row chains (rows h = 4 i + c go to acc[c]): independent loads in flight, short rounding chains
            for (int h0 = 0; h0 < H; h0 += 4) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int h = h0 + c;
                    if (h < H) {
                        double inner = 0.0;
#pragma unroll
                        for (int k = 0; k < NLO; ++k)
                            if (gl + G * k < L) inner = fma(__ldg(T + (long long)h * L + G * k), a[k], inner);
                        acc[c] = (H == 1) ? inner : fma(inner, s_hi[grp][h], acc[c]);
                    }
                }
            }
        }
        double s = (acc[0] + acc[1]) + (acc[2] + acc[3]);
#pragma unroll
        for (int m = G / 2; m >= 1; m >>= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
        if (live && gl == 0) out[q] = (real_t)(isn ? (double)NAN : s);
        __syncwarp();                                      // s_v / s_hi / s_ws are rewritten by the next query
    }
}

int spl_variance_table_launch(const GridParams &gp, const double *d_AB, long long lda, double *d_W, cudaStream_t st,
                              int nsm) {
    const long long total = spl_variance_table_len(gp);
    const long long want = (total + VAR_THREADS - 1) / VAR_THREADS;
    const int blocks = (int)(want < 16LL * nsm ? want : 16LL * nsm);
    switch (gp.ndim) {
    case 1: spl_variance_table_kernel<1><<<blocks, VAR_THREADS, 0, st>>>(gp, d_AB, lda, d_W, total); break;
    case 2: spl_variance_table_kernel<2><<<blocks, VAR_THREADS, 0, st>>>(gp, d_AB, lda, d_W, total); break;
    case 3: spl_variance_table_kernel<3><<<blocks, VAR_THREADS, 0, st>>>(gp, d_AB, lda, d_W, total); break;
    case 4: spl_variance_table_kernel<4><<<blocks, VAR_THREADS, 0, st>>>(gp, d_AB, lda, d_W, total); break;
    default: return SPLPAK_ERR_NDIM;
    }
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

template <int NDIM>
static int variance_launch_t(const GridParams &gp, int4 nd, const real_t *d_x, int l1x, long long nq, const double *d_W,
                             real_t *d_out, cudaStream_t st, int nsm) {
    // grid-stride over one resident wave
    static int bps = 0;
    if (bps == 0) {
        int b = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, spl_variance_kernel<NDIM>, VAR_THREADS, 0) != cudaSuccess ||
            b < 1) {
            cudaGetLastError();
            b = 1;
        }
        bps = b;
    }
    const long long qpb = (long long)(VAR_THREADS / 32) * (32 / VarCfg<NDIM>::G);   // queries per block and step
    const long long want = (nq + qpb - 1) / qpb;
    const long long cap = (long long)bps * nsm;
    const int blocks = (int)(want < cap ? want : cap);
    spl_variance_kernel<NDIM><<<blocks, VAR_THREADS, 0, st>>>(gp, nd, d_x, l1x, nq, d_W, d_out);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// nderiv: HOST array of ndim entries in 0..2 (checked by the caller), NULL = values
int spl_variance_launch(const GridParams &gp, const int *nderiv, const real_t *d_x, int l1x, long long nq,
                        const double *d_W, real_t *d_out, cudaStream_t st, int nsm) {
    if (nq <= 0) return SPLPAK_OK;
    int v[4] = {0, 0, 0, 0};
    for (int d = 0; d < gp.ndim && nderiv; ++d) v[d] = nderiv[d];
    const int4 nd = make_int4(v[0], v[1], v[2], v[3]);
    switch (gp.ndim) {
    case 1: return variance_launch_t<1>(gp, nd, d_x, l1x, nq, d_W, d_out, st, nsm);
    case 2: return variance_launch_t<2>(gp, nd, d_x, l1x, nq, d_W, d_out, st, nsm);
    case 3: return variance_launch_t<3>(gp, nd, d_x, l1x, nq, d_W, d_out, st, nsm);
    case 4: return variance_launch_t<4>(gp, nd, d_x, l1x, nq, d_W, d_out, st, nsm);
    }
    return SPLPAK_ERR_NDIM;
}
