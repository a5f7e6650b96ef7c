// selinv.cu -- exact band selected inverse of the Cholesky factor and the generalized cross-validation score of a
// smoothing fit (splpak_b200_fit_smoothing_score; DESIGN §4.12), and the reductions of the REML score (§4.14).
//
// After spl_solve_launch, AB holds L in band storage (below the 64 x 64 diagonal blocks) and the workspace behind it the
// block inverses Linv_K = L_KK^-1 (row-major, 4096 doubles per panel).  Sigma = M^-1 = L^-T L^-1 is formed on the band
// by the blocked Takahashi recurrence, panels from the last to the first.  Panel K (columns j0 .. j0+63, m <= b rows B
// below it):
//     X     = L_BK Linv_K                       (m x 64)                        spl_selinv_x_kernel
//     S_BK  = -Sigma_BB X                       (m x m) (m x 64), split-K       spl_selinv_sbk_kernel
//     S_KK  = Linv_K^T Linv_K - X^T S_BK        (64 x 64, lower part)            spl_selinv_reduce_kernel (X^T S_BK by
//                                                                                tile row) + spl_selinv_diag_kernel
// IN PLACE: S_BK replaces L_BK (dead once X is formed), S_KK the diagonal block.  Sigma_BB is a block of columns already
// processed, so reads and writes never overlap; the band of Sigma is closed under the recurrence (every entry it reads
// lies within the half bandwidth).  The only extra memory is X (lda x 64) and the split-K partials.  Both products run on
// the FP64 tensor cores (mma.sync.m8n8k4.f64); there are no atomics: split-K partials and tile-row products are summed
// in a fixed order, so Sigma is bit-reproducible.  The 4 x n/64 launches are captured once into a CUDA graph.
//
// GCV (fixed-order reductions, FP64):
//   spl_gcv_ywy_kernel      sum (w y)^2 of an add_points chunk (per-CTA partials, spl_gcv_ywy_finish adds them in order)
//   spl_gcv_stencil_kernel  edf = sum Sigma_ij G0_ij, c^T G0 c and c.g0 over the 7^ndim stencil of every column
//
// REML (splpak_b200_fit_reml_score; DESIGN §4.14), on the factor alone (no selected inverse):
//   spl_reml_stencil_kernel c^T M c over the same stencil walk, c.g, and sum log L_jj from the stored block inverses
#include <stdlib.h>
#include <string.h>
#include <new>

#include "basis.cuh"
#include "tiles.cuh"

#define SI_NB 64
#define SI_THREADS 256
#define SI_SPLIT_TARGET 296         // CTAs a split-K step aims for (fixed: the split, hence the sum order, must not
                                    // depend on the device)
#define GCV_BLOCKS 512              // fixed grids of the GCV reductions: the same partial sums on every device
#define YWY_BLOCKS 256

// acc += A B over one staged 64-deep k tile; A(m, k) at sA[m * am + k * ak], B(k, n) at sB[k * bk + n * bn].  The warp
// owns rows wy .. wy+15 and the column blocks 2 ni + wodd (8 columns each), as spl_l21_mma.  With one of the two strides
// 1 and the other TILE_LD every fragment load is conflict-free.
__device__ __forceinline__ void si_mma64(double (&acc)[2][4][2], const double *sA, const int am, const int ak,
                                         const double *sB, const int bk, const int bn, const int wy, const int wodd,
                                         const int gq, const int t4) {
#pragma unroll 4
    for (int k0 = 0; k0 < 64; k0 += 4) {
        double af[2], bf[4];
#pragma unroll
        for (int mi = 0; mi < 2; ++mi) af[mi] = sA[(wy + mi * 8 + gq) * am + (k0 + t4) * ak];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) bf[ni] = sB[(k0 + t4) * bk + ((2 * ni + wodd) * 8 + gq) * bn];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
            for (int mi = 0; mi < 2; ++mi) spl_dmma_8x8x4(acc[mi][ni][0], acc[mi][ni][1], af[mi], bf[ni]);
    }
}

// fragment (mi, ni, h) of the calling thread -> (row, column) of the 64 x 64 output tile
#define SI_FOR_FRAG(body)                                                                                    \
    _Pragma("unroll") for (int mi = 0; mi < 2; ++mi) _Pragma("unroll") for (int ni = 0; ni < 4; ++ni)      \
        _Pragma("unroll") for (int h = 0; h < 2; ++h) {                                                     \
        const int row = wy + mi * 8 + gq, col = (2 * ni + wodd) * 8 + 2 * t4 + h;                           \
        body                                                                                                 \
    }

// X tile I = L_BK tile I * Linv_K.  One CTA per 64-row tile of B.
__global__ void __launch_bounds__(SI_THREADS)
spl_selinv_x_kernel(const double *__restrict__ AB, long long lda, long long j0, int m, const double *__restrict__ linv,
                    double *__restrict__ X, long long ldx) {
    extern __shared__ __align__(16) double s_si[];
    double *sA = s_si, *sB = s_si + 64 * TILE_LD;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, gq = lane >> 2, t4 = lane & 3;
    const int wy = (warp >> 1) * 16, wodd = warp & 1;
    const int R = blockIdx.x * 64;
    const long long r0 = j0 + SI_NB;
    spl_tile_load16(sA, AB + (r0 + R) + j0 * lda, lda, m - R, 64, tid);          // sA[k][row]
    spl_tile_load16(sB, linv, 64, 64, 64, tid);                                  // sB[k][n] = Linv[k][n]
    spl_cp_async_wait_all();
    __syncthreads();
    double acc[2][4][2] = {};
    si_mma64(acc, sA, 1, TILE_LD, sB, TILE_LD, 1, wy, wodd, gq, t4);
    SI_FOR_FRAG(if (R + row < m) X[(R + row) + col * ldx] = acc[mi][ni][h];)
}

// partial[s][I] = sum over the tiles J = s, s + ks, ... of Sigma_BB(I, J) X(J).  Sigma_BB is read through its lower band:
// a tile above the diagonal is the transpose of the stored one, the diagonal tile is symmetrized in shared memory.
__global__ void __launch_bounds__(SI_THREADS)
spl_selinv_sbk_kernel(const double *__restrict__ AB, long long lda, long long r0, int m, const double *__restrict__ X,
                      long long ldx, double *__restrict__ part, int T) {
    extern __shared__ __align__(16) double s_si[];
    double *sA = s_si, *sB = s_si + 64 * TILE_LD;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, gq = lane >> 2, t4 = lane & 3;
    const int wy = (warp >> 1) * 16, wodd = warp & 1;
    const int I = blockIdx.x, s = blockIdx.y, ks = gridDim.y;
    const int RI = I * 64;
    double acc[2][4][2] = {};
    for (int J = s; J < T; J += ks) {
        const int RJ = J * 64;
        const int cj = min(64, m - RJ);
        int am = 1, ak = TILE_LD;
        if (I >= J) {
            spl_tile_load16(sA, AB + (r0 + RI) + (r0 + RJ) * lda, lda, m - RI, cj, tid);      // sA[k][row]
        } else {
            spl_tile_load16(sA, AB + (r0 + RJ) + (r0 + RI) * lda, lda, m - RJ, min(64, m - RI), tid);   // sA[row][k]
            am = TILE_LD;
            ak = 1;
        }
        spl_tile_load16(sB, X + RJ, ldx, m - RJ, 64, tid);                                      // sB[n][k]
        spl_cp_async_wait_all();
        __syncthreads();
        if (I == J) {
            // the stored lower triangle: (r, c), r >= c, at sA[c * TILE_LD + r]; mirror it onto r < c
            for (int e = tid; e < 64 * 64; e += SI_THREADS) {
                const int r = e & 63, c = e >> 6;
                if (r < c) sA[c * TILE_LD + r] = sA[r * TILE_LD + c];
            }
            __syncthreads();
        }
        si_mma64(acc, sA, am, ak, sB, 1, TILE_LD, wy, wodd, gq, t4);
        __syncthreads();
    }
    double *out = part + ((long long)s * T + I) * 4096;
    SI_FOR_FRAG(out[col * 64 + row] = acc[mi][ni][h];)
}

// S_BK tile I = -sum_s partial[s][I] (fixed order) -> AB; q[I] = X(I)^T S_BK(I), the tile row's share of X^T S_BK.
__global__ void __launch_bounds__(SI_THREADS)
spl_selinv_reduce_kernel(double *__restrict__ AB, long long lda, long long j0, int m, const double *__restrict__ part,
                         int ks, int T, const double *__restrict__ X, long long ldx, double *__restrict__ q) {
    extern __shared__ __align__(16) double s_si[];
    double *sA = s_si, *sB = s_si + 64 * TILE_LD;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, gq = lane >> 2, t4 = lane & 3;
    const int wy = (warp >> 1) * 16, wodd = warp & 1;
    const int I = blockIdx.x, RI = I * 64;
    const long long r0 = j0 + SI_NB;
    spl_tile_load16(sA, X + RI, ldx, m - RI, 64, tid);                           // sA[c1][row]: A(c1, row) = X(row, c1)
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (int e = tid; e < 4096; e += SI_THREADS) {
        const int row = e & 63, col = e >> 6;
        double v = 0.0;
        for (int s = 0; s < ks; ++s) v += part[((long long)s * T + I) * 4096 + e];
        v = -v;
        if (RI + row < m) AB[(r0 + RI + row) + (j0 + col) * lda] = v;
        sB[col * TILE_LD + row] = v;                                             // sB[n][k]
    }
    spl_cp_async_wait_all();
    __syncthreads();
    double acc[2][4][2] = {};
    si_mma64(acc, sA, TILE_LD, 1, sB, 1, TILE_LD, wy, wodd, gq, t4);
    double *out = q + (long long)I * 4096;
    SI_FOR_FRAG(out[col * 64 + row] = acc[mi][ni][h];)
}

// S_KK = Linv^T Linv - sum_I q[I] (fixed order), lower part -> the diagonal block of AB.  One thread per entry.
__global__ void __launch_bounds__(SI_THREADS)
spl_selinv_diag_kernel(double *__restrict__ AB, long long lda, long long j0, int nb, const double *__restrict__ linv,
                       const double *__restrict__ q, int T) {
    const int e = blockIdx.x * SI_THREADS + threadIdx.x;
    const int r = e & 63, c = e >> 6;
    if (r < c || r >= nb) return;
    double v = 0.0;
    for (int k = r; k < nb; ++k) v = fma(linv[k * 64 + r], linv[k * 64 + c], v);
    double w = 0.0;
    for (int I = 0; I < T; ++I) w += q[(long long)I * 4096 + e];
    AB[(j0 + r) + (j0 + c) * lda] = v - w;
}

// ------------------------------------------------------------------------------------------
// host driver
// ------------------------------------------------------------------------------------------
long long spl_band_lda(int bw);
int spl_half_bandwidth(const GridParams &gp);

static int selinv_split(int T) {
    int ks = (SI_SPLIT_TARGET + T - 1) / T;
    return ks < 1 ? 1 : (ks > T ? T : ks);
}

// doubles of the scratch spl_selinv_launch needs: X (lda x 64), the split-K partials and the tile-row products
long long spl_selinv_scratch(const GridParams &gp) {
    const int bw = spl_half_bandwidth(gp);
    const long long lda = spl_band_lda(bw);
    const int T = (bw + 63) / 64;
    long long maxpart = 0;
    for (int t = 1; t <= T; ++t) {
        const long long p = (long long)selinv_split(t) * t;
        if (p > maxpart) maxpart = p;
    }
    return lda * 64 + (maxpart + T + 1) * 4096;
}

static cudaError_t enqueue_selinv(long long n, int bw, long long lda, double *d_AB, const double *d_linv, double *d_X,
                                  double *d_part, double *d_q, cudaStream_t st, long long *nlaunch) {
    const long long nblk = (n + SI_NB - 1) / SI_NB;
    const size_t smem = sizeof(double) * 2 * 64 * TILE_LD;
    long long count = 0;
    for (long long kb = nblk - 1; kb >= 0; --kb) {
        const long long j0 = kb * SI_NB;
        const int nb = (int)((n - j0 < SI_NB) ? n - j0 : SI_NB);
        long long mm = n - (j0 + nb);
        if (mm > bw) mm = bw;
        const int m = (int)mm;
        const int T = (m + 63) / 64;
        const double *linv = d_linv + kb * 4096;
        if (m > 0) {
            const int ks = selinv_split(T);
            spl_selinv_x_kernel<<<T, SI_THREADS, smem, st>>>(d_AB, lda, j0, m, linv, d_X, lda);
            spl_selinv_sbk_kernel<<<dim3(T, ks), SI_THREADS, smem, st>>>(d_AB, lda, j0 + SI_NB, m, d_X, lda, d_part, T);
            spl_selinv_reduce_kernel<<<T, SI_THREADS, smem, st>>>(d_AB, lda, j0, m, d_part, ks, T, d_X, lda, d_q);
            count += 3;
        }
        spl_selinv_diag_kernel<<<4096 / SI_THREADS, SI_THREADS, 0, st>>>(d_AB, lda, j0, nb, linv, d_q, T);
        ++count;
    }
    *nlaunch = count;
    return cudaGetLastError();
}

struct SelinvGraph {
    cudaGraphExec_t exec = nullptr;
    const double *key_AB = nullptr, *key_scr = nullptr;
    long long n = 0, nlaunch = 0;
    int bw = 0;
};

void spl_selinv_cache_free(void *cache) {
    SelinvGraph *sg = static_cast<SelinvGraph *>(cache);
    if (!sg) return;
    if (sg->exec) cudaGraphExecDestroy(sg->exec);
    delete sg;
}

// Sigma on the band of d_AB, in place, from the factor spl_solve_launch left in d_AB / d_work.  d_scr: the
// spl_selinv_scratch doubles.  The launches are captured once per (buffers, shape) into a graph kept in *cache.
int spl_selinv_launch(const GridParams &gp, double *d_AB, const double *d_work, double *d_scr, cudaStream_t st,
                      void **cache) {
    const long long n = gp.ncol;
    const int bw = spl_half_bandwidth(gp);
    const long long lda = spl_band_lda(bw);
    const int T = (bw + 63) / 64;
    long long maxpart = 0;
    for (int t = 1; t <= T; ++t) {
        const long long p = (long long)selinv_split(t) * t;
        if (p > maxpart) maxpart = p;
    }
    double *d_X = d_scr, *d_part = d_scr + lda * 64, *d_q = d_part + maxpart * 4096;
    const size_t smem = sizeof(double) * 2 * 64 * TILE_LD;
    SPL_CUDA_TRY(cudaFuncSetAttribute(spl_selinv_x_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SPL_CUDA_TRY(cudaFuncSetAttribute(spl_selinv_sbk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SPL_CUDA_TRY(cudaFuncSetAttribute(spl_selinv_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SelinvGraph *sg = static_cast<SelinvGraph *>(*cache);
    if (!sg || sg->key_AB != d_AB || sg->key_scr != d_scr || sg->n != n || sg->bw != bw) {
        spl_selinv_cache_free(sg);
        *cache = nullptr;
        sg = new (std::nothrow) SelinvGraph();
        if (!sg) return SPLPAK_ERR_ALLOC;
        cudaGraph_t gr = nullptr;
        cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
        if (e == cudaSuccess) {
            const cudaError_t eq = enqueue_selinv(n, bw, lda, d_AB, d_work, d_X, d_part, d_q, st, &sg->nlaunch);
            e = cudaStreamEndCapture(st, &gr);
            if (eq != cudaSuccess) e = eq;
        }
        if (e == cudaSuccess) e = cudaGraphInstantiate(&sg->exec, gr, 0);
        if (gr) cudaGraphDestroy(gr);
        if (e != cudaSuccess) {
            fprintf(stderr, "splpak_b200: CUDA graph capture of the selected inverse failed (%s)\n", cudaGetErrorString(e));
            spl_selinv_cache_free(sg);
            return SPLPAK_ERR_CUDA;
        }
        sg->key_AB = d_AB;
        sg->key_scr = d_scr;
        sg->n = n;
        sg->bw = bw;
        *cache = sg;
    }
    SPL_CUDA_TRY(cudaGraphLaunch(sg->exec, st));
    g_spl_launches += sg->nlaunch;
    return SPLPAK_OK;
}

// ------------------------------------------------------------------------------------------
// GCV reductions
// ------------------------------------------------------------------------------------------
// block sum of NV values per thread in a fixed order (xor shuffles, then the warps in order); thread 0 returns it
template <int NV>
__device__ __forceinline__ void gcv_block_sum(double (&v)[NV]) {
    __shared__ double s_w[NV][32];
#pragma unroll
    for (int k = 0; k < NV; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    if ((threadIdx.x & 31) == 0)
#pragma unroll
        for (int k = 0; k < NV; ++k) s_w[k][threadIdx.x >> 5] = v[k];
    __syncthreads();
    if (threadIdx.x == 0)
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            double t = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_w[k][w];
            v[k] = t;
        }
}

__global__ void __launch_bounds__(256)
spl_gcv_ywy_kernel(const real_t *__restrict__ y, const real_t *__restrict__ w, int weighted, long long n,
                   double *__restrict__ part) {
    double v[1] = {0.0};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double wy = (weighted ? (double)w[i] : 1.0) * (double)y[i];
        v[0] = fma(wy, wy, v[0]);
    }
    gcv_block_sum<1>(v);
    if (threadIdx.x == 0) part[blockIdx.x] = v[0];
}

__global__ void spl_gcv_ywy_finish(const double *__restrict__ part, double *__restrict__ ywy) {
    double t = 0.0;
    for (int b = 0; b < YWY_BLOCKS; ++b) t += part[b];
    *ywy += t;
}

// sum (w y)^2 of a chunk added to *d_ywy; d_part: YWY_BLOCKS doubles of scratch
int spl_gcv_ywy_launch(const real_t *d_y, const real_t *d_w, int weighted, long long n, double *d_part, double *d_ywy,
                       cudaStream_t st) {
    spl_gcv_ywy_kernel<<<YWY_BLOCKS, 256, 0, st>>>(d_y, d_w, weighted, n, d_part);
    spl_gcv_ywy_finish<<<1, 1, 0, st>>>(d_part, d_ywy);
    g_spl_launches += 2;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// The stencil pair (i, j) of column j (node digits jd) at the signed offset tuple cc (base 7, one digit per dimension: the offset + 3),
// the walk of spl_expand_band_kernel: false when node i lies outside the grid; otherwise *i and *slot, the position of
// the pair's entry in orthant-stencil storage (node * nsten + sten).
__device__ __forceinline__ bool gcv_stencil_pair(const GridParams &gp, const int (&jd)[SPL_MAXDIM], const long long j,
                                                 int cc, long long *i, long long *slot) {
    int sten = 0, sstride = 1;
    long long off = 0, node = 0, nstride = 1;
    bool inside = true;
    for (int d = 0; d < gp.ndim; ++d) {
        const int dd = cc % 7 - 3;
        cc /= 7;
        const int id = jd[d] + dd;
        if (id < 0 || id >= gp.nodes[d]) inside = false;
        off += (long long)dd * nstride;
        node += (long long)(dd < 0 ? id : jd[d]) * nstride;
        sten += (dd < 0 ? -dd : dd) * sstride;
        nstride *= gp.nodes[d];
        sstride *= 4;
    }
    *i = j + off;
    *slot = node * gp.nsten + sten;
    return inside;
}

// One CTA per column j (grid-stride), the threads over the 7^ndim signed offsets (the walk of spl_expand_band_kernel):
// for every stencil neighbour i of j,  edf += Sigma_ij G0_ij,  cGc += c_i G0_ij c_j;  and c.g0 += c_j g0_j.
__global__ void __launch_bounds__(256)
spl_gcv_stencil_kernel(const __grid_constant__ GridParams gp, const double *__restrict__ S, const double *__restrict__ AB,
                       long long lda, const double *__restrict__ c, const double *__restrict__ g0,
                       double *__restrict__ part) {
    int ncombo = 1;
    for (int d = 0; d < gp.ndim; ++d) ncombo *= 7;
    double v[3] = {0.0, 0.0, 0.0};
    for (long long j = blockIdx.x; j < gp.ncol; j += gridDim.x) {
        int jd[SPL_MAXDIM];
        {
            long long kj = j;
            for (int d = 0; d < gp.ndim; ++d) {
                jd[d] = (int)(kj % gp.nodes[d]);
                kj /= gp.nodes[d];
            }
        }
        const double cj = c[j];
        if (threadIdx.x == 0) v[2] = fma(cj, g0[j], v[2]);
        for (int cc0 = threadIdx.x; cc0 < ncombo; cc0 += blockDim.x) {
            long long i, slot;
            if (!gcv_stencil_pair(gp, jd, j, cc0, &i, &slot)) continue;
            const double gij = S[slot];
            const double sij = i >= j ? AB[i + j * lda] : AB[j + i * lda];
            v[0] = fma(sij, gij, v[0]);
            v[1] = fma(c[i] * gij, cj, v[1]);
        }
    }
    gcv_block_sum<3>(v);
    if (threadIdx.x == 0) {
        part[blockIdx.x] = v[0];
        part[GCV_BLOCKS + blockIdx.x] = v[1];
        part[2 * GCV_BLOCKS + blockIdx.x] = v[2];
    }
}

__global__ void spl_gcv_stencil_finish(const double *__restrict__ part, double *__restrict__ out3) {
    if (threadIdx.x >= 3) return;
    double t = 0.0;
    for (int b = 0; b < GCV_BLOCKS; ++b) t += part[threadIdx.x * GCV_BLOCKS + b];
    out3[threadIdx.x] = t;
}

// out3 = {edf, c^T G0 c, c.g0}; Sigma on the band of d_AB (spl_selinv_launch), G0 in stencil storage; d_part:
// 3 * GCV_BLOCKS doubles of scratch
long long spl_gcv_part_len() { return 3LL * GCV_BLOCKS; }
int spl_gcv_stencil_launch(const GridParams &gp, const double *d_S, const double *d_AB, const double *d_c,
                           const double *d_g0, double *d_part, double *d_out3, cudaStream_t st) {
    const long long lda = spl_band_lda(spl_half_bandwidth(gp));
    spl_gcv_stencil_kernel<<<GCV_BLOCKS, 256, 0, st>>>(gp, d_S, d_AB, lda, d_c, d_g0, d_part);
    spl_gcv_stencil_finish<<<1, 32, 0, st>>>(d_part, d_out3);
    g_spl_launches += 2;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// ------------------------------------------------------------------------------------------
// REML reductions (splpak_b200_fit_reml_score; DESIGN §4.14)
// ------------------------------------------------------------------------------------------
// One CTA per column j (grid-stride), the threads over the 7^ndim signed offsets as spl_gcv_stencil_kernel:
// for every stencil neighbour i of j,  cMc += c_i M_ij c_j  (M in stencil storage: the score's copy S1 + lambda R, which
// the band expansion and the solve only read);  and  c.g += c_j g_j,  logL -= log Linv_jj = log L_jj, the diagonal of
// the stored block inverses read as spl_pivot_range_kernel reads it (both solver paths store them).
__global__ void __launch_bounds__(256)
spl_reml_stencil_kernel(const __grid_constant__ GridParams gp, const double *__restrict__ M, const double *__restrict__ c,
                        const double *__restrict__ g, const double *__restrict__ linv, double *__restrict__ part) {
    int ncombo = 1;
    for (int d = 0; d < gp.ndim; ++d) ncombo *= 7;
    double v[3] = {0.0, 0.0, 0.0};
    for (long long j = blockIdx.x; j < gp.ncol; j += gridDim.x) {
        int jd[SPL_MAXDIM];
        {
            long long kj = j;
            for (int d = 0; d < gp.ndim; ++d) {
                jd[d] = (int)(kj % gp.nodes[d]);
                kj /= gp.nodes[d];
            }
        }
        const double cj = c[j];
        if (threadIdx.x == 0) {
            v[1] = fma(cj, g[j], v[1]);
            v[2] -= log(linv[(j / SI_NB) * 4096 + (j % SI_NB) * 65]);
        }
        for (int cc0 = threadIdx.x; cc0 < ncombo; cc0 += blockDim.x) {
            long long i, slot;
            if (!gcv_stencil_pair(gp, jd, j, cc0, &i, &slot)) continue;
            v[0] = fma(c[i] * M[slot], cj, v[0]);
        }
    }
    gcv_block_sum<3>(v);
    if (threadIdx.x == 0) {
        part[blockIdx.x] = v[0];
        part[GCV_BLOCKS + blockIdx.x] = v[1];
        part[2 * GCV_BLOCKS + blockIdx.x] = v[2];
    }
}

// out3 = {c^T M c, c.g, sum_j log L_jj}; M in stencil storage, d_linv the block inverses the solve left behind; d_part:
// spl_gcv_part_len() doubles of scratch.  The partials are added in order by spl_gcv_stencil_finish.
int spl_reml_stencil_launch(const GridParams &gp, const double *d_M, const double *d_c, const double *d_g,
                            const double *d_linv, double *d_part, double *d_out3, cudaStream_t st) {
    spl_reml_stencil_kernel<<<GCV_BLOCKS, 256, 0, st>>>(gp, d_M, d_c, d_g, d_linv, d_part);
    spl_gcv_stencil_finish<<<1, 32, 0, st>>>(d_part, d_out3);
    g_spl_launches += 2;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}
