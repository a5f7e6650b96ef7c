// solve.cu -- derivative-constraint rows, band expansion and the blocked FP64 Cholesky solve.
//
// Replaces, for the normal equations G c = g assembled by assemble.cu:
//   * the data-sparse smoothing rows of splcw (src/splpak.F90:862-1048), added to G as rank-1
//     updates (their right-hand side is zero, :866);
//   * the triangular reduction and back-substitution of suprls (:1481-1693).  suprls reduces the
//     dense m x n row stream with Householder/Givens transforms to R with R^T R = G; here G is
//     factored directly, G = L L^T, in LOWER BAND storage (half bandwidth
//     b = 3 * sum_d prod_{d'<d} nodes(d'), SURVEY 8a), which is the dense algorithm when b = n-1.
//
// Band storage: element (i, j), 0 <= i-j < lda, lives at AB[i + j*lda] -- LAPACK band storage with
// ldab = lda + 1 viewed as a dense column-major matrix with leading dimension lda = b + NB, so every
// block kernel below is an ordinary dense column-major kernel on a sub-block (ncol*(lda+1) doubles).
//
// Right-looking blocked Cholesky, panel width NB = 64.  The same device code runs in two drivers:
//   * spl_factor_persistent_kernel / spl_backsolve_persistent_kernel: the whole loop in one cooperative
//     kernel each, phases separated by a grid-wide barrier (default where the panel chain dominates);
//   * one kernel per phase (spl_panel_kernel, spl_syrk_kernel, spl_backsolve_kernel), two streams with
//     look-ahead, captured into CUDA graphs (update-bound shapes, SPLPAK_B200_SOLVER=graph, or when a
//     cooperative launch is refused).
// The phases:
//   spl_panel_body     every CTA factors the NB x NB diagonal block AND inverts the factor (blocked
//                      inversion on the tensor cores; redundantly in every CTA: it is a latency chain, and
//                      this saves a dependency per panel), forward-solves the right-hand side of the block, then
//                      forms its 64 rows of the sub-diagonal panel L21 = A21 L11^-T as a tensor-core
//                      GEMM against the inverse and updates the right-hand side below: the forward
//                      solve L y = g rides along with the factorization.
//   spl_syrk_tile      trailing update A22 -= L21 L21^T on the lower-triangular 64 x 64 tiles of
//                      the (<= b) x (<= b) window, with FP64 tensor-core MMA
//                      (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4), operands staged k-major in
//                      shared memory.
// Back-substitution L^T c = y runs block by block from the end: every CTA
// forms c_k = L11^-T y_k from the stored block inverse, then eliminates c_k from its slice of the b
// preceding entries.
#include <stdlib.h>
#include <string.h>
#include <new>

#include <vector>

#include "basis.cuh"
#include "tiles.cuh"

#define SOLVE_NB 64

// ------------------------------------------------------------------------------------------
// constraint rows (:862-1048).  One warp per node.
// ------------------------------------------------------------------------------------------
template <int NDIM>
__global__ void __launch_bounds__(128)
spl_constraints_kernel(const __grid_constant__ GridParams gp, double xtrap,
                       const double *__restrict__ cnt, const double *__restrict__ totals_in,
                       double *__restrict__ S, double *__restrict__ totals_out) {
    const int lane = threadIdx.x & 31;
    const long long warp_global = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const double spcrit = 0.75;                                  // :696
    long long nrect = 1;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) nrect *= (gp.nodes[d] - 1);
    const double wtprrc = __ddiv_rn(totals_in[0], (double)nrect);   // :910
    constexpr int NPAIR = NDIM * (NDIM + 1) / 2;
    constexpr int NCOMBO = spl_ipow(6, NDIM);

    for (long long node = warp_global; node < gp.ncol; node += nwarps) {
        int in[NDIM];
        {
            long long k = node;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) {
                in[d] = (int)(k % gp.nodes[d]);
                k /= gp.nodes[d];
            }
        }
        double expect = wtprrc;
#pragma unroll
        for (int d = 0; d < NDIM; ++d)
            if (in[d] == 0 || in[d] == gp.nodes[d] - 1) expect = spl_mul(0.5, expect);   // :927-929
        const double have = cnt[node];
        if (!(have < spl_mul(spcrit, expect))) continue;                                // :936
        const double dcwght = spl_mul(xtrap, spl_sub(expect, have));                     // :938, :960

        int ibmn[NDIM], nbox[NDIM];
        double xn[NDIM];
#pragma unroll
        for (int d = 0; d < NDIM; ++d) {
            xn[d] = spl_add(gp.xmin[d], spl_mul((double)in[d], gp.dx[d]));               // :943
            int lo = in[d] - 1, hi = in[d] + 1;
            if (in[d] == 0) lo = 0;
            if (in[d] == gp.nodes[d] - 1) hi = gp.nodes[d] - 1;
            ibmn[d] = lo;
            nbox[d] = hi - lo + 1;
        }

        for (int idm = 0; idm < NDIM; ++idm) {
            for (int jdm = idm; jdm < NDIM; ++jdm) {
                int nder[NDIM];
#pragma unroll
                for (int d = 0; d < NDIM; ++d) nder[d] = 0;
                bool boundary = true;
                double rowwt = spl_mul(2.0, dcwght);                                     // :983
                if (jdm == idm) {
                    rowwt = dcwght;
                    nder[jdm] = 2;
                    if (in[idm] != 0 && in[idm] != gp.nodes[idm] - 1) boundary = false;
                }
                if (boundary) {
                    nder[idm] = 1;
                    nder[jdm] = 1;
                }
                // phi[d][k]: 1-D factor of box node k in dimension d (same in every lane)
                double phi[NDIM][3];
#pragma unroll
                for (int d = 0; d < NDIM; ++d)
#pragma unroll
                    for (int k = 0; k < 3; ++k)
                        phi[d][k] = (k < nbox[d]) ? spl_bas1(ibmn[d] + k, gp.nodes[d], nder[d], xn[d],
                                                             gp.xmin[d], gp.dx[d], gp.dxin[d])
                                                  : 0.0;
                const double rw2 = rowwt * rowwt;
                // all per-dimension pairs (k <= k') of box nodes: 6 per dimension
                for (int c = lane; c < NCOMBO; c += 32) {
                    int cc = c;
                    double v = rw2;
                    long long nd = 0, nstride = 1;
                    int sten = 0, sstride = 1;
                    bool ok = true;
#pragma unroll
                    for (int d = 0; d < NDIM; ++d) {
                        const int pr = cc % 6;
                        cc /= 6;
                        // pairs of {0,1,2}: (0,0)(0,1)(0,2)(1,1)(1,2)(2,2)
                        const int k0 = (pr >= 3) + (pr >= 5);
                        const int k1 = (pr < 3) ? pr : (pr < 5 ? pr - 2 : 2);
                        if (k1 >= nbox[d]) ok = false;
                        v *= phi[d][k0] * phi[d][k1];
                        nd += (long long)(ibmn[d] + k0) * nstride;
                        sten += (k1 - k0) * sstride;
                        nstride *= gp.nodes[d];
                        sstride *= 4;
                    }
                    if (ok && v != 0.0) spl_add_S(gp, S, nd * gp.nsten + sten, v);
                }
            }
        }
        if (lane == 0 && !gp.fxpass) atomicAdd(totals_out + 1, (double)NPAIR);   // constraint rows count as rows (integers: exact in any order)
    }
}

// Refinement (capi.cu): the constraint rows' share of A^T (b - A c), i.e. -C^T (C c), computed ROW BY ROW
// (v = row . c first, then g -= rowwt^2 * row * v) instead of through the formed C^T C, whose entries are
// ~dxin^4 times larger than v and would cancel catastrophically.  Same node selection and row weights as
// spl_constraints_kernel.
template <int NDIM>
__global__ void __launch_bounds__(128)
spl_constraints_residual_kernel(const __grid_constant__ GridParams gp, double xtrap,
                                const double *__restrict__ cnt, const double *__restrict__ totals_in,
                                const double *__restrict__ coef, double *__restrict__ g) {
    const int lane = threadIdx.x & 31;
    const long long warp_global = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const double spcrit = 0.75;
    long long nrect = 1;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) nrect *= (gp.nodes[d] - 1);
    const double wtprrc = __ddiv_rn(totals_in[0], (double)nrect);
    constexpr int NBOX = spl_ipow(3, NDIM);
    constexpr int PER = (NBOX + 31) / 32;

    for (long long node = warp_global; node < gp.ncol; node += nwarps) {
        int in[NDIM];
        {
            long long k = node;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) {
                in[d] = (int)(k % gp.nodes[d]);
                k /= gp.nodes[d];
            }
        }
        double expect = wtprrc;
#pragma unroll
        for (int d = 0; d < NDIM; ++d)
            if (in[d] == 0 || in[d] == gp.nodes[d] - 1) expect = spl_mul(0.5, expect);
        const double have = cnt[node];
        if (!(have < spl_mul(spcrit, expect))) continue;
        const double dcwght = spl_mul(xtrap, spl_sub(expect, have));
        int ibmn[NDIM], nbox[NDIM];
        double xn[NDIM];
#pragma unroll
        for (int d = 0; d < NDIM; ++d) {
            xn[d] = spl_add(gp.xmin[d], spl_mul((double)in[d], gp.dx[d]));
            int lo = in[d] - 1, hi = in[d] + 1;
            if (in[d] == 0) lo = 0;
            if (in[d] == gp.nodes[d] - 1) hi = gp.nodes[d] - 1;
            ibmn[d] = lo;
            nbox[d] = hi - lo + 1;
        }
        for (int idm = 0; idm < NDIM; ++idm) {
            for (int jdm = idm; jdm < NDIM; ++jdm) {
                int nder[NDIM];
#pragma unroll
                for (int d = 0; d < NDIM; ++d) nder[d] = 0;
                bool boundary = true;
                double rowwt = spl_mul(2.0, dcwght);
                if (jdm == idm) {
                    rowwt = dcwght;
                    nder[jdm] = 2;
                    if (in[idm] != 0 && in[idm] != gp.nodes[idm] - 1) boundary = false;
                }
                if (boundary) {
                    nder[idm] = 1;
                    nder[jdm] = 1;
                }
                double phi[NDIM][3];
#pragma unroll
                for (int d = 0; d < NDIM; ++d)
#pragma unroll
                    for (int k = 0; k < 3; ++k)
                        phi[d][k] = (k < nbox[d]) ? spl_bas1(ibmn[d] + k, gp.nodes[d], nder[d], xn[d],
                                                             gp.xmin[d], gp.dx[d], gp.dxin[d])
                                                  : 0.0;
                // row entries owned by this lane: b[e], column nd[e]
                double b[PER];
                long long col[PER];
                double v = 0.0;
#pragma unroll
                for (int e = 0; e < PER; ++e) {
                    const int c = lane + 32 * e;
                    b[e] = 0.0;
                    col[e] = 0;
                    if (c < NBOX) {
                        int cc = c;
                        double bv = 1.0;
                        long long nd = 0, nstride = 1;
                        bool ok = true;
#pragma unroll
                        for (int d = 0; d < NDIM; ++d) {
                            const int k = cc % 3;
                            cc /= 3;
                            if (k >= nbox[d]) ok = false;
                            bv *= phi[d][k];
                            nd += (long long)(ibmn[d] + k) * nstride;
                            nstride *= gp.nodes[d];
                        }
                        if (ok) {
                            b[e] = bv;
                            col[e] = nd;
                            v = fma(bv, coef[nd], v);
                        }
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                const double scale = -(rowwt * rowwt) * v;
#pragma unroll
                for (int e = 0; e < PER; ++e)
                    if (b[e] != 0.0) spl_add_g(gp, g, col[e], scale * b[e]);
            }
        }
    }
}

// deterministic mode (assemble.cu): scale-finding pass, exponent, adding pass, limb sums -> S / g
int spl_fx_begin(const GridParams &gp, cudaStream_t st);
int spl_fx_scale(const GridParams &gp, int *fxe, cudaStream_t st);
int spl_fx_finish(const GridParams &gp, double *d_S, double *d_g, cudaStream_t st);

template <int NDIM>
static void constraints_residual_once(const GridParams &gp, unsigned blocks, double xtrap, const double *d_cnt,
                                      const double *d_totals_in, const double *d_coef, double *d_g, cudaStream_t st) {
    spl_constraints_residual_kernel<NDIM><<<blocks, 128, 0, st>>>(gp, xtrap, d_cnt, d_totals_in, d_coef, d_g);
    ++g_spl_launches;
}
template <int NDIM>
static void constraints_once(const GridParams &gp, unsigned blocks, double xtrap, const double *d_cnt,
                             const double *d_totals_in, double *d_S, double *d_totals_out, cudaStream_t st) {
    spl_constraints_kernel<NDIM><<<blocks, 128, 0, st>>>(gp, xtrap, d_cnt, d_totals_in, d_S, d_totals_out);
    ++g_spl_launches;
}

int spl_constraints_residual_launch(const GridParams &gp, double xtrap, const double *d_cnt,
                                    const double *d_totals_in, const double *d_coef, double *d_g,
                                    cudaStream_t st, int nsm) {
    long long blocks = (gp.ncol + 3) / 4;
    if (blocks > (long long)nsm * 16) blocks = (long long)nsm * 16;
    const bool det = gp.fxS != nullptr;
    GridParams gpp = gp;
    if (det) {
        const int rf = spl_fx_begin(gp, st);
        if (rf != SPLPAK_OK) return rf;
    }
    for (int pass = det ? 1 : 0; pass >= 0; --pass) {
        gpp.fxpass = pass;
        switch (gp.ndim) {
        case 1: constraints_residual_once<1>(gpp, (unsigned)blocks, xtrap, d_cnt, d_totals_in, d_coef, d_g, st); break;
        case 2: constraints_residual_once<2>(gpp, (unsigned)blocks, xtrap, d_cnt, d_totals_in, d_coef, d_g, st); break;
        case 3: constraints_residual_once<3>(gpp, (unsigned)blocks, xtrap, d_cnt, d_totals_in, d_coef, d_g, st); break;
        case 4: constraints_residual_once<4>(gpp, (unsigned)blocks, xtrap, d_cnt, d_totals_in, d_coef, d_g, st); break;
        default: return SPLPAK_ERR_NDIM;
        }
        if (pass == 1) {
            const int rf = spl_fx_scale(gp, const_cast<int *>(gp.fxe), st);
            if (rf != SPLPAK_OK) return rf;
        }
    }
    if (det) {
        const int rf = spl_fx_finish(gp, nullptr, d_g, st);
        if (rf != SPLPAK_OK) return rf;
    }
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

int spl_constraints_launch(const GridParams &gp, double xtrap, const double *d_cnt,
                           const double *d_totals_in, double *d_S, double *d_totals_out,
                           cudaStream_t st, int nsm) {
    long long blocks = (gp.ncol + 3) / 4;
    if (blocks > (long long)nsm * 16) blocks = (long long)nsm * 16;
    const bool det = gp.fxS != nullptr;
    GridParams gpp = gp;
    if (det) {
        const int rf = spl_fx_begin(gp, st);
        if (rf != SPLPAK_OK) return rf;
    }
    for (int pass = det ? 1 : 0; pass >= 0; --pass) {
        gpp.fxpass = pass;
        switch (gp.ndim) {
        case 1: constraints_once<1>(gpp, (unsigned)blocks, xtrap, d_cnt, d_totals_in, d_S, d_totals_out, st); break;
        case 2: constraints_once<2>(gpp, (unsigned)blocks, xtrap, d_cnt, d_totals_in, d_S, d_totals_out, st); break;
        case 3: constraints_once<3>(gpp, (unsigned)blocks, xtrap, d_cnt, d_totals_in, d_S, d_totals_out, st); break;
        case 4: constraints_once<4>(gpp, (unsigned)blocks, xtrap, d_cnt, d_totals_in, d_S, d_totals_out, st); break;
        default: return SPLPAK_ERR_NDIM;
        }
        if (pass == 1) {
            const int rf = spl_fx_scale(gp, const_cast<int *>(gp.fxe), st);
            if (rf != SPLPAK_OK) return rf;
        }
    }
    if (det) {
        const int rf = spl_fx_finish(gp, d_S, nullptr, st);
        if (rf != SPLPAK_OK) return rf;
    }
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// ------------------------------------------------------------------------------------------
// S (orthant stencil) -> lower band storage
// ------------------------------------------------------------------------------------------
// One CTA per column j (grid-stride): the column's node index is decomposed once, the threads walk the 7^ndim signed
// offset tuples (d_1..d_n), d in -3..3, of the stencil -- base 7 with constant divisors -- and keep those inside the grid
// with i = j + sum d_d stride_d >= j (the lower band).  The first version ran one thread per (column, band offset)
// pair with two runtime 64-bit divisions per dimension for every one of the n (b + 1) pairs, 58 % of which hold no
// entry in 4-D: 1.39 ms at cfg4 (12^4 nodes, b = 5,655), 0.25 ms at cfg3.
__global__ void __launch_bounds__(256)
spl_expand_band_kernel(const __grid_constant__ GridParams gp, const double *__restrict__ S,
                       double *__restrict__ AB, long long lda, int bw) {
    int ncombo = 1;
    for (int d = 0; d < gp.ndim; ++d) ncombo *= 7;
    for (long long j = blockIdx.x; j < gp.ncol; j += gridDim.x) {
        int jd[SPL_MAXDIM];
        {
            long long kj = j;
            for (int d = 0; d < gp.ndim; ++d) {
                jd[d] = (int)(kj % gp.nodes[d]);
                kj /= gp.nodes[d];
            }
        }
        for (int c = threadIdx.x; c < ncombo; c += blockDim.x) {
            int cc = c, sten = 0, sstride = 1;
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
            if (inside && off >= 0 && off <= bw) AB[(j + off) + j * lda] = S[node * gp.nsten + sten];
        }
    }
}

// ------------------------------------------------------------------------------------------
// panel: diagonal-block Cholesky + inverse (registers), rhs forward solve, TRSM as a DMMA GEMM
// ------------------------------------------------------------------------------------------
#define PANEL_THREADS 256
// CTA barrier of the 256 working threads.  The pieces below run in 256-thread CTAs (where this IS __syncthreads) and in
// the data-flow kernel, whose CTAs carry a ninth warp that must not take part.
#define SPL_SYNC256() asm volatile("bar.sync 0, 256;" ::: "memory")
#define PANEL_LDT 36    // 32 + 4, same bank argument as TILE_LD
// One doubling level of the blocked triangular inversion: for every pair of SZ x SZ diagonal blocks (instance q)
//   X21 = -X22 (L21 X11),
// both products as 8 x 8 output tiles on the FP64 tensor cores (one or two tiles per warp).  The inversion is IN
// PLACE (sL == sX): X11 and X22 already replaced their L blocks, L21 is dead once T = L21 X11 is formed.  The array is
// row-major with stride TILE_LD, T (sT) with stride PANEL_LDT, so every fragment load is conflict-free and a
// "k-major" operand is just the other index order of the same array.  A scalar version of this level was bound by
// shared-memory wavefronts (2,570 clocks per 32^3 product: an LDS.64 whose lanes share addresses still costs 2).
template <int SZ>
__device__ __forceinline__ void spl_inv_level(const double *sL, double *sX, double *__restrict__ sT, int tid) {
    constexpr int TR = SZ / 8, TPI = TR * TR, NTILE = (64 / (2 * SZ)) * TPI;     // 4, 8, 16 tiles
    const int warp = tid >> 5, lane = tid & 31, gq = lane >> 2, t4 = lane & 3;
    for (int tl = warp; tl < NTILE; tl += PANEL_THREADS / 32) {                  // T = L21 X11
        const int q = tl / TPI, rem = tl % TPI, ti = rem / TR, tj = rem % TR;
        const int rb = (2 * q + 1) * SZ, cb = 2 * q * SZ;
        const double *pa = sL + (rb + ti * 8 + gq) * TILE_LD + cb + t4;
        const double *pb = sX + (cb + t4) * TILE_LD + cb + tj * 8 + gq;
        double c0 = 0.0, c1 = 0.0, d0 = 0.0, d1 = 0.0;
#pragma unroll
        for (int k0 = 0; k0 < SZ; k0 += 8) {
            spl_dmma_8x8x4(c0, c1, pa[k0], pb[k0 * TILE_LD]);
            spl_dmma_8x8x4(d0, d1, pa[k0 + 4], pb[(k0 + 4) * TILE_LD]);
        }
        *reinterpret_cast<double2 *>(sT + (q * SZ + ti * 8 + gq) * PANEL_LDT + tj * 8 + 2 * t4) =
            make_double2(c0 + d0, c1 + d1);
    }
    SPL_SYNC256();
    for (int tl = warp; tl < NTILE; tl += PANEL_THREADS / 32) {                  // X21 = -X22 T
        const int q = tl / TPI, rem = tl % TPI, ti = rem / TR, tj = rem % TR;
        const int rb = (2 * q + 1) * SZ, cb = 2 * q * SZ;
        const double *pa = sX + (rb + ti * 8 + gq) * TILE_LD + rb + t4;
        const double *pb = sT + (q * SZ + t4) * PANEL_LDT + tj * 8 + gq;
        double c0 = 0.0, c1 = 0.0, d0 = 0.0, d1 = 0.0;
#pragma unroll
        for (int k0 = 0; k0 < SZ; k0 += 8) {
            spl_dmma_8x8x4(c0, c1, pa[k0], pb[k0 * PANEL_LDT]);
            spl_dmma_8x8x4(d0, d1, pa[k0 + 4], pb[(k0 + 4) * PANEL_LDT]);
        }
        *reinterpret_cast<double2 *>(sX + (rb + ti * 8 + gq) * TILE_LD + cb + tj * 8 + 2 * t4) =
            make_double2(-(c0 + d0), -(c1 + d1));
    }
    SPL_SYNC256();
}

// ---- pieces of the diagonal-block chain, shared by spl_panel_body and the data-flow kernel's diagonal CTA ----
// Thread (ri, rc) = (tid / 4, tid % 4) owns u[kk] = A11[ri][4 kk + rc], kk = 0..15 (lower triangle, identity padding).
//
// Right-looking Cholesky in the square-root-free form, one barrier per column.  Column j of the Schur complement is
// published unscaled (u_ij); every thread forms 1/d_j itself (d_j = u_jj) and applies  u_ik -= (u_ij / d_j) u_kj  to its
// 16 entries.  The dependent chain per pivot is publish -> barrier -> reciprocal -> one multiply -> one FMA (the entry
// of column j+1), instead of a 4 x 4 block factorisation + two triangular solves per four pivots; L = U diag(d)^-1/2
// is formed afterwards (spl_linv64).  s_rd[j] = d_j on return; *s_bad is set on a non-positive (or NaN) pivot.
template <int JLO = 0, int JHI = 64>      // pivots [JLO, JHI): the caller may put work between two halves
__device__ __forceinline__ void spl_chol64(double (&u)[16], double *s_col, double *s_rd, int *s_bad, const int tid) {
    const int ri = tid >> 2, rc = tid & 3;
#pragma unroll
    for (int j = JLO; j < JHI; ++j) {
        const int kj = j >> 2, cj = j & 3;
        double *col = s_col + (j & 1) * 64;
        if (rc == cj) col[ri] = u[kj];
        SPL_SYNC256();
        const double d = col[j];
        // 1/d: hardware seed + one cubically convergent step: y0 (1 + e + e^2), e = 1 - d y0 ~ 2^-23 -> 2^-69 (three
        // dependent operations; two Newton steps are four, and FP64 latency is what this loop is made of)
        double ci;
        {
            double y0;
            asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(d));
            const double e = fma(-d, y0, 1.0);
            const double e2 = fma(e, e, e);
            // ci = col[ri] / d = t (1 + e2), t = col[ri] y0: t does not wait for e, so forming ci directly is
            // one dependent FP64 operation shorter than rinv = y0 (1 + e2) followed by col[ri] * rinv
            const double t = col[ri] * y0;
            ci = fma(t, e2, t);
        }
        if (tid == 0) {
            s_rd[j] = d;                                     // d_j for now; 1 / L_jj after spl_linv64
            if (!(d > 0.0)) *s_bad = 1;                      // non-positive (or NaN) pivot -> 107
        }
#pragma unroll
        for (int kk = kj; kk < 16; ++kk) {
            const int k = 4 * kk + rc;
            if (k > j) u[kk] = fma(-ci, col[k], u[kk]);
        }
    }
    if (JHI == 64) SPL_SYNC256();
}

// 1 / L_jj = d_j^-1/2 (seed + two Goldschmidt steps), L11 = U diag(d)^-1/2 -> sX (row-major, stride TILE_LD), then
// X = L11^-1 IN PLACE, blocked: the eight 8 x 8 diagonal blocks by forward substitution (64 threads, an 8-step chain
// each), then three doubling levels  X21 = -X22 (L21 X11)  on the tensor cores.  One thread per column running the
// whole 64-step substitution took 14.1k clocks.
__device__ __forceinline__ void spl_linv64(const double (&u)[16], double *s_rd, double *sX, double *sT, const int tid) {
    const int ri = tid >> 2, rc = tid & 3;
    if (tid < 64) {
        const double d = s_rd[tid];
        double y0;
        asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(d));
        double gq2 = d * y0;
        double hq = 0.5 * y0;
#pragma unroll
        for (int itn = 0; itn < 2; ++itn) {
            const double rr = fma(-gq2, hq, 0.5);
            gq2 = fma(gq2, rr, gq2);
            hq = fma(hq, rr, hq);
        }
        s_rd[tid] = 2.0 * hq;
    }
    SPL_SYNC256();
    double *sL = sX;
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
        const int k = 4 * kk + rc;
        sL[ri * TILE_LD + k] = (k <= ri) ? u[kk] * s_rd[k] : 0.0;
    }
    SPL_SYNC256();
    {
        const int b0 = tid & 56, cj = tid & 7;            // threads >= 64 compute nothing
        double Lb[8][8], X[8];
        if (tid < 64) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int c = 0; c < i; ++c) Lb[i][c] = sL[(b0 + i) * TILE_LD + b0 + c];
        }
        SPL_SYNC256();                                  // the block is in registers: X may overwrite it
        if (tid < 64) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                double s0 = 0.0, s1 = 0.0;
#pragma unroll
                for (int c = 0; c < i; ++c) {
                    if (c & 1) s1 = fma(Lb[i][c], X[c], s1);
                    else s0 = fma(Lb[i][c], X[c], s0);
                }
                const double rhs = (i == cj) ? 1.0 : 0.0;
                X[i] = (rhs - (s0 + s1)) * s_rd[b0 + i];
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) sX[(b0 + i) * TILE_LD + b0 + cj] = X[i];
        }
    }
    SPL_SYNC256();
    spl_inv_level<8>(sL, sX, sT, tid);
    spl_inv_level<16>(sL, sX, sT, tid);
    spl_inv_level<32>(sL, sX, sT, tid);
}

// y1[ri] = sum_k Linv[ri][k] g1[k]: four threads per row (ri, rc), 16 products each (k = rc + 4 q: conflict-free),
// combined with two shuffles; every thread of the row returns the sum.
__device__ __forceinline__ double spl_y1_64(const double *sX, const double *s_g, const int tid) {
    const int ri = tid >> 2, rc = tid & 3;
    double y1c = 0.0, y1d = 0.0;
#pragma unroll
    for (int q = 0; q < 16; q += 2) {
        y1c = fma(sX[ri * TILE_LD + rc + 4 * q], s_g[rc + 4 * q], y1c);
        y1d = fma(sX[ri * TILE_LD + rc + 4 * q + 4], s_g[rc + 4 * q + 4], y1d);
    }
    y1c += y1d;
    y1c += __shfl_xor_sync(0xffffffffu, y1c, 1);
    y1c += __shfl_xor_sync(0xffffffffu, y1c, 2);
    return y1c;
}

// L21 tile = A21 tile * Linv^T: out[r][c] = sum_k A21[r][k] Linv[c][k] for the 64 rows R0.. (relative to r0) whose A21
// tile is in sA (k-major); stored into AB, and (WITH_G) the right-hand side below the block is updated: g2 -= L21 y1
// (s_g = y1) with atomic adds into g -- the data-flow kernel's workers do that later from the tile left in sA
// (spl_g_update), so that the diagonal CTA can publish L11^-1 before it has formed y1.
// keep_l21: leave the L21 tile in sA, k-major, where the tile update expects its A operand.
// acc = A21 tile * Linv^T for the calling warp's 16 rows (wy..) and its four column blocks cb = 2 ni + wodd (8 columns
// each; interleaved over the two warp classes so that both do the same work).  Linv is lower triangular: column block
// cb needs k < 8 cb + 8 only, so the k range is cut in four segments of 16 and segment s feeds the blocks ni >= s --
// 80 of the 128 MMAs of the full product, in straight-line code (a test per block and k step made the loop
// latency-bound: 4.4k clocks for 64 MMAs).
__device__ __forceinline__ void spl_l21_mma(double (&acc)[2][4][2], const double *sA, const double *sX, const int wy,
                                            const int wodd, const int gq, const int t4) {
#pragma unroll
    for (int mi = 0; mi < 2; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
#pragma unroll
    for (int sgm = 0; sgm < 4; ++sgm) {
#pragma unroll
        for (int k0 = 16 * sgm; k0 < 16 * sgm + 16; k0 += 4) {
            double af[2], bf[4];
#pragma unroll
            for (int mi = 0; mi < 2; ++mi) af[mi] = sA[(k0 + t4) * TILE_LD + wy + mi * 8 + gq];
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
                if (ni >= sgm) bf[ni] = sX[((2 * ni + wodd) * 8 + gq) * TILE_LD + k0 + t4];    // B[k][n] = Linv[n][k]
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
                if (ni >= sgm) {
#pragma unroll
                    for (int mi = 0; mi < 2; ++mi) spl_dmma_8x8x4(acc[mi][ni][0], acc[mi][ni][1], af[mi], bf[ni]);
                }
        }
    }
}

template <bool WITH_G = true>
__device__ __forceinline__ void spl_l21_gemm(double *AB, long long lda, long long j0, int nb, int m, long long r0,
                                             int R0, double *g, double *sA, const double *sX, const double *s_g,
                                             const bool keep_l21, const int tid) {
    const int warp = tid >> 5, lane = tid & 31;
    const int gq = lane >> 2, t4 = lane & 3;
    const int wy = (warp >> 1) * 16, wodd = warp & 1;
    double acc[2][4][2];
    double gpart[2] = {0.0, 0.0};
    spl_l21_mma(acc, sA, sX, wy, wodd, gq, t4);
    // store L21 and update the right-hand side below the block: g2 -= L21 y1
#pragma unroll
    for (int mi = 0; mi < 2; ++mi) {
        const int r = R0 + wy + mi * 8 + gq;
        double part = 0.0;
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int c = (2 * ni + wodd) * 8 + 2 * t4 + h;
                const double v = acc[mi][ni][h];
                if (r < m && c < nb) AB[(r0 + r) + (j0 + c) * lda] = v;
                if (WITH_G) part = fma(v, s_g[c], part);
            }
        if (WITH_G) {
            part += __shfl_xor_sync(0xffffffffu, part, 1);
            part += __shfl_xor_sync(0xffffffffu, part, 2);
            gpart[mi] = part;
        }
    }
    if (WITH_G) {
        // the two warps that hold the column halves of a row combine their shares in a fixed order and the row gets ONE
        // addition per panel (two atomics per row made g -- and the coefficients -- depend on which warp arrived first)
        __shared__ double s_gpart[64];
#pragma unroll
        for (int mi = 0; mi < 2; ++mi)
            if (wodd && t4 == 0) s_gpart[wy + mi * 8 + gq] = gpart[mi];
        SPL_SYNC256();
#pragma unroll
        for (int mi = 0; mi < 2; ++mi) {
            const int r = R0 + wy + mi * 8 + gq;
            if (!wodd && t4 == 0 && r < m) {
                const double both = gpart[mi] + s_gpart[wy + mi * 8 + gq];
                if (both != 0.0) atomicAdd(g + r0 + r, -both);
            }
        }
    }
    if (keep_l21) {
        SPL_SYNC256();                                      // everyone is done reading sA (A21)
#pragma unroll
        for (int mi = 0; mi < 2; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    sA[((2 * ni + wodd) * 8 + 2 * t4 + h) * TILE_LD + wy + mi * 8 + gq] = acc[mi][ni][h];
    }
}

// g2 -= L21 y1 for the 64 rows R0.. from the L21 tile in sA (k-major) and y1 in s_g: four threads per row (16
// products each, conflict-free), two shuffles, one atomic add per row.
__device__ __forceinline__ void spl_g_update(double *g, long long r0, int R0, int m, const double *sA, const double *s_g,
                                             const int tid) {
    const int ri = tid >> 2, rc = tid & 3;
    double p0 = 0.0, p1 = 0.0;
#pragma unroll
    for (int q = 0; q < 16; q += 2) {
        p0 = fma(sA[(rc + 4 * q) * TILE_LD + ri], s_g[rc + 4 * q], p0);
        p1 = fma(sA[(rc + 4 * q + 4) * TILE_LD + ri], s_g[rc + 4 * q + 4], p1);
    }
    p0 += p1;
    p0 += __shfl_xor_sync(0xffffffffu, p0, 1);
    p0 += __shfl_xor_sync(0xffffffffu, p0, 2);
    if (rc == 0 && R0 + ri < m && p0 != 0.0) atomicAdd(g + r0 + R0 + ri, -p0);
}

// Every CTA factors the nb x nb diagonal block A11 = L11 L11^T (four threads per row, 16 entries each in
// registers, one barrier per pivot, pivot column broadcast through double-buffered shared memory) and
// inverts L11.  Doing this redundantly in every CTA costs no time (it is a latency chain) and saves a
// launch + dependency per panel.
// Then  y1 = L11^-1 g1,  L21 = A21 L11^-T  for this CTA's 64 rows (FP64 tensor-core MMA against the
// inverse, so no per-row substitution chain) and  g2 -= L21 y1.
// CTA 0 stores L11^-1 (for the back-substitution) and y1.
// cta / ncta: this CTA's index among the CTAs working on the panel and their number (the stand-alone kernel passes
// blockIdx.x / gridDim.x; the barrier-phased persistent kernel its first CTAs).  failed: an earlier panel failed.
__device__ __forceinline__ void spl_panel_body(double *AB, long long lda, long long j0, int nb, int m, double *g,
                                               double *ysol, double *linv_blk, int *fail, long long *dbg,
                                               double *s_pan, const int cta, const int ncta, const int failed,
                                               const bool keep_l21 = false) {
#define PANEL_STAMP(i) do { if (dbg && cta == 0 && threadIdx.x == 0) dbg[i] = clock64(); } while (0)
    PANEL_STAMP(0);
    double *sA = s_pan;                          // [k][row]  A21 tile, 64 x TILE_LD
    double *sX = s_pan + 64 * TILE_LD;           // [n][k]    L11, then L11^-1, row-major, stride TILE_LD
    double *s_col = sX + 64 * TILE_LD;           // 2 x 64   pivot column (double buffered)
    double *s_g = s_col + 128;                   // 64       g1, then y1
    double *s_rd = s_g + 64;                     // 64       d_k, then 1 / L11[k][k]
    double *sT = s_rd + 64;                      // 32 x PANEL_LDT  L21 X11 of the current inversion level
    int *s_bad = reinterpret_cast<int *>(sT + 32 * PANEL_LDT);
    const int tid = threadIdx.x;
    const int R0 = cta * 64;                     // first row of this CTA's tile, relative to j0 + nb
    const long long r0 = j0 + nb;

    // ---- load A11: thread (i, c) = (tid / 4, tid % 4) owns u[kk] = A[i][4 kk + c], kk = 0..15 ----
    const int ri = tid >> 2, rc = tid & 3;
    double u[16];
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
        const int k = 4 * kk + rc;
        double v = (ri == k) ? 1.0 : 0.0;                     // identity padding when nb < 64
        if (ri < nb && k < nb && k <= ri) v = AB[(j0 + ri) + (j0 + k) * lda];
        u[kk] = v;
    }
    if (tid < 64) s_g[tid] = (tid < nb) ? g[j0 + tid] : 0.0;
    if (tid == 0) *s_bad = 0;

    // ---- start streaming this CTA's A21 tile into shared memory; it lands under the factorization ----
    spl_tile_load16(sA, AB + (r0 + R0) + j0 * lda, lda, m - R0, nb, tid);
    asm volatile("cp.async.commit_group;" ::: "memory");
    if (failed) {
        spl_cp_async_wait_all();
        return;
    }

    PANEL_STAMP(1);
    spl_chol64(u, s_col, s_rd, s_bad, tid);
    PANEL_STAMP(2);
    if (*s_bad) {
        if (cta == 0 && tid == 0) *fail = 1;
        spl_cp_async_wait_all();
        return;
    }
    spl_linv64(u, s_rd, sX, sT, tid);
    // L11^-1 for the back-substitution: every CTA has it, each stores a slice of its rows
    {
        const int rows = (64 + ncta - 1) / ncta;
        const int rlo = cta * rows, rhi = min(64, rlo + rows);
        for (int e = rlo * 64 + tid; e < rhi * 64; e += PANEL_THREADS) linv_blk[e] = sX[(e >> 6) * TILE_LD + (e & 63)];
    }
    PANEL_STAMP(3);
    spl_cp_async_wait_all();
    __syncthreads();
    PANEL_STAMP(4);
    const double y1c = spl_y1_64(sX, s_g, tid);
    __syncthreads();
    if (rc == 0) {
        s_g[ri] = y1c;
        if (cta == 0 && ri < nb) ysol[j0 + ri] = y1c;
    }
    __syncthreads();
    PANEL_STAMP(5);
    if (m <= 0) return;
    spl_l21_gemm(AB, lda, j0, nb, m, r0, R0, g, sA, sX, s_g, keep_l21, tid);
    PANEL_STAMP(6);
}

__global__ void __launch_bounds__(PANEL_THREADS)
spl_panel_kernel(double *__restrict__ AB, long long lda, long long j0, int nb, int m,
                 double *__restrict__ g, double *__restrict__ ysol, double *__restrict__ linv_blk,
                 int *__restrict__ fail, long long *__restrict__ dbg) {
    extern __shared__ __align__(16) double s_pan[];
    // the flag is loaded now and tested inside the body after the loads have been issued, so its L2 round trip is
    // not on the chain
    const int failed = *reinterpret_cast<const volatile int *>(fail);
    spl_panel_body(AB, lda, j0, nb, m, g, ysol, linv_blk, fail, dbg, s_pan, (int)blockIdx.x, (int)gridDim.x, failed);
}

// ------------------------------------------------------------------------------------------
// trailing update with FP64 tensor-core MMA
// ------------------------------------------------------------------------------------------
#define SYRK_TILE 64
#define SYRK_THREADS 128

// C[I,J] -= P[I,:] P[J,:]^T over the lower-triangular tiles of the m x m window whose first
// row/column is global index r0; P = panel rows r0.., columns j0..j0+nb-1.  Operand tiles are
// streamed with cp.async (k-major, conflict-free fragment reads); the C tile is prefetched into the
// accumulators while the operands are in flight, so the kernel is one global round trip long.
// part 0: the first tile column (tj = 0, one CTA per tile row) -- all the next panel depends on;
// part 1: every other lower-triangular tile (ti >= tj >= 1), launched on the auxiliary stream so that it
// overlaps the next panel's latency chain (look-ahead).
// One 64 x 64 tile (ti, tj), ti >= tj, with NTHR threads (128: 2 x 2 warps of 32 x 32; 256: 4 x 2 warps of 16 x 32).
// A_READY: the A operand (rows of tile row ti, k-major) is already in shared memory.
template <int NTHR, bool A_READY = false>
__device__ __forceinline__ void spl_syrk_tile(double *AB, long long lda, long long r0, long long j0, int nb, int m,
                                              int ti, int tj, double *s_ab) {
    constexpr int MI = (NTHR == 128) ? 4 : 2;
    double *sA = s_ab;                          // [k][row]
    double *sB = s_ab + 64 * TILE_LD;
    const int I0 = ti * SYRK_TILE, J0 = tj * SYRK_TILE;
    const int t = threadIdx.x;
    const bool diag = (ti == tj);

    {
        // thread t owns row r = t % 64 of both operand tiles and every (NTHR / 64)-th k: pointers advance by a constant,
        // no index arithmetic per element (the per-element form made the tile issue-bound in its load phase)
        constexpr int KS = NTHR / 64;
        const int r = t & 63, kq = t >> 6;
        const bool a_ok = I0 + r < m, b_ok = J0 + r < m;
        const double *ga = AB + (r0 + I0 + r) + (j0 + kq) * lda;
        const double *gb = AB + (r0 + J0 + r) + (j0 + kq) * lda;
        double *da = sA + kq * TILE_LD + r, *db = sB + kq * TILE_LD + r;
        const long long gstep = (long long)KS * lda;
#pragma unroll 4
        for (int k = kq; k < 64; k += KS) {
            if (!A_READY) {
                if (a_ok && k < nb) spl_cp_async8(da, ga);
                else *da = 0.0;
            }
            if (!diag) {
                if (b_ok && k < nb) spl_cp_async8(db, gb);
                else *db = 0.0;
            }
            ga += gstep;
            gb += gstep;
            da += KS * TILE_LD;
            db += KS * TILE_LD;
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");

    const int warp = t >> 5, lane = t & 31;
    const int g = lane >> 2, t4 = lane & 3;
    const int wy = (warp >> 1) * (MI * 8), wx = (warp & 1) * 32;
    // the C tile: element (mi, ni, h) of this thread at pc[mi * 8 + (ni * 8 + h) * lda]
    double *pc = AB + (r0 + I0 + wy + g) + (r0 + J0 + wx + 2 * t4) * lda;
    const bool inside = !diag && I0 + 64 <= m && J0 + 64 <= m;     // every element valid: no per-element tests
    // prefetch the C tile into the accumulators (lower triangle, inside the window)
    double acc[MI][4][2];
    if (inside) {
#pragma unroll
        for (int mi = 0; mi < MI; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int h = 0; h < 2; ++h) acc[mi][ni][h] = pc[mi * 8 + (long long)(ni * 8 + h) * lda];
    } else {
#pragma unroll
        for (int mi = 0; mi < MI; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int li = I0 + wy + mi * 8 + g;
                    const int lj = J0 + wx + ni * 8 + 2 * t4 + h;
                    acc[mi][ni][h] = (li < m && lj < m && li >= lj) ? pc[mi * 8 + (long long)(ni * 8 + h) * lda] : 0.0;
                }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    const double *pB = diag ? sA : sB;

#pragma unroll 4
    for (int k0 = 0; k0 < 64; k0 += 4) {
        double a[MI], b[4];
#pragma unroll
        for (int mi = 0; mi < MI; ++mi) a[mi] = -sA[(k0 + t4) * TILE_LD + wy + mi * 8 + g];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) b[ni] = pB[(k0 + t4) * TILE_LD + wx + ni * 8 + g];
#pragma unroll
        for (int mi = 0; mi < MI; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) spl_dmma_8x8x4(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
    }
    if (inside) {
#pragma unroll
        for (int mi = 0; mi < MI; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int h = 0; h < 2; ++h) pc[mi * 8 + (long long)(ni * 8 + h) * lda] = acc[mi][ni][h];
    } else {
#pragma unroll
        for (int mi = 0; mi < MI; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int li = I0 + wy + mi * 8 + g;
                    const int lj = J0 + wx + ni * 8 + 2 * t4 + h;
                    if (li < m && lj < m && li >= lj) pc[mi * 8 + (long long)(ni * 8 + h) * lda] = acc[mi][ni][h];
                }
    }
}

// Half of a 64 x 64 tile (rows half*32 .. +32) with 256 threads (4 x 2 warps of 8 x 32): the persistent factor kernel
// splits the tiles of the last, partial round among its helper CTAs so that nobody carries a whole extra tile.
__device__ __forceinline__ void spl_syrk_half_tile(double *AB, long long lda, long long r0, long long j0, int nb, int m,
                                                   int ti, int tj, int half, double *s_ab) {
    double *sA = s_ab;                          // [k][row 0..31]
    double *sB = s_ab + 64 * TILE_LD;
    const int I0 = ti * SYRK_TILE + half * 32, J0 = tj * SYRK_TILE;
    const int t = threadIdx.x;
    for (int e = t; e < 64 * 64; e += PANEL_THREADS) {
        const int k = e >> 6, r = e & 63;
        if (r < 32) {
            double *da = sA + k * TILE_LD + r;
            if (k < nb && I0 + r < m) spl_cp_async8(da, AB + (r0 + I0 + r) + (j0 + k) * lda);
            else *da = 0.0;
        }
        double *db = sB + k * TILE_LD + r;
        if (k < nb && J0 + r < m) spl_cp_async8(db, AB + (r0 + J0 + r) + (j0 + k) * lda);
        else *db = 0.0;
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    const int warp = t >> 5, lane = t & 31;
    const int g = lane >> 2, t4 = lane & 3;
    const int wy = (warp >> 1) * 8, wx = (warp & 1) * 32;
    double acc[4][2];
#pragma unroll
    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int li = I0 + wy + g;
            const int lj = J0 + wx + ni * 8 + 2 * t4 + h;
            acc[ni][h] = (li < m && lj < m && li >= lj) ? AB[(r0 + li) + (r0 + lj) * lda] : 0.0;
        }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
#pragma unroll 4
    for (int k0 = 0; k0 < 64; k0 += 4) {
        const double a = -sA[(k0 + t4) * TILE_LD + wy + g];
        double b[4];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) b[ni] = sB[(k0 + t4) * TILE_LD + wx + ni * 8 + g];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) spl_dmma_8x8x4(acc[ni][0], acc[ni][1], a, b[ni]);
    }
#pragma unroll
    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int li = I0 + wy + g;
            const int lj = J0 + wx + ni * 8 + 2 * t4 + h;
            if (li < m && lj < m && li >= lj) AB[(r0 + li) + (r0 + lj) * lda] = acc[ni][h];
        }
}

// rest-of-update tile number (0 .. (T-1) T / 2 - 1)  ->  (ti, tj) with ti >= tj >= 1
__device__ __forceinline__ void spl_rest_tile(int tile, int &ti, int &tj) {
    ti = (int)((sqrt(8.0 * (double)tile + 1.0) - 1.0) * 0.5);
    while ((long long)(ti + 1) * (ti + 2) / 2 <= tile) ++ti;
    while ((long long)ti * (ti + 1) / 2 > tile) --ti;
    tj = tile - ti * (ti + 1) / 2 + 1;
    ti += 1;
}

__global__ void __launch_bounds__(SYRK_THREADS)
spl_syrk_kernel(double *__restrict__ AB, long long lda, long long r0, long long j0, int nb, int m,
                const int *__restrict__ fail, int part) {
    extern __shared__ __align__(16) double s_ab[];
    if (*fail) return;
    int ti, tj;
    if (part == 0) {
        ti = blockIdx.x;
        tj = 0;
    } else {
        spl_rest_tile((int)blockIdx.x, ti, tj);
    }
    spl_syrk_tile<SYRK_THREADS>(AB, lda, r0, j0, nb, m, ti, tj, s_ab);
}

// ------------------------------------------------------------------------------------------
// Update tile for 256 threads, split in two halves so that a CTA with a list of tiles can have the operands of the
// next tile in flight under the MMA stream of the current one:
//   spl_tile_issue   operands of tile (ti, tj) -> shared memory buffer (sA | sB), k-major, 16-byte cp.async, one
//                    committed group;
//   spl_tile_finish  C tile -> accumulators (128-bit loads), wait for the operands, 64 x 64 x 64 on the FP64 tensor
//                    cores, 128-bit stores.  The product is formed TRANSPOSED (the MMA's rows are the tile's columns
//                    J, the MMA's column pairs are consecutive rows I), so the two accumulators of a fragment are
//                    adjacent in the column-major band matrix.
// Warp w of 8: rows I in [32 (w & 1), +32), columns J in [16 (w >> 1), +16).
// ------------------------------------------------------------------------------------------
// half = -1: the whole tile; 0 / 1: its rows [32 half, +32) only (the last, partial round of a helper list is split
// in row halves so that nobody carries a whole extra tile) -- the A operand then holds 32 rows, B all 64 even on the
// diagonal, and the eight warps take 32 x 8 each (MJ = 1) instead of 32 x 16.
template <bool A_READY>
__device__ __forceinline__ void spl_tile_issue(const double *AB, long long lda, long long r0, long long j0, int nb,
                                               int m, int ti, int tj, double *s_ab, const int half = -1) {
    const int t = threadIdx.x;
    const int I0 = ti * SYRK_TILE + (half > 0 ? 32 : 0), J0 = tj * SYRK_TILE;
    if (!A_READY) {
        int rows = m - I0;
        if (half >= 0 && rows > 32) rows = 32;
        spl_tile_load16(s_ab, AB + (r0 + I0) + j0 * lda, lda, rows, nb, t);
    }
    if (ti != tj || half >= 0) spl_tile_load16(s_ab + 64 * TILE_LD, AB + (r0 + J0) + j0 * lda, lda, m - J0, nb, t);
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// C tile of (ti, tj) -> accumulators.  Thread layout, MJ = 2 (warp w of 8: rows I in [32 (w & 1), +32), columns J in
// [16 (w >> 1), +16)) or MJ = 1 (half tile: rows [0, 32) of the half, columns [8 w, +8)):
// accumulator (mj, ni, h) = C[I0 + wI + ni 8 + 2 t4 + h][J0 + wJ + mj 8 + g].
template <int MJ>
__device__ __forceinline__ void spl_tile_cload(double (&acc)[2][4][2], const double *AB, long long lda, long long r0,
                                               int m, int ti, int tj, const int half = -1) {
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int g = lane >> 2, t4 = lane & 3;
    const int wI = (MJ == 2) ? (warp & 1) * 32 : 0, wJ = (MJ == 2) ? (warp >> 1) * 16 : warp * 8;
    const int I0 = ti * SYRK_TILE + (half > 0 ? 32 : 0), J0 = tj * SYRK_TILE;
    const double *pc = AB + (r0 + I0 + wI + 2 * t4) + (r0 + J0 + wJ + g) * lda;
    const bool inside = ti != tj && I0 + (MJ == 2 ? 64 : 32) <= m && J0 + 64 <= m;   // no per-element tests
    if (inside) {
#pragma unroll
        for (int mj = 0; mj < MJ; ++mj)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) {
                const double2 v = __ldcg(reinterpret_cast<const double2 *>(pc + ni * 8 + (long long)(mj * 8) * lda));
                acc[mj][ni][0] = v.x;
                acc[mj][ni][1] = v.y;
            }
    } else {
#pragma unroll
        for (int mj = 0; mj < MJ; ++mj)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    // raw, unconditional loads; spl_tile_mma_store masks them when it starts, i.e. when they have landed
                    // (a conditional load becomes a branch per element, and a select right here would wait for the L2
                    // round trip before the previous tile's MMA stream instead of under it).  The address of an element
                    // outside the window or above the diagonal is still inside the band array: a column has
                    // lda >= bw + 64 rows and the array 64 spare elements behind the last column.
                    acc[mj][ni][h] = __ldcg(pc + ni * 8 + h + (long long)(mj * 8) * lda);
                }
    }
}

template <int PENDING, int MJ>   // PENDING: cp.async groups that may stay in flight (1: the next tile's operands)
__device__ __forceinline__ void spl_tile_mma_store(double (&acc)[2][4][2], double *AB, long long lda, long long r0,
                                                   int m, int ti, int tj, const double *s_ab, const int half = -1) {
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int g = lane >> 2, t4 = lane & 3;
    const int wI = (MJ == 2) ? (warp & 1) * 32 : 0, wJ = (MJ == 2) ? (warp >> 1) * 16 : warp * 8;
    const int I0 = ti * SYRK_TILE + (half > 0 ? 32 : 0), J0 = tj * SYRK_TILE;
    const bool diag = (ti == tj);
    const double *sA = s_ab;
    const double *sB = (diag && half < 0) ? s_ab : s_ab + 64 * TILE_LD;
    double *pc = AB + (r0 + I0 + wI + 2 * t4) + (r0 + J0 + wJ + g) * lda;
    const bool inside = !diag && I0 + (MJ == 2 ? 64 : 32) <= m && J0 + 64 <= m;
    if (PENDING == 0) asm volatile("cp.async.wait_group 0;" ::: "memory");
    else asm volatile("cp.async.wait_group 1;" ::: "memory");
    SPL_SYNC256();
    if (!inside) {
#pragma unroll
        for (int mj = 0; mj < MJ; ++mj)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int li = I0 + wI + ni * 8 + 2 * t4 + h;
                    const int lj = J0 + wJ + mj * 8 + g;
                    if (!(li < m && lj < m && li >= lj)) acc[mj][ni][h] = 0.0;
                }
    }
#pragma unroll 4
    for (int k0 = 0; k0 < 64; k0 += 4) {
        double a[MJ], b[4];
#pragma unroll
        for (int mj = 0; mj < MJ; ++mj) a[mj] = -sB[(k0 + t4) * TILE_LD + wJ + mj * 8 + g];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) b[ni] = sA[(k0 + t4) * TILE_LD + wI + ni * 8 + g];
#pragma unroll
        for (int mj = 0; mj < MJ; ++mj)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) spl_dmma_8x8x4(acc[mj][ni][0], acc[mj][ni][1], a[mj], b[ni]);
    }
    if (inside) {
#pragma unroll
        for (int mj = 0; mj < MJ; ++mj)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
                *reinterpret_cast<double2 *>(pc + ni * 8 + (long long)(mj * 8) * lda) =
                    make_double2(acc[mj][ni][0], acc[mj][ni][1]);
    } else {
#pragma unroll
        for (int mj = 0; mj < MJ; ++mj)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int li = I0 + wI + ni * 8 + 2 * t4 + h;
                    const int lj = J0 + wJ + mj * 8 + g;
                    if (li < m && lj < m && li >= lj) pc[ni * 8 + h + (long long)(mj * 8) * lda] = acc[mj][ni][h];
                }
    }
}

template <int PENDING>
__device__ __forceinline__ void spl_tile_finish(double *AB, long long lda, long long r0, int m, int ti, int tj,
                                                const double *s_ab) {
    double acc[2][4][2];
    spl_tile_cload<2>(acc, AB, lda, r0, m, ti, tj);
    spl_tile_mma_store<PENDING, 2>(acc, AB, lda, r0, m, ti, tj, s_ab);
}

template <bool A_READY>
__device__ __forceinline__ void spl_tile256(double *AB, long long lda, long long r0, long long j0, int nb, int m,
                                            int ti, int tj, double *s_ab) {
    spl_tile_issue<A_READY>(AB, lda, r0, j0, nb, m, ti, tj, s_ab);
    spl_tile_finish<0>(AB, lda, r0, m, ti, tj, s_ab);
}

// The same tile launch with the 256-thread tile (16-byte cp.async operands, 128-bit C accesses): the kernel-per-phase
// driver's trailing update (SPLPAK_B200_SYRK=128 selects the older 128-thread tile for A/B).
__global__ void __launch_bounds__(PANEL_THREADS, 3)
spl_syrk256_kernel(double *__restrict__ AB, long long lda, long long r0, long long j0, int nb, int m,
                   const int *__restrict__ fail, int part) {
    extern __shared__ __align__(16) double s_ab[];
    if (*fail) return;
    int ti, tj;
    if (part == 0) {
        ti = blockIdx.x;
        tj = 0;
    } else {
        spl_rest_tile((int)blockIdx.x, ti, tj);
    }
    spl_tile256<false>(AB, lda, r0, j0, nb, m, ti, tj, s_ab);
}

// ------------------------------------------------------------------------------------------
// Two-level blocking for the update-bound shape (cfg4: half bandwidth 5,655 = 89 tile rows, 3,916 update tiles per
// panel).  With one 64-column panel per trailing update every 64 x 64 tile of the 128 MB band window is read and
// written once per 64 x 64 x 64 product: 8 flops per byte of C traffic plus the operand tiles, and the kernel-per-phase
// loop ran at 51 % of the DMMA peak.  Here KB (8; SPLPAK_B200_KBLOCK) panels form an outer block: inside the block a panel's update only
// touches the block's own remaining columns (spl_syrk_cols_kernel: <= KB - 1 tile columns, the existing K = 64 tile),
// and the trailing matrix beyond the block gets ONE update with K = 64 KB (spl_syrk_kblock_kernel): the C tile stays in
// the accumulators while the 2 KB operand half-chunks (32 columns of one panel) stream through a double-buffered
// 2 x 34.8 KB staging area -- a quarter of the C traffic, and the tile's prologue / epilogue amortised over 4x the MMAs.
// The band windows of the block's panels differ (panel p reaches KB - 1 - p tile rows less far than the last one):
// rows beyond a panel's window are zero-filled by the operand loader, and half-chunks whose window ends above the
// tile are skipped.  Same arithmetic as the unblocked loop (every C element receives the panels' contributions in
// panel order), so the two agree to the rounding of the MMA's internal order.
// ------------------------------------------------------------------------------------------
#define KBLOCK_MAX 8

// NK (32) k-columns of an operand tile: like spl_tile_load16 with every column present; 4 pieces per thread
template <int NK>
__device__ __forceinline__ void spl_tile_loadk(double *s, const double *src, const long long lda, const int rows,
                                               const int t) {
    const int r = 2 * (t & 31);
    const int k = t >> 5;
    const double *gp = src + r + (long long)k * lda;
    double *dp = s + k * TILE_LD + r;
    const int valid = rows - r;
    const long long gstep = 8 * lda;
#pragma unroll
    for (int q = 0; q < NK / 8; ++q) {
        spl_tile_piece(dp, gp, valid, true);
        gp += gstep;
        dp += 8 * TILE_LD;
    }
}

// Update of the block's own columns by panel (j0, nb): tiles (ti = blockIdx.x, tj = blockIdx.y < gridDim.y), ti >= tj.
__global__ void __launch_bounds__(PANEL_THREADS, 3)
spl_syrk_cols_kernel(double *__restrict__ AB, long long lda, long long r0, long long j0, int nb, int m,
                     const int *__restrict__ fail) {
    extern __shared__ __align__(16) double s_ab[];
    const int ti = blockIdx.x, tj = blockIdx.y;
    if (ti < tj || *fail) return;
    spl_tile256<false>(AB, lda, r0, j0, nb, m, ti, tj, s_ab);
}

// Trailing update by the np panels of the outer block that starts at column jb (all 64 wide; R0 = jb + 64 np is the
// first trailing row / column).  part 0: tile columns [0, c0) (what the next outer block factors: the critical path),
// grid (T, c0); part 1: tile columns >= c0, the lower triangle enumerated linearly.
__global__ void __launch_bounds__(PANEL_THREADS, 3)
spl_syrk_kblock_kernel(double *__restrict__ AB, long long lda, long long jb, int np, long long n, int bw,
                       const int *__restrict__ fail, int part, int c0) {
    extern __shared__ __align__(16) double s_ab[];
    constexpr int HALF = 32 * TILE_LD;            // one operand half-chunk (32 k-columns)
    constexpr int BUF = 2 * HALF;                 // A | B
    int ti, tj;
    if (part == 0) {
        ti = blockIdx.x;
        tj = blockIdx.y;
        if (ti < tj) return;
    } else {
        spl_rest_tile((int)blockIdx.x, ti, tj);
        ti += c0 - 1;
        tj += c0 - 1;
    }
    if (*fail) return;
    const long long R0 = jb + (long long)np * SOLVE_NB;
    const int M = (int)((n - R0 < bw) ? n - R0 : bw);             // window of the last panel = the update's extent
    const int I0 = ti * SYRK_TILE, J0 = tj * SYRK_TILE;
    if (I0 >= M) return;
    const bool diag = (ti == tj);
    const int t = threadIdx.x;
    // window of panel p in R0-relative rows: Mp = min(bw, n - r0_p) - 64 (np - 1 - p), non-decreasing in p
    int pfirst = 0;
    while (pfirst < np - 1) {
        const long long r0p = jb + (long long)(pfirst + 1) * SOLVE_NB;
        const long long mp = (n - r0p < bw) ? n - r0p : bw;
        if (mp - (long long)SOLVE_NB * (np - 1 - pfirst) > I0) break;
        ++pfirst;
    }
    const int h0 = 2 * pfirst, H = 2 * np;
    // window (R0-relative rows) of the first contributing panel: when it covers the whole tile row, every operand
    // piece of every half-chunk is a full 16-byte cp.async and the loads are pointer bumps without tests
    int Mfirst;
    {
        const long long r0p = jb + (long long)(pfirst + 1) * SOLVE_NB;
        const long long mp = (n - r0p < bw) ? n - r0p : bw;
        Mfirst = (int)(mp - (long long)SOLVE_NB * (np - 1 - pfirst));
    }
    const bool full = I0 + 64 <= Mfirst;
    const int lr = 2 * (t & 31), lk = t >> 5;
    const double *ga = AB + (R0 + I0 + lr) + (jb + 32LL * h0 + lk) * lda;      // half-chunk h0, this thread's first piece
    const double *gb = AB + (R0 + J0 + lr) + (jb + 32LL * h0 + lk) * lda;
    const uint32_t sdst = (uint32_t)__cvta_generic_to_shared(s_ab + lk * TILE_LD + lr);
    const long long gstep = 8 * lda;
    auto issue = [&](int h) {
        if (full) {
            const uint32_t d = sdst + (uint32_t)((h & 1) * BUF * sizeof(double));
#pragma unroll
            for (int q = 0; q < 4; ++q)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + (uint32_t)(q * 8 * TILE_LD * sizeof(double))),
                             "l"(ga + q * gstep) : "memory");
            if (!diag) {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + (uint32_t)((HALF + q * 8 * TILE_LD) * sizeof(double))),
                                 "l"(gb + q * gstep) : "memory");
            }
            ga += 4 * gstep;
            gb += 4 * gstep;
        } else {
            const int p = h >> 1;
            const long long j0p = jb + (long long)p * SOLVE_NB + 32 * (h & 1);
            const long long r0p = jb + (long long)(p + 1) * SOLVE_NB;
            const long long mp = (n - r0p < bw) ? n - r0p : bw;
            const int Mp = (int)(mp - (long long)SOLVE_NB * (np - 1 - p));
            double *buf = s_ab + (h & 1) * BUF;
            spl_tile_loadk<32>(buf, AB + (R0 + I0) + j0p * lda, lda, Mp - I0, t);
            if (!diag) spl_tile_loadk<32>(buf + HALF, AB + (R0 + J0) + j0p * lda, lda, Mp - J0, t);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    issue(h0);
    double acc[2][4][2];
    spl_tile_cload<2>(acc, AB, lda, R0, M, ti, tj);

    const int warp = t >> 5, lane = t & 31;
    const int g = lane >> 2, t4 = lane & 3;
    const int wI = (warp & 1) * 32, wJ = (warp >> 1) * 16;
    const bool inside = !diag && I0 + 64 <= M && J0 + 64 <= M;
    for (int h = h0; h < H; ++h) {
        // one barrier per half-chunk: behind it every warp has finished the MMAs of h - 1, so their buffer is free for
        // h + 1, and everybody's pieces of h have landed
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        if (h + 1 < H) issue(h + 1);
        if (h == h0 && !inside) {
#pragma unroll
            for (int mj = 0; mj < 2; ++mj)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        const int li = I0 + wI + ni * 8 + 2 * t4 + hh;
                        const int lj = J0 + wJ + mj * 8 + g;
                        if (!(li < M && lj < M && li >= lj)) acc[mj][ni][hh] = 0.0;
                    }
        }
        const double *sA = s_ab + (h & 1) * BUF;
        const double *sB = diag ? sA : sA + HALF;
#pragma unroll 4
        for (int k0 = 0; k0 < 32; k0 += 4) {
            double a[2], b[4];
#pragma unroll
            for (int mj = 0; mj < 2; ++mj) a[mj] = -sB[(k0 + t4) * TILE_LD + wJ + mj * 8 + g];
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) b[ni] = sA[(k0 + t4) * TILE_LD + wI + ni * 8 + g];
#pragma unroll
            for (int mj = 0; mj < 2; ++mj)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) spl_dmma_8x8x4(acc[mj][ni][0], acc[mj][ni][1], a[mj], b[ni]);
        }
    }
    double *pc = AB + (R0 + I0 + wI + 2 * t4) + (R0 + J0 + wJ + g) * lda;
    if (inside) {
#pragma unroll
        for (int mj = 0; mj < 2; ++mj)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
                *reinterpret_cast<double2 *>(pc + ni * 8 + (long long)(mj * 8) * lda) =
                    make_double2(acc[mj][ni][0], acc[mj][ni][1]);
    } else {
#pragma unroll
        for (int mj = 0; mj < 2; ++mj)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int li = I0 + wI + ni * 8 + 2 * t4 + hh;
                    const int lj = J0 + wJ + mj * 8 + g;
                    if (li < M && lj < M && li >= lj) pc[ni * 8 + hh + (long long)(mj * 8) * lda] = acc[mj][ni][hh];
                }
    }
}

// ------------------------------------------------------------------------------------------
// persistent factorisation: the whole right-looking loop in ONE cooperative kernel (one 256-thread CTA per SM),
// phases separated by grid-wide barriers instead of kernel boundaries and cross-stream events:
//   step kb, phase P:  CTAs [0, pblocks) run panel(kb)  ||  the other CTAs finish the trailing update of step kb-1
//                      (tiles with tj >= 1: nothing panel(kb) reads -- the look-ahead of the two-stream version)
//            grid barrier
//            phase C:  tile column 0 of update kb (all panel(kb+1) needs) on CTAs [0, T); every other CTA takes ONE
//                      tile of the rest of update kb, so the phase is one tile long for everyone
//            grid barrier
// The kernel-boundary version spent 11 us per step between its panel kernels (column-0 kernel + two boundaries)
// and its two streams slowed each other down (6.8 ms for 216 steps at cfg3).
// ------------------------------------------------------------------------------------------
// Grid-wide barrier of the persistent kernel (all CTAs are co-resident: cooperative launch).  One monotonically
// increasing counter; the k-th barrier is passed when it reaches k * G.  cooperative_groups' grid.sync() cost 3 us
// per barrier here, a third of the step.
__device__ __forceinline__ void spl_grid_barrier(unsigned *counter, unsigned &target, unsigned G) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += G;
        // release: the CTA's writes (ordered before this thread by the bar.sync above) are visible to whoever
        // observes the increment with an acquire load -- one instruction instead of a fence + a relaxed atomic,
        // and the acquire poll needs no fence after it
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
        unsigned v;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
        } while (v < target);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(PANEL_THREADS, 1)
spl_factor_persistent_kernel(double *AB, long long lda, long long n, int bw, double *g, double *ysol, double *linv,
                             int *fail, long long *dbg, unsigned *bar) {
    extern __shared__ __align__(16) double s_dyn_f[];
    const int G = (int)gridDim.x, cta = (int)blockIdx.x;
    unsigned bar_target = 0;
    const long long nblk = (n + SOLVE_NB - 1) / SOLVE_NB;
    // trailing update still owed from the previous step: window (r0, j0, nb, m), first rest tile not yet done
    long long pr0 = 0, pj0 = 0;
    int pnb = 0, pm = 0, pfirst = 0, pntiles = 0;
    for (long long kb = 0; kb < nblk; ++kb) {
        const long long j0 = kb * SOLVE_NB;
        const int nb = (int)((n - j0 < SOLVE_NB) ? n - j0 : SOLVE_NB);
        const long long r0 = j0 + nb;
        long long mm = n - r0;
        if (mm > bw) mm = bw;
        const int m = (int)mm;
        int pblocks = (m + 63) / 64;
        if (pblocks < 1) pblocks = 1;
        const bool one_row_each = pblocks <= G && m > 0;      // CTA c holds L21 of tile row c after the panel
        if (pblocks > G) pblocks = G;            // (never at the sizes this library targets: bw <= 64 G)
        // ---- phase P ----
        if (cta < pblocks) {
            // every panel CTA covers rows cta, cta + pblocks, .. (one tile row each unless bw > 64 G)
            for (int c = cta; c * 64 < (m > 0 ? m : 1); c += pblocks) {
                spl_panel_body(AB, lda, j0, nb, m, g, ysol, linv + kb * 4096, fail,
                               (kb == nblk / 2) ? dbg : nullptr, s_dyn_f, c, (m + 63) / 64 > 0 ? (m + 63) / 64 : 1, 0,
                               one_row_each);
                __syncthreads();
            }
        } else if (pntiles > pfirst) {
            // whole rounds of full tiles; the tiles of the last, partial round are split into row halves when that
            // lets every helper finish one half instead of some a whole tile (the barrier waits for the slowest)
            const int helpers = G - pblocks, me = cta - pblocks;
            const int todo = pntiles - pfirst;
            const int nfull = (todo / helpers) * helpers, rem = todo - nfull;
            for (int u = me; u < nfull; u += helpers) {
                int ti, tj;
                spl_rest_tile(pfirst + u, ti, tj);
                spl_tile256<false>(AB, lda, pr0, pj0, pnb, pm, ti, tj, s_dyn_f);
                __syncthreads();
            }
            if (2 * rem <= helpers) {
                if (me < 2 * rem) {
                    int ti, tj;
                    spl_rest_tile(pfirst + nfull + (me >> 1), ti, tj);
                    if (ti != tj) spl_syrk_half_tile(AB, lda, pr0, pj0, pnb, pm, ti, tj, me & 1, s_dyn_f);
                    else if ((me & 1) == 0) spl_tile256<false>(AB, lda, pr0, pj0, pnb, pm, ti, tj, s_dyn_f);
                }
            } else if (me < rem) {
                int ti, tj;
                spl_rest_tile(pfirst + nfull + me, ti, tj);
                spl_tile256<false>(AB, lda, pr0, pj0, pnb, pm, ti, tj, s_dyn_f);
            }
        }
        if (dbg && kb == nblk / 2 && cta == 0 && threadIdx.x == 0) dbg[12] = clock64();
        spl_grid_barrier(bar, bar_target, (unsigned)G);
        if (dbg && kb == nblk / 2 && cta == 0 && threadIdx.x == 0) dbg[13] = clock64();
        if (*reinterpret_cast<volatile int *>(fail)) return;     // uniform: everybody reads it after the barrier
        // ---- phase C ----
        const int T = (m + SYRK_TILE - 1) / SYRK_TILE;
        const int ntiles = (T > 1) ? (T - 1) * T / 2 : 0;
        int first = 0;
        if (m > 0) {
            if (cta < T) {
                for (int ti = cta; ti < T; ti += G) {
                    if (one_row_each && ti == cta) spl_tile256<true>(AB, lda, r0, j0, nb, m, ti, 0, s_dyn_f);
                    else spl_tile256<false>(AB, lda, r0, j0, nb, m, ti, 0, s_dyn_f);
                    __syncthreads();
                }
            } else if (cta - T < ntiles) {
                int ti, tj;
                spl_rest_tile(cta - T, ti, tj);
                spl_tile256<false>(AB, lda, r0, j0, nb, m, ti, tj, s_dyn_f);
            }
            first = (G - T > 0) ? ((G - T < ntiles) ? G - T : ntiles) : 0;
        }
        pr0 = r0;
        pj0 = j0;
        pnb = nb;
        pm = m;
        pfirst = first;
        pntiles = ntiles;
        if (dbg && kb == nblk / 2 && cta == 0 && threadIdx.x == 0) dbg[14] = clock64();
        spl_grid_barrier(bar, bar_target, (unsigned)G);
        if (dbg && kb == nblk / 2 && cta == 0 && threadIdx.x == 0) dbg[15] = clock64();
    }
}

// ------------------------------------------------------------------------------------------
// DATA-FLOW factorisation (default where the panel chain dominates): one cooperative kernel, one CTA per SM, three
// roles coupled by release/acquire flags instead of grid-wide phases.  The critical path of the right-looking loop is
//   chol(k) -> L11^-1 -> L[k+1,k] -> update of block (k+1,k+1) -> chol(k+1);
// the barrier-phased kernel above put two grid barriers, a global round trip of the diagonal block and the slowest
// helper's tile on it (43k clocks per step at cfg3 for a 28k chain).  Here
//   CTA 0 (diagonal)    eight compute warps run exactly that chain and touch shared memory only: the updated
//                       diagonal block never leaves the SM.  A NINTH warp does everything that talks to the rest of
//                       the GPU, coupled to the compute warps by named barriers: it waits for the two blocks the step
//                       reads (flags T10, T11: one step behind) and streams them in under the factorization, stores
//                       L11^-1 and y1 and raises LINV, stores L[k+1,k], forms this CTA's share of g2 -= L21 y1 and
//                       raises L10 -- fences, flag polls and global stores are off the chain.
//   CTAs 1 .. Tmax-1    tile rows 1.. of the panel: wait for LINV, L21 = A21 L11^-T, g2 -= L21 y1  | barrier B1 (all
//   (panel workers)     workers) | column-0 tile of their row (A operand still in shared memory; B = L[k+1,k], flag
//                       L10); CTA 1 raises T10 | barrier B2 (panel workers only: the next A21 tiles are final) | one
//                       rest tile from the end of the list while the diagonal CTA factors the next block.
//   the other CTAs      B1(k), then the rest tiles (ti >= tj >= 1) of update k as ONE list with the next tile's
//   (helpers)           operands and C tile in flight under the current MMA stream; helper 0 starts with (1,1) and
//                       raises T11.
// Every spin gives up when the failure flag is set or after a watchdog interval (which sets it), so the kernel
// cannot hang; a failure is reported as 107 like a non-positive pivot.
// ------------------------------------------------------------------------------------------
#define DF_THREADS 288                     // 8 working warps + the diagonal CTA's communication warp
#define DF_FLAG_STRIDE 32                  // unsigneds between flags: one 128-byte line each
enum { DF_B1 = 0, DF_B2 = 1, DF_LINV = 2, DF_L10 = 3, DF_T10 = 4, DF_T11 = 5, DF_NFLAGS = 6 };
#define DF_WATCHDOG_CLOCKS (1LL << 32)     // ~2 s
// named barriers of the diagonal CTA (all 288 threads: one side arrives, the other waits)
#define DF_STR_(x) #x
#define DF_STR(x) DF_STR_(x)
#define DF_BAR_SYNC(id) asm volatile("bar.sync " DF_STR(id) ", 288;" ::: "memory")
#define DF_BAR_ARRIVE(id) asm volatile("bar.arrive " DF_STR(id) ", 288;" ::: "memory")
#define DF_NB_OPER 1        // comm -> compute: the flags of the two blocks this step reads are acquired (and the
                            //                  communication warp is done with the previous step)
#define DF_NB_LINV 2        // compute -> comm: L11^-1 stored
#define DF_NB_L10 3         // compute -> comm: y1 and L[k+1,k] stored, L[k+1,k] also in sA (k-major), y1 in s_g

__device__ __forceinline__ unsigned spl_ld_acquire(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// one thread spins until *flag >= target: relaxed polls (an acquire load invalidates the SM's L1 every time, next
// to warps whose shared-memory chain is the critical path), then ONE acquire load of the flag.  (Measured: relaxed polls
// followed by a fence.acq_rel.gpu are slower, 33.4k -> 39k clocks per step -- the two-way fence waits for the CTA's
// own stores and cp.async prefetches in flight, the one-way acquire load does not.)
__device__ __forceinline__ unsigned spl_ld_relaxed(const unsigned *p) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
template <int SLEEP_NS = 20>
__device__ __forceinline__ void spl_df_spin(const unsigned *flag, const unsigned target, int *fail) {
    if (spl_ld_acquire(flag) >= target) return;
    const long long t0 = clock64();
    unsigned it = 0;
    while (spl_ld_relaxed(flag) < target) {
        __nanosleep(SLEEP_NS);
        if ((++it & 63u) == 0u) {
            if (*reinterpret_cast<volatile int *>(fail)) return;
            if (clock64() - t0 > DF_WATCHDOG_CLOCKS) {
                *reinterpret_cast<volatile int *>(fail) = 2;
                return;
            }
        }
    }
    (void)spl_ld_acquire(flag);
}
__device__ __forceinline__ void spl_df_wait(const unsigned *flag, const unsigned target, int *fail) {
    if (threadIdx.x == 0) spl_df_spin(flag, target, fail);
    SPL_SYNC256();
}
// the CTA's writes so far become visible to whoever acquires the flag
__device__ __forceinline__ void spl_df_post(unsigned *flag, const unsigned value) {
    SPL_SYNC256();
    if (threadIdx.x == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}
// barrier among P CTAs on a monotonically increasing counter (every CTA keeps `target` in step, participant or not)
__device__ __forceinline__ void spl_df_barrier(unsigned *counter, unsigned &target, const unsigned P, int *fail) {
    SPL_SYNC256();
    target += P;
    if (threadIdx.x == 0) {
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
        spl_df_spin(counter, target, fail);
    }
    SPL_SYNC256();
}

#define DF_STAMP(i) do { if (stamp && (threadIdx.x & 255) == 0) dbg[i] = clock64(); } while (0)
// nanoseconds on the device-wide timer: the only clock two CTAs can be compared on
#define DF_STAMP_NS(i) do { if (stamp && (threadIdx.x & 255) == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); dbg[i] = (long long)t_; } } while (0)

__global__ void __launch_bounds__(DF_THREADS, 1)
spl_factor_dataflow_kernel(double *AB, long long lda, long long n, int bw, double *g, double *ysol, double *linv,
                           int *fail, long long *dbg, unsigned *flags) {
    extern __shared__ __align__(16) double s_df[];
    const int G = (int)gridDim.x, cta = (int)blockIdx.x, tid = threadIdx.x;
    const long long nblk = (n + SOLVE_NB - 1) / SOLVE_NB;
    const int Tmax = (bw + SYRK_TILE - 1) / SYRK_TILE > 1 ? (bw + SYRK_TILE - 1) / SYRK_TILE : 1;
    unsigned *f_b1 = flags + DF_B1 * DF_FLAG_STRIDE, *f_b2 = flags + DF_B2 * DF_FLAG_STRIDE;
    unsigned *f_linv = flags + DF_LINV * DF_FLAG_STRIDE, *f_l10 = flags + DF_L10 * DF_FLAG_STRIDE;
    unsigned *f_t10 = flags + DF_T10 * DF_FLAG_STRIDE, *f_t11 = flags + DF_T11 * DF_FLAG_STRIDE;

    if (cta == 0) {
        // ================================ diagonal CTA ================================
        double *sA = s_df;                           // [k][row]  A21 tile row 0, then L[k+1,k] (k-major)
        double *sX = s_df + 64 * TILE_LD;            // L11, then L11^-1 (row-major)
        double *sC = sX + 64 * TILE_LD;              // [col][row] the NEXT diagonal block
        double *s_col = sC + 64 * TILE_LD;           // 2 x 64
        double *s_g = s_col + 128;                   // 64  g1, then y1
        double *s_rd = s_g + 64;                     // 64
        double *s_gn = s_rd + 64;                    // 2 x 64  this CTA's own g2 -= L21 y1 for the next block
        double *sT = s_gn + 128;                     // 32 x PANEL_LDT
        int *s_bad = reinterpret_cast<int *>(sT + 32 * PANEL_LDT);     // [0] bad pivot, [1] quit, [2] see below
        if (tid < 4) s_bad[tid] = 0;                                  // [2] step whose operands may be loaded
        __syncthreads();                                              // all 288 threads
        if (tid >= 256) {
            // -------- communication warp --------
            const int lane = tid - 256;
            for (long long kb = 0; kb < nblk; ++kb) {
                const bool stamp = dbg && kb == nblk / 2 && lane == 0;
                const long long j0 = kb * SOLVE_NB;
                const int nb = (int)((n - j0 < SOLVE_NB) ? n - j0 : SOLVE_NB);
                const long long r0 = j0 + nb;
                long long mm = n - r0;
                if (mm > bw) mm = bw;
                const int m = (int)mm;
                if (stamp) dbg[32] = clock64();
                // the two blocks this step reads were last written by the workers during step kb-1
                if (kb > 0) {
                    long long pm = n - j0;                            // window of step kb-1
                    if (pm > bw) pm = bw;
                    if (pm > SYRK_TILE) {
                        if (lane == 0) {
                            spl_df_spin<200>(f_t10, (unsigned)kb, fail);
                            spl_df_spin<200>(f_t11, (unsigned)kb, fail);
                        }
                        __syncwarp();
                    }
                }
                if (stamp) dbg[33] = clock64();
                if (lane == 0) *reinterpret_cast<volatile int *>(s_bad + 2) = (int)kb + 1;    // seen by the mid-chol check
                DF_BAR_ARRIVE(DF_NB_OPER);
                if (stamp) dbg[34] = clock64();
                DF_BAR_SYNC(DF_NB_LINV);                              // the compute warps have stored L11^-1
                if (stamp) dbg[35] = clock64();
                if (lane == 0) {
                    if (s_bad[1]) *reinterpret_cast<volatile int *>(fail) = 1;
                    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(f_linv), "r"((unsigned)(kb + 1)) : "memory");
                }
                if (s_bad[1]) return;                                 // the workers leave after B1
                if (stamp) dbg[36] = clock64();
                if (m <= 0) continue;
                DF_BAR_SYNC(DF_NB_L10);                               // L[k+1,k] stored, and in sA (k-major)
                if (stamp) dbg[37] = clock64();
                if (lane == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(f_l10), "r"((unsigned)(kb + 1)) : "memory");
                {
                    // this CTA's share of g2 -= L21 y1 for the next block: rows 2 lane, 2 lane + 1
                    const int r = 2 * lane;
                    double p[4][2];
#pragma unroll
                    for (int q = 0; q < 4; ++q) p[q][0] = p[q][1] = 0.0;
#pragma unroll 4
                    for (int c = 0; c < 64; c += 4) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const double2 v = *reinterpret_cast<const double2 *>(sA + (c + q) * TILE_LD + r);
                            const double y = s_g[c + q];
                            p[q][0] = fma(v.x, y, p[q][0]);
                            p[q][1] = fma(v.y, y, p[q][1]);
                        }
                    }
                    double *gn = s_gn + ((kb + 1) & 1) * 64;
                    gn[r] = -((p[0][0] + p[1][0]) + (p[2][0] + p[3][0]));
                    gn[r + 1] = -((p[0][1] + p[1][1]) + (p[2][1] + p[3][1]));
                }
                if (stamp) dbg[38] = clock64();
            }
            return;
        }
        // -------- compute warps --------
        const int ri = tid >> 2, rc = tid & 3;
        if (tid < 128) s_gn[tid] = 0.0;
        // block (0,0) -> sC
        spl_tile_load16(sC, AB, lda, (int)(n < 64 ? n : 64), (int)(n < 64 ? n : 64), tid);
        spl_cp_async_wait_all();
        SPL_SYNC256();
        for (long long kb = 0; kb < nblk; ++kb) {
            const bool stamp = dbg && kb == nblk / 2;
            const long long j0 = kb * SOLVE_NB;
            const int nb = (int)((n - j0 < SOLVE_NB) ? n - j0 : SOLVE_NB);
            const long long r0 = j0 + nb;
            long long mm = n - r0;
            if (mm > bw) mm = bw;
            const int m = (int)mm;
            DF_STAMP(0);
            DF_STAMP_NS(8);
            double u[16];
#pragma unroll
            for (int kk = 0; kk < 16; ++kk) {
                const int k = 4 * kk + rc;
                double v = (ri == k) ? 1.0 : 0.0;                 // identity padding when nb < 64
                if (ri < nb && k < nb && k <= ri) v = sC[k * TILE_LD + ri];
                u[kk] = v;
            }
            // the workers' shares of g1 are complete: they precede the flags the communication warp acquired one step ago
            const double g1r = (tid < nb) ? __ldcg(g + j0 + tid) : 0.0;
            // operands of this step (A21 tile row 0 -> sA, the next diagonal block -> sC): issued in the shadow of the
            // (latency-bound) factorization as soon as the communication warp has acquired the workers' flags
            const int nbn = (int)((n - r0 < SOLVE_NB) ? n - r0 : SOLVE_NB);
            bool issued = false;
            spl_chol64<0, 56>(u, s_col, s_rd, s_bad, tid);
            if (tid == 0) s_bad[3] = *reinterpret_cast<volatile int *>(s_bad + 2) >= (int)kb + 1;
            SPL_SYNC256();                                        // one thread decides for all
            if (s_bad[3]) {
                DF_BAR_SYNC(DF_NB_OPER);                          // (does not wait: the flag is written before the arrive)
                if (m > 0) {
                    spl_tile_load16(sA, AB + r0 + j0 * lda, lda, m, nb, tid);
                    spl_tile_load16(sC, AB + r0 + r0 * lda, lda, nbn, nbn, tid);
                }
                issued = true;
            }
            spl_chol64<56, 64>(u, s_col, s_rd, s_bad, tid);
            DF_STAMP(1);
            if (s_bad[0]) {
                if (tid == 0) s_bad[1] = 1;
                if (!issued) DF_BAR_SYNC(DF_NB_OPER);             // (the communication warp arrives there first)
                spl_cp_async_wait_all();
                DF_BAR_ARRIVE(DF_NB_LINV);
                return;
            }
            if (!issued) {
                DF_BAR_SYNC(DF_NB_OPER);
                if (m > 0) {
                    spl_tile_load16(sA, AB + r0 + j0 * lda, lda, m, nb, tid);
                    spl_tile_load16(sC, AB + r0 + r0 * lda, lda, nbn, nbn, tid);
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
            spl_linv64(u, s_rd, sX, sT, tid);
            DF_STAMP(2);
            {
                double *lb = linv + kb * 4096;                    // (fire and forget: the communication warp fences)
                for (int e = 2 * tid; e < 4096; e += 2 * PANEL_THREADS)
                    *reinterpret_cast<double2 *>(lb + e) =
                        *reinterpret_cast<const double2 *>(sX + (e >> 6) * TILE_LD + (e & 63));
            }
            DF_BAR_ARRIVE(DF_NB_LINV);
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            SPL_SYNC256();
            DF_STAMP(3);
            if (tid < 64) {
                double *gn = s_gn + (kb & 1) * 64;
                s_g[tid] = g1r + gn[tid];
            }
            SPL_SYNC256();
            const double y1c = spl_y1_64(sX, s_g, tid);
            SPL_SYNC256();
            if (rc == 0) {
                s_g[ri] = y1c;
                if (ri < nb) ysol[j0 + ri] = y1c;                 // visible with L10 (or, in the last step, at the kernel's end)
            }
            DF_STAMP(4);
            if (m <= 0) continue;
            // ---- L[k+1,k] = A21 tile row 0 * Linv^T (spl_l21_mma), left in sA k-major ----
            {
                const int warp = tid >> 5, lane = tid & 31;
                const int gq = lane >> 2, t4 = lane & 3;
                const int wy = (warp >> 1) * 16, wodd = warp & 1;
                double acc[2][4][2];
                spl_l21_mma(acc, sA, sX, wy, wodd, gq, t4);
                DF_STAMP(40);
                SPL_SYNC256();                                    // everyone is done reading sA (A21)
                DF_STAMP(41);
#pragma unroll
                for (int mi = 0; mi < 2; ++mi)
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                        for (int h = 0; h < 2; ++h)
                            sA[((2 * ni + wodd) * 8 + 2 * t4 + h) * TILE_LD + wy + mi * 8 + gq] = acc[mi][ni][h];
            }
            SPL_SYNC256();
            DF_STAMP(42);
            {
                // L[k+1,k] -> band matrix, from shared memory: a warp stores whole columns (512 contiguous bytes)
                const int r = 2 * (tid & 31);
                double *dst = AB + (r0 + r) + j0 * lda;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int c = (tid >> 5) + 8 * q;
                    if (c < nb) {
                        const double2 v = *reinterpret_cast<const double2 *>(sA + c * TILE_LD + r);
                        if (r + 1 < m) *reinterpret_cast<double2 *>(dst + (long long)c * lda) = v;
                        else if (r < m) dst[(long long)c * lda] = v.x;
                    }
                }
            }
            DF_BAR_ARRIVE(DF_NB_L10);
            DF_STAMP(5);
            // ---- block (k+1,k+1) -= L10 L10^T in shared memory, lower triangle only: 36 of the 64 8 x 8 blocks.  Block
            // rows ib = p and 7 - p hold 9 blocks together; warps 2p, 2p + 1 take 5 and 4 of them.  Transposed product
            // as in spl_tile_mma_store: the MMA's rows are the block's columns. ----
            {
                const int warp = tid >> 5, lane = tid & 31, gq = lane >> 2, t4 = lane & 3;
                const int p = warp >> 1, q0 = (warp & 1) ? 5 : 0, nq = (warp & 1) ? 4 : 5;
                double acc[5][2];
                int ibq[5], jbq[5];
#pragma unroll
                for (int q = 0; q < 5; ++q) {
                    const int qq = q0 + q;
                    ibq[q] = (qq <= p) ? p : 7 - p;
                    jbq[q] = (qq <= p) ? qq : qq - p - 1;
                    if (q < nq) {
                        const double2 v =
                            *reinterpret_cast<const double2 *>(sC + (jbq[q] * 8 + gq) * TILE_LD + ibq[q] * 8 + 2 * t4);
                        acc[q][0] = v.x;
                        acc[q][1] = v.y;
                    }
                }
#pragma unroll 4
                for (int k0 = 0; k0 < 64; k0 += 4) {
                    const double *row = sA + (k0 + t4) * TILE_LD + gq;
                    const double b_lo = row[p * 8], b_hi = row[(7 - p) * 8];
#pragma unroll
                    for (int q = 0; q < 5; ++q)
                        if (q < nq) {
                            const double a = -row[jbq[q] * 8];
                            spl_dmma_8x8x4(acc[q][0], acc[q][1], a, (ibq[q] == p) ? b_lo : b_hi);
                        }
                }
#pragma unroll
                for (int q = 0; q < 5; ++q)
                    if (q < nq)
                        *reinterpret_cast<double2 *>(sC + (jbq[q] * 8 + gq) * TILE_LD + ibq[q] * 8 + 2 * t4) =
                            make_double2(acc[q][0], acc[q][1]);
            }
            SPL_SYNC256();
            DF_STAMP(6);
        }
        return;
    }

    // ================================ workers ================================
    if (tid >= 256) return;                                       // only the diagonal CTA has a ninth warp
    const unsigned nwork = (unsigned)(G - 1);
    unsigned tgt1 = 0, tgt2 = 0;
    const bool panel_worker = cta < Tmax;
    const int NH = G - Tmax, me = cta - Tmax;                     // helpers
    double *sA = s_df, *sX = s_df + 64 * TILE_LD;
    double *s_g = s_df + 4 * 64 * TILE_LD;                        // behind the helpers' two operand buffers
    int *s_flag = reinterpret_cast<int *>(s_g + 64);
    for (long long kb = 0; kb < nblk; ++kb) {
        const bool stamp = dbg && kb == nblk / 2 && (cta == 1 || cta == Tmax);
        const long long j0 = kb * SOLVE_NB;
        const int nb = (int)((n - j0 < SOLVE_NB) ? n - j0 : SOLVE_NB);
        const long long r0 = j0 + nb;
        long long mm = n - r0;
        if (mm > bw) mm = bw;
        const int m = (int)mm;
        const int T = (m + SYRK_TILE - 1) / SYRK_TILE;
        const int ntiles = (T > 1) ? (T - 1) * T / 2 : 0;
        const int npw = 0;              // rest tiles the panel workers take from the end of the list (measured: none --
                                        // a panel worker that is late for LINV delays B1 for everybody)
        const int nth = ntiles - npw;                             // the helpers' list
        const bool active = panel_worker && cta < T;
        const int sbase = (cta == 1) ? 16 : 24;
        DF_STAMP(sbase + 0);
        DF_STAMP_NS(sbase + 6);
        bool b_issued = false;
        if (active) {
            // ---- tile row `cta` of the panel ----
            spl_tile_load16(sA, AB + (r0 + (long long)cta * 64) + j0 * lda, lda, m - cta * 64, nb, tid);
            asm volatile("cp.async.commit_group;" ::: "memory");
            spl_df_wait(f_linv, (unsigned)(kb + 1), fail);
            DF_STAMP(sbase + 1);
            {
                const double *lb = linv + kb * 4096;
                for (int e = 2 * tid; e < 4096; e += 2 * PANEL_THREADS)
                    spl_cp_async16(sX + (e >> 6) * TILE_LD + (e & 63), lb + e);
            }
            spl_cp_async_wait_all();
            SPL_SYNC256();
            spl_l21_gemm<false>(AB, lda, j0, nb, m, r0, cta * 64, g, sA, sX, s_g, true, tid);
            // L[k+1,k] is usually there by now: start the column-0 tile's B operand before the barrier
            if (tid == 0) *s_flag = spl_ld_acquire(f_l10) >= (unsigned)(kb + 1);
            SPL_SYNC256();
            if (*s_flag) {
                spl_tile_issue<true>(AB, lda, r0, j0, nb, m, cta, 0, s_df);
                b_issued = true;
            }
            DF_STAMP(sbase + 2);
        }
        if (dbg && kb == nblk / 2 && tid == 0) {                  // arrival of every worker at B1, device-wide timer
            unsigned long long t_;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));
            dbg[64 + cta] = (long long)t_;
        }
        spl_df_barrier(f_b1, tgt1, nwork, fail);
        DF_STAMP(sbase + 3);
        DF_STAMP_NS(sbase + 7);
        if (*reinterpret_cast<volatile int *>(fail)) {            // uniform: written before the flag B1 chains from
            spl_cp_async_wait_all();
            return;
        }
        if (active) {
            // ---- column-0 tile of the same row: A operand = the L21 tile left in sA, B = L[k+1,k] ----
            if (!b_issued) {
                spl_df_wait(f_l10, (unsigned)(kb + 1), fail);
                spl_tile_issue<true>(AB, lda, r0, j0, nb, m, cta, 0, s_df);
            }
            // g2 -= L21 y1 for this tile row (y1 is published with L[k+1,k]), under the B operand's flight
            if (tid < 64) s_g[tid] = (tid < nb) ? __ldcg(ysol + j0 + tid) : 0.0;
            SPL_SYNC256();
            spl_g_update(g, r0, cta * 64, m, sA, s_g, tid);
            spl_tile_finish<0>(AB, lda, r0, m, cta, 0, s_df);
            if (cta == 1) spl_df_post(f_t10, (unsigned)(kb + 1));
            DF_STAMP(sbase + 4);
        }
        if (panel_worker) {
            if (active) spl_df_barrier(f_b2, tgt2, (unsigned)(T - 1), fail);
            else if (T > 1) tgt2 += (unsigned)(T - 1);
            DF_STAMP(sbase + 5);
            if (active && cta - 1 < npw) {
                // one rest tile from the end of the list while the diagonal CTA factors the next block
                int ti, tj;
                spl_rest_tile(ntiles - 1 - (cta - 1), ti, tj);
                spl_tile256<false>(AB, lda, r0, j0, nb, m, ti, tj, s_df);
                SPL_SYNC256();
            }
        } else if (me < nth) {
            // ---- rest tiles of update kb: me, me + NH, .. with the next tile's operands and C tile in flight; the tiles
            // of the last, partial round are split in row halves when that gives everybody half a tile instead of some a
            // whole one (the barrier B1 waits for the longest list) ----
            const int base = nth / NH, rem = nth - base * NH;
            const bool halves = base >= 1 && 2 * rem <= NH;
            const int nfull = base + ((!halves && me < rem) ? 1 : 0);
            const int cnt = nfull + ((halves && me < 2 * rem) ? 1 : 0);
            auto item = [&](const int idx, int &ti_, int &tj_, int &half_) {
                if (idx < nfull) {
                    spl_rest_tile(me + NH * idx, ti_, tj_);
                    half_ = -1;
                } else {
                    spl_rest_tile(base * NH + (me >> 1), ti_, tj_);
                    half_ = me & 1;
                }
            };
            int cur = 0, ti, tj, half;
            double accn[2][4][2];
            item(0, ti, tj, half);
            spl_tile_issue<false>(AB, lda, r0, j0, nb, m, ti, tj, s_df, half);
            if (half < 0) spl_tile_cload<2>(accn, AB, lda, r0, m, ti, tj);
            else spl_tile_cload<1>(accn, AB, lda, r0, m, ti, tj, half);
            for (int idx = 0; idx < cnt; ++idx) {
                double *bcur = s_df + cur * (2 * 64 * TILE_LD);
                double acc[2][4][2];
#pragma unroll
                for (int mj = 0; mj < 2; ++mj)
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) {
                        acc[mj][ni][0] = accn[mj][ni][0];
                        acc[mj][ni][1] = accn[mj][ni][1];
                    }
                if (idx + 1 < cnt) {
                    int tin, tjn, halfn;
                    item(idx + 1, tin, tjn, halfn);
                    spl_tile_issue<false>(AB, lda, r0, j0, nb, m, tin, tjn, s_df + (cur ^ 1) * (2 * 64 * TILE_LD), halfn);
                    if (halfn < 0) spl_tile_cload<2>(accn, AB, lda, r0, m, tin, tjn);
                    else spl_tile_cload<1>(accn, AB, lda, r0, m, tin, tjn, halfn);
                    if (half < 0) spl_tile_mma_store<1, 2>(acc, AB, lda, r0, m, ti, tj, bcur);
                    else spl_tile_mma_store<1, 1>(acc, AB, lda, r0, m, ti, tj, bcur, half);
                    ti = tin;
                    tj = tjn;
                    half = halfn;
                } else {
                    if (half < 0) spl_tile_mma_store<0, 2>(acc, AB, lda, r0, m, ti, tj, bcur);
                    else spl_tile_mma_store<0, 1>(acc, AB, lda, r0, m, ti, tj, bcur, half);
                }
                if (me == 0 && idx == 0) spl_df_post(f_t11, (unsigned)(kb + 1));      // tile (1,1), always whole
                else SPL_SYNC256();                                // buffer `cur` is refilled by the next issue
                if (idx == 0) DF_STAMP(sbase + 4);
                cur ^= 1;
            }
            DF_STAMP(sbase + 5);
        }
    }
}

// ------------------------------------------------------------------------------------------
// back-substitution L^T c = y, block by block from the end, using the stored block inverses
// ------------------------------------------------------------------------------------------
#define BACK_THREADS 128
__global__ void __launch_bounds__(BACK_THREADS)
spl_backsolve_kernel(const double *__restrict__ AB, long long lda, long long j0, int nb, int bw,
                     const double *__restrict__ linv_blk, double *__restrict__ ysol,
                     double *__restrict__ csol, const int *__restrict__ fail) {
    __shared__ double s_li[64 * 65];
    __shared__ double s_y[64];
    __shared__ double s_c[64];
    const int t = threadIdx.x;
    if (*fail) return;
    // the column this thread eliminates from, prefetched while the block solve runs
    const long long jlo = (j0 - bw > 0) ? j0 - bw : 0;
    const long long j = jlo + (long long)blockIdx.x * BACK_THREADS + t;
    double colv[64];
    if (j < j0) {
        const double *col = AB + j0 + j * lda;     // rows j0.. of column j, contiguous
#pragma unroll
        for (int i = 0; i < 64; ++i) colv[i] = (i < nb) ? col[i] : 0.0;
    }
    // stage L11^-1 (row-major [r][c]) and y_k
#pragma unroll
    for (int e = 0; e < 32; ++e) {
        const int idx = t + e * BACK_THREADS;
        s_li[(idx >> 6) * 65 + (idx & 63)] = linv_blk[idx];
    }
    if (t < 64) s_y[t] = (t < nb) ? ysol[j0 + t] : 0.0;
    __syncthreads();
    // c_k = L11^-T y_k:  c[i] = sum_{r >= i} Linv[r][i] y[r]
    if (t < 64) {
        double c0 = 0.0, c1 = 0.0;
#pragma unroll
        for (int r = 0; r < 64; r += 2) {
            c0 = fma(s_li[r * 65 + t], s_y[r], c0);
            c1 = fma(s_li[(r + 1) * 65 + t], s_y[r + 1], c1);
        }
        const double c = c0 + c1;
        s_c[t] = c;
        if (blockIdx.x == 0 && t < nb) csol[j0 + t] = c;
    }
    __syncthreads();
    // eliminate c_k from the bw preceding unknowns: y[j] -= sum_i L[i][j] c[i], i in the block
    if (j < j0) {
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int i = 0; i < 64; i += 2) {
            s0 = fma(colv[i], s_c[i], s0);
            s1 = fma(colv[i + 1], s_c[i + 1], s1);
        }
        ysol[j] -= (s0 + s1);
    }
}

// ------------------------------------------------------------------------------------------
// persistent back-substitution: the whole block loop in ONE cooperative kernel (ceil(bw / 256) CTAs), one grid
// barrier per 64-column block instead of one kernel launch (216 launches of 5.8 us at cfg3).  The next block's
// inverse (cp.async, double-buffered) and every thread's next column of L (registers) are fetched before the barrier
// they will be needed after: L and the block inverses are final, only y changes between the steps, and y is
// read with ld.global.cg (other CTAs wrote it).
// ------------------------------------------------------------------------------------------
#define BACKP_THREADS 256
#define BACKP_NC 8                                // columns per warp and step: grid = ceil((bw + 64) / (8 warps x 8))
#define BACKP_LBP 66                              // pitch of the staged L[k,k-1] block: 16-byte pieces, 2-way conflicts at most
#define BACKP_SMEM_DOUBLES (2 * 2 * 4096 + 2 * 64 * BACKP_LBP + 256)
// Two blocks per grid barrier: every CTA forms c_k = L11(k)^-T y_k, then y'_{k-1} = y_{k-1} - L[k,k-1]^T c_k and
// c_{k-1} = L11(k-1)^-T y'_{k-1} itself (the 64 x 64 block L[k,k-1] rides along with the two inverses), and
// eliminates BOTH from its columns of the bw columns in front of block k-1.  The barrier, the y round trip and the
// reductions are paid once per 128 columns: 216 x 3.6 us -> 108 x 4.2 us at cfg3.
__global__ void __launch_bounds__(BACKP_THREADS, 1)
spl_backsolve_persistent_kernel(const double *__restrict__ AB, long long lda, long long n, int bw,
                                const double *__restrict__ linv, double *ysol, double *__restrict__ csol,
                                const int *__restrict__ fail, unsigned *bar) {
    extern __shared__ __align__(16) double s_bk[];
    double *s_li = s_bk;                        // 2 buffers x {top, bottom} x 64 x 64  block inverses, row-major [r][c]
    double *s_lb = s_bk + 4 * 4096;             // 2 buffers x 64 x LBP  L[k,k-1], [c][r]: c = column in block k-1, r = row in block k
    double *s_y = s_lb + 2 * 64 * BACKP_LBP;    // 128: y_k | y_{k-1}
    double *s_c = s_y + 128;                    // 128: c_k | c_{k-1}
    const int t = threadIdx.x, lane = t & 31;
    const unsigned G = gridDim.x;
    const int gw = (int)blockIdx.x * (BACKP_THREADS / 32) + (t >> 5), nw = (int)G * (BACKP_THREADS / 32);
    unsigned target = 0;
    if (*fail) return;                          // uniform across the grid
    const long long nblk = (n + SOLVE_NB - 1) / SOLVE_NB;
    // step with top block kb: pair (kb, kb-1) when kb >= 1, else block 0 alone.  jt / jb: first column of the top / of the
    // lowest block of the step; the step eliminates from the columns [max(0, jb - bw), jb).
    double colr[BACKP_NC][4];                   // rows l, l+32 of the lowest block | rows l, l+32 of the top block (pairs)
    auto fetch = [&](long long kb, int buf) {
        const bool pair = kb >= 1;
        const long long jt = kb * SOLVE_NB, jb = pair ? jt - SOLVE_NB : jt;
        const int nbt = (int)((n - jt < SOLVE_NB) ? n - jt : SOLVE_NB);
        {
            const double *src = linv + kb * 4096;
            double *dst = s_li + buf * 8192;
            for (int e = 2 * t; e < 4096; e += 2 * BACKP_THREADS) spl_cp_async16(dst + e, src + e);
            if (pair) {
                const double *src2 = linv + (kb - 1) * 4096;
                for (int e = 2 * t; e < 4096; e += 2 * BACKP_THREADS) spl_cp_async16(dst + 4096 + e, src2 + e);
                // L[k,k-1], column by column (rows contiguous) in 16-byte pieces; outside the band -- half bandwidth
                // < 127 -- the address would run into the next column, so those entries are zeros written here
                double *lb = s_lb + buf * (64 * BACKP_LBP);
                for (int e = t; e < 2048; e += BACKP_THREADS) {
                    const int c = e >> 5, r = 2 * (e & 31);
                    double *dst = lb + c * BACKP_LBP + r;
                    const double *src = AB + (jt + r) + (jb + c) * lda;
                    const bool ok0 = r < nbt && SOLVE_NB + r - c <= bw;
                    const bool ok1 = r + 1 < nbt && SOLVE_NB + r + 1 - c <= bw;
                    if (ok0 && ok1) {
                        spl_cp_async16(dst, src);
                    } else {
                        if (ok0) spl_cp_async8(dst, src);
                        else dst[0] = 0.0;
                        dst[1] = 0.0;
                    }
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        const long long jlo = (jb - bw > 0) ? jb - bw : 0;
#pragma unroll
        for (int q = 0; q < BACKP_NC; ++q) {
            const long long j = jlo + gw + (long long)q * nw;
            colr[q][0] = colr[q][1] = colr[q][2] = colr[q][3] = 0.0;
            if (j < jb) {
                const double *col = AB + jb + j * lda;                // rows of the lowest block: always inside the band
                const int nbb = pair ? SOLVE_NB : nbt;
                if (lane < nbb) colr[q][0] = col[lane];
                if (lane + 32 < nbb) colr[q][1] = col[lane + 32];
                if (pair && j >= jt - bw) {                           // rows of the top block, where the band reaches them
                    if (lane < nbt) colr[q][2] = col[64 + lane];
                    if (lane + 32 < nbt) colr[q][3] = col[64 + lane + 32];
                }
            }
        }
    };
    // c[i] = sum_r Linv[r][i] y[r]: thread (i, part) sums r = part, part + 4, ..; every thread of the row returns it
    auto matvec_t = [&](const double *li, const double *y) {
        const int i = t >> 2, part = t & 3;
        double c0 = 0.0, c1 = 0.0;
#pragma unroll
        for (int q = 0; q < 16; q += 2) {
            c0 = fma(li[(part + 4 * q) * 64 + i], y[part + 4 * q], c0);
            c1 = fma(li[(part + 4 * q + 4) * 64 + i], y[part + 4 * q + 4], c1);
        }
        double c = c0 + c1;
        c += __shfl_xor_sync(0xffffffffu, c, 1);
        c += __shfl_xor_sync(0xffffffffu, c, 2);
        return c;
    };
    fetch(nblk - 1, 0);
    int buf = 0;
    for (long long kb = nblk - 1; kb >= 0;) {
        const bool pair = kb >= 1;
        const long long jt = kb * SOLVE_NB, jb = pair ? jt - SOLVE_NB : jt;
        const int nbt = (int)((n - jt < SOLVE_NB) ? n - jt : SOLVE_NB);
        const long long jlo = (jb - bw > 0) ? jb - bw : 0;
        const double *li = s_li + buf * 8192;
        if (t < 64) s_y[t] = (t < nbt) ? __ldcg(ysol + jt + t) : 0.0;
        else if (t < 128 && pair) s_y[t] = __ldcg(ysol + jb + (t - 64));
        // the entries this warp will update, fetched now (other CTAs wrote them before the barrier)
        double yold = 0.0;
        if (lane < BACKP_NC) {
            const long long j = jlo + gw + (long long)lane * nw;
            if (j < jb) yold = __ldcg(ysol + j);
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        {
            const double c = matvec_t(li, s_y);                    // c_k
            const int i = t >> 2;
            if ((t & 3) == 0) {
                s_c[i] = c;
                if (blockIdx.x == 0 && i < nbt) csol[jt + i] = c;
            }
        }
        __syncthreads();
        if (pair) {
            // (L[k,k-1]^T c_k)[column i of block k-1]: thread (i, part) sums the rows part, part + 4, ..
            const int i = t >> 2, part = t & 3;
            double tc;
            {
                const double *lcol = s_lb + buf * (64 * BACKP_LBP) + i * BACKP_LBP;
                double c0 = 0.0, c1 = 0.0;
#pragma unroll
                for (int q = 0; q < 16; q += 2) {
                    c0 = fma(lcol[part + 4 * q], s_c[part + 4 * q], c0);
                    c1 = fma(lcol[part + 4 * q + 4], s_c[part + 4 * q + 4], c1);
                }
                tc = c0 + c1;
                tc += __shfl_xor_sync(0xffffffffu, tc, 1);
                tc += __shfl_xor_sync(0xffffffffu, tc, 2);
            }
            if ((t & 3) == 0) s_y[64 + i] -= tc;                   // (nobody reads y_{k-1} in this phase)
            __syncthreads();
            const double c = matvec_t(li + 4096, s_y + 64);        // c_{k-1}
            if ((t & 3) == 0) {
                s_c[64 + i] = c;
                if (blockIdx.x == 0) csol[jb + i] = c;
            }
            __syncthreads();
        }
        // eliminate from the bw columns in front of the lowest block: y[j] -= sum_i L[i][j] c[i]
        {
            const double *cl = pair ? s_c + 64 : s_c;              // c of the lowest block
            const double ca = cl[lane], cb = cl[lane + 32];
            const double ta = pair ? s_c[lane] : 0.0, tb = pair ? s_c[lane + 32] : 0.0;
            double mine = 0.0;
#pragma unroll
            for (int q = 0; q < BACKP_NC; ++q) {
                double v = fma(colr[q][0], ca, colr[q][1] * cb);
                v = fma(colr[q][2], ta, fma(colr[q][3], tb, v));
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == q) mine = v;
            }
            if (lane < BACKP_NC) {
                const long long j = jlo + gw + (long long)lane * nw;
                if (j < jb) ysol[j] = yold - mine;
            }
        }
        kb -= pair ? 2 : 1;
        if (kb >= 0) {
            // grid barrier with the next step's prefetch between the arrive and the wait: issued in front of the
            // release, the fence of the arrive would wait for the 96 KB in flight
            buf ^= 1;
            __syncthreads();
            if (t == 0) {
                target += G;
                asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(bar) : "memory");
            }
            fetch(kb, buf);
            if (t == 0) {
                unsigned v;
                do {
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
                } while (v < target);
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------
// persistent forward substitution L y = g against the STORED factor (refinement steps, capi.cu: the
// factorisation of G is reused, only the right-hand side is new).  Mirror image of the kernel above: per 64-column
// block every CTA forms y_k = L11^-1 g_k from the stored block inverse, then warp pairs eliminate y_k from the (<= bw)
// rows below -- lane = row, the two warps of a pair take 32 columns each (a column's rows are contiguous: coalesced
// 256-byte loads, prefetched before the barrier because L is final) and are combined in a fixed order, so the
// result is deterministic.  One grid barrier per block.
// ------------------------------------------------------------------------------------------
#define FWDP_THREADS 256
#define FWDP_LD 65
__global__ void __launch_bounds__(FWDP_THREADS, 1)
spl_forwardsolve_persistent_kernel(const double *__restrict__ AB, long long lda, long long n, int bw,
                                   const double *__restrict__ linv, double *g, double *__restrict__ ysol,
                                   const int *__restrict__ fail, unsigned *bar) {
    extern __shared__ __align__(16) double s_fw[];
    double *s_li = s_fw;                        // 2 x 64 x FWDP_LD  block inverse, row-major [r][c], padded
    double *s_g = s_fw + 2 * 64 * FWDP_LD;      // 64  g_k
    double *s_y = s_g + 64;                     // 64  y_k
    double *s_part = s_y + 64;                  // 8 x 32 partial row sums of the warps
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const unsigned G = gridDim.x;
    const int gw = (int)blockIdx.x * (FWDP_THREADS / 32) + warp;
    const int pair = gw >> 1, hc = gw & 1;      // rows r0 + 32 pair + lane, columns 32 hc .. 32 hc + 31 of the block
    unsigned target = 0;
    if (*fail) return;                          // uniform across the grid
    const long long nblk = (n + SOLVE_NB - 1) / SOLVE_NB;
    auto fetch_inv = [&](long long kb, int buf) {
        const double *src = linv + kb * 4096;
        double *dst = s_li + buf * 64 * FWDP_LD;
        for (int e = t; e < 4096; e += FWDP_THREADS) spl_cp_async8(dst + (e >> 6) * FWDP_LD + (e & 63), src + e);
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    double lreg[32];
    auto fetch_rows = [&](long long kb) {
        const long long j0 = kb * SOLVE_NB;
        const int nb = (int)((n - j0 < SOLVE_NB) ? n - j0 : SOLVE_NB);
        const long long r0 = j0 + nb;
        long long mm = n - r0;
        if (mm > bw) mm = bw;
        const long long rl = (long long)pair * 32 + lane;
        const bool ok = rl < mm;
        const double *src = AB + (r0 + rl) + (j0 + hc * 32) * lda;
#pragma unroll
        for (int c = 0; c < 32; ++c) lreg[c] = (ok && hc * 32 + c < nb) ? src[(long long)c * lda] : 0.0;
    };
    fetch_inv(0, 0);
    fetch_rows(0);
    for (long long kb = 0; kb < nblk; ++kb) {
        const long long j0 = kb * SOLVE_NB;
        const int nb = (int)((n - j0 < SOLVE_NB) ? n - j0 : SOLVE_NB);
        const long long r0 = j0 + nb;
        long long mm = n - r0;
        if (mm > bw) mm = bw;
        const double *li = s_li + (kb & 1) * 64 * FWDP_LD;
        if (t < 64) s_g[t] = (t < nb) ? __ldcg(g + j0 + t) : 0.0;
        const long long rl = (long long)pair * 32 + lane;
        double gold = 0.0;
        if (hc == 0 && rl < mm) gold = __ldcg(g + r0 + rl);
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        // y_k = L11^-1 g_k: thread (r, part) sums c = part, part + 4, ..
        {
            const int r = t >> 2, part = t & 3;
            double y0 = 0.0, y1 = 0.0;
#pragma unroll
            for (int q = 0; q < 16; q += 2) {
                y0 = fma(li[r * FWDP_LD + part + 4 * q], s_g[part + 4 * q], y0);
                y1 = fma(li[r * FWDP_LD + part + 4 * q + 4], s_g[part + 4 * q + 4], y1);
            }
            double y = y0 + y1;
            y += __shfl_xor_sync(0xffffffffu, y, 1);
            y += __shfl_xor_sync(0xffffffffu, y, 2);
            if (part == 0) {
                s_y[r] = y;
                if (blockIdx.x == 0 && r < nb) ysol[j0 + r] = y;
            }
        }
        __syncthreads();
        // g[i] -= sum_c L[i][j0 + c] y[c] for the rows below the block
        {
            double p0 = 0.0, p1 = 0.0;
#pragma unroll
            for (int c = 0; c < 32; c += 2) {
                p0 = fma(lreg[c], s_y[hc * 32 + c], p0);
                p1 = fma(lreg[c + 1], s_y[hc * 32 + c + 1], p1);
            }
            s_part[warp * 32 + lane] = p0 + p1;
        }
        __syncthreads();
        if (hc == 0 && rl < mm) g[r0 + rl] = gold - (s_part[warp * 32 + lane] + s_part[(warp + 1) * 32 + lane]);
        if (kb + 1 < nblk) {
            fetch_inv(kb + 1, (int)((kb + 1) & 1));
            fetch_rows(kb + 1);
            spl_grid_barrier(bar, target, G);
        }
    }
}

// ------------------------------------------------------------------------------------------
// host driver
// ------------------------------------------------------------------------------------------
// even: columns of the band matrix then start at 16-byte boundaries, which the 16-byte cp.async of the operand tiles
// and the 128-bit accesses of the update tiles need
long long spl_band_lda(int bw) { return ((long long)bw + SOLVE_NB + 1) & ~1LL; }

int spl_half_bandwidth(const GridParams &gp) {
    long long b = 0, stride = 1;
    for (int d = 0; d < gp.ndim; ++d) {
        b += 3 * stride;
        stride *= gp.nodes[d];
    }
    if (b > gp.ncol - 1) b = gp.ncol - 1;
    return (int)b;
}

// Doubles of the band matrix, i.e. the offset of the workspace behind it.  Element (i, j) lives at i + j*lda, so the
// last one, (n-1, n-1), is at (n-1)*(lda+1); even, so that the workspace stays 16-byte aligned.
long long spl_band_elems(const GridParams &gp) {
    const long long lda = spl_band_lda(spl_half_bandwidth(gp));
    return (gp.ncol * (lda + 1) + 64 + 1) & ~1LL;
}

// Workspace (doubles) next to the band matrix, at spl_band_elems: block inverses (64*64 per panel) + ysol (n) + csol (n).
long long spl_solve_workspace(const GridParams &gp) {
    const long long nblk = (gp.ncol + SOLVE_NB - 1) / SOLVE_NB;
    return nblk * 64 * 64 + 2 * (gp.ncol + 64);
}

// AB must hold ncol*(lda+1) doubles and be zero-filled on entry.  g enters as the right-hand side
// (destroyed); the solution is left in d_work + nblk*4096 + (ncol+64)  (returned through *d_coef_out).
// The factorisation is ~650 small dependent launches with cross-stream events: issued from the host it
// is bound by the CPU's launch rate (45 us per panel), so both loops are captured once per handle into
// CUDA graphs and replayed.
struct SolveGraphs {
    cudaGraphExec_t factor = nullptr, back = nullptr;
    const double *key_AB = nullptr, *key_g = nullptr;
    long long n = 0;
    int bw = 0;
    long long nfactor = 0, nback = 0;     // kernel nodes
    bool persistent = false;              // the factor loop is the cooperative kernel: no factor graph
    int kblock = 0;                       // panels per outer block the factor graph was captured with
};

void spl_solve_cache_free(void *cache) {
    SolveGraphs *sg = static_cast<SolveGraphs *>(cache);
    if (!sg) return;
    if (sg->factor) cudaGraphExecDestroy(sg->factor);
    if (sg->back) cudaGraphExecDestroy(sg->back);
    delete sg;
}

// Right-looking factor loop with look-ahead over two streams.  Panel k+1 depends only on the first tile
// column of trailing update k, so
//   st     : panel(k) -> [wait rest(k-1)] -> syrk column 0 (k) -> panel(k+1) ...
//   st_aux : [wait panel(k)] -> syrk rest (k)
// and the rest of update k runs under panel k+1's diagonal-block latency chain.  Ordering on shared tiles:
// rest(k)'s tiles with tj >= 1 are columns 0.. of window k+1, hence the wait before syrk column 0 (k+1);
// rest(k) and rest(k+1) are ordered by st_aux itself.
// SPLPAK_B200_PANELCLK=1: phase clocks of one mid-matrix panel (device buffer handed to that launch only)
static long long *spl_panel_dbg_buffer() {
    static long long *buf = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        if (getenv("SPLPAK_B200_PANELCLK")) {
            if (cudaMalloc((void **)&buf, 512 * sizeof(long long)) != cudaSuccess) buf = nullptr;
            else cudaMemset(buf, 0, 512 * sizeof(long long));
        }
    }
    return buf;
}

static cudaError_t enqueue_factor(long long n, int bw, long long lda, double *d_AB, double *d_g, double *d_ysol,
                                  double *d_linv, int *d_fail, cudaStream_t st, cudaStream_t st_aux,
                                  size_t panel_smem, size_t syrk_smem, long long *nlaunch) {
    const long long nblk = (n + SOLVE_NB - 1) / SOLVE_NB;
    const char *syrk_mode = getenv("SPLPAK_B200_SYRK");
    const bool syrk256 = !(syrk_mode && strcmp(syrk_mode, "128") == 0);
    cudaEvent_t ev_panel = nullptr, ev_rest = nullptr;
    cudaError_t e;
    if ((e = cudaEventCreateWithFlags(&ev_panel, cudaEventDisableTiming)) != cudaSuccess) return e;
    if ((e = cudaEventCreateWithFlags(&ev_rest, cudaEventDisableTiming)) != cudaSuccess) return e;
    bool rest_pending = false;
    long long count = 0;
    for (long long kb = 0; kb < nblk && e == cudaSuccess; ++kb) {
        const long long j0 = kb * SOLVE_NB;
        const int nb = (int)((n - j0 < SOLVE_NB) ? n - j0 : SOLVE_NB);
        const long long r0 = j0 + nb;
        long long mm = n - r0;
        if (mm > bw) mm = bw;
        const int m = (int)mm;
        int pblocks = (m + 63) / 64;
        if (pblocks < 1) pblocks = 1;
        spl_panel_kernel<<<pblocks, PANEL_THREADS, panel_smem, st>>>(d_AB, lda, j0, nb, m, d_g, d_ysol,
                                                                     d_linv + kb * 4096, d_fail,
                                                                     kb == nblk / 2 ? spl_panel_dbg_buffer() : nullptr);
        ++count;
        if (m > 0) {
            const int T = (m + SYRK_TILE - 1) / SYRK_TILE;
            if (T > 1) {
                if ((e = cudaEventRecord(ev_panel, st)) != cudaSuccess) break;
                if ((e = cudaStreamWaitEvent(st_aux, ev_panel, 0)) != cudaSuccess) break;
                if (syrk256) spl_syrk256_kernel<<<(T - 1) * T / 2, PANEL_THREADS, syrk_smem, st_aux>>>(d_AB, lda, r0, j0, nb, m, d_fail, 1);
                else spl_syrk_kernel<<<(T - 1) * T / 2, SYRK_THREADS, syrk_smem, st_aux>>>(d_AB, lda, r0, j0, nb, m, d_fail, 1);
                ++count;
            }
            if (rest_pending && (e = cudaStreamWaitEvent(st, ev_rest, 0)) != cudaSuccess) break;   // rest(k-1) done
            rest_pending = false;
            if (syrk256) spl_syrk256_kernel<<<T, PANEL_THREADS, syrk_smem, st>>>(d_AB, lda, r0, j0, nb, m, d_fail, 0);
            else spl_syrk_kernel<<<T, SYRK_THREADS, syrk_smem, st>>>(d_AB, lda, r0, j0, nb, m, d_fail, 0);
            ++count;
            if (T > 1) {
                if ((e = cudaEventRecord(ev_rest, st_aux)) != cudaSuccess) break;
                rest_pending = true;
            }
        }
    }
    if (e == cudaSuccess && rest_pending) e = cudaStreamWaitEvent(st, ev_rest, 0);   // join st_aux
    cudaEventDestroy(ev_panel);
    cudaEventDestroy(ev_rest);
    if (e == cudaSuccess) e = cudaGetLastError();
    *nlaunch = count;
    return e;
}

// Two-level blocked factor loop (see spl_syrk_kblock_kernel): outer blocks of KB panels.
//   st     : [panel(p) -> block-column update(p)] p = 0..np-1 -> [wait rest(k-1)] -> K-blocked update, tile columns
//            of the next block (k) -> next block ...
//   st_aux : [wait the block's last panel] -> K-blocked update, every other tile column (k)
// so the latency chain of the next block's KB panels runs under the bulk of update k, as in enqueue_factor.
static int spl_kblock() {
    const char *s = getenv("SPLPAK_B200_KBLOCK");
    int kb = s ? atoi(s) : KBLOCK_MAX;
    if (kb < 1) kb = 1;
    if (kb > KBLOCK_MAX) kb = KBLOCK_MAX;
    return kb;
}

static cudaError_t enqueue_factor_blocked(long long n, int bw, long long lda, double *d_AB, double *d_g, double *d_ysol,
                                          double *d_linv, int *d_fail, cudaStream_t st, cudaStream_t st_aux,
                                          size_t panel_smem, size_t syrk_smem, int KB, long long *nlaunch) {
    const long long nblk = (n + SOLVE_NB - 1) / SOLVE_NB;
    cudaEvent_t ev_panel = nullptr, ev_rest = nullptr;
    cudaError_t e;
    if ((e = cudaEventCreateWithFlags(&ev_panel, cudaEventDisableTiming)) != cudaSuccess) return e;
    if ((e = cudaEventCreateWithFlags(&ev_rest, cudaEventDisableTiming)) != cudaSuccess) return e;
    bool rest_pending = false;
    long long count = 0;
    for (long long ob = 0; ob < nblk && e == cudaSuccess; ob += KB) {
        const int np = (int)((nblk - ob < KB) ? nblk - ob : KB);
        const long long jb = ob * SOLVE_NB;
        for (int p = 0; p < np; ++p) {
            const long long kb = ob + p;
            const long long j0 = kb * SOLVE_NB;
            const int nb = (int)((n - j0 < SOLVE_NB) ? n - j0 : SOLVE_NB);
            const long long r0 = j0 + nb;
            long long mm = n - r0;
            if (mm > bw) mm = bw;
            const int m = (int)mm;
            int pblocks = (m + 63) / 64;
            if (pblocks < 1) pblocks = 1;
            spl_panel_kernel<<<pblocks, PANEL_THREADS, panel_smem, st>>>(d_AB, lda, j0, nb, m, d_g, d_ysol,
                                                                         d_linv + kb * 4096, d_fail,
                                                                         kb == nblk / 2 ? spl_panel_dbg_buffer() : nullptr);
            ++count;
            const int T = (m + SYRK_TILE - 1) / SYRK_TILE;
            int cols = np - 1 - p;
            if (cols > T) cols = T;
            if (m > 0 && cols > 0) {
                spl_syrk_cols_kernel<<<dim3(T, cols), PANEL_THREADS, syrk_smem, st>>>(d_AB, lda, r0, j0, nb, m, d_fail);
                ++count;
            }
        }
        const long long R0 = jb + (long long)np * SOLVE_NB;
        long long MM = n - R0;
        if (MM > bw) MM = bw;
        if (MM > 0) {
            const int T = (int)((MM + SYRK_TILE - 1) / SYRK_TILE);
            long long next_np = nblk - (ob + np);
            if (next_np > KB) next_np = KB;
            int c0 = (int)next_np;
            if (c0 > T) c0 = T;
            if (c0 < 1) c0 = 1;
            const int TR = T - c0;                                 // tile columns of the rest
            if (TR > 0) {
                if ((e = cudaEventRecord(ev_panel, st)) != cudaSuccess) break;
                if ((e = cudaStreamWaitEvent(st_aux, ev_panel, 0)) != cudaSuccess) break;
                spl_syrk_kblock_kernel<<<TR * (TR + 1) / 2, PANEL_THREADS, syrk_smem, st_aux>>>(d_AB, lda, jb, np, n, bw,
                                                                                                 d_fail, 1, c0);
                ++count;
            }
            if (rest_pending && (e = cudaStreamWaitEvent(st, ev_rest, 0)) != cudaSuccess) break;   // rest(k-1) done
            rest_pending = false;
            spl_syrk_kblock_kernel<<<dim3(T, c0), PANEL_THREADS, syrk_smem, st>>>(d_AB, lda, jb, np, n, bw, d_fail, 0, c0);
            ++count;
            if (TR > 0) {
                if ((e = cudaEventRecord(ev_rest, st_aux)) != cudaSuccess) break;
                rest_pending = true;
            }
        }
    }
    if (e == cudaSuccess && rest_pending) e = cudaStreamWaitEvent(st, ev_rest, 0);   // join st_aux
    cudaEventDestroy(ev_panel);
    cudaEventDestroy(ev_rest);
    if (e == cudaSuccess) e = cudaGetLastError();
    *nlaunch = count;
    return e;
}

// Per-node priorities of the captured factor graph: the kernels of the latency chain (panels, block-column updates, the
// tile columns the next block factors: `part` == 0) get the highest priority, the bulk of the trailing update (the
// look-ahead branch) the lowest, and the graph is instantiated with cudaGraphInstantiateFlagUseNodePriority.  Without it
// every node runs at the priority of the stream the graph is launched into, the CTAs of a bulk update -- all queued before
// the next chain's kernels -- take every free SM slot first, and the chain only overlaps the bulk's last wave.
// SPLPAK_B200_GRAPHPRIO=0 disables (A/B).
static cudaError_t spl_graph_priorities(cudaGraph_t gr) {
    const char *env = getenv("SPLPAK_B200_GRAPHPRIO");
    if (env && atoi(env) == 0) return cudaErrorNotSupported;
    int least = 0, greatest = 0;
    cudaError_t e = cudaDeviceGetStreamPriorityRange(&least, &greatest);
    if (e != cudaSuccess || greatest >= least) return e != cudaSuccess ? e : cudaErrorNotSupported;
    size_t nn = 0;
    if ((e = cudaGraphGetNodes(gr, nullptr, &nn)) != cudaSuccess) return e;
    std::vector<cudaGraphNode_t> nodes(nn);
    if (nn && (e = cudaGraphGetNodes(gr, nodes.data(), &nn)) != cudaSuccess) return e;
    for (size_t k = 0; k < nn; ++k) {
        cudaGraphNodeType ty;
        if (cudaGraphNodeGetType(nodes[k], &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
        cudaKernelNodeParams kp;
        if (cudaGraphKernelNodeGetParams(nodes[k], &kp) != cudaSuccess) continue;
        bool chain = kp.func == (void *)spl_panel_kernel || kp.func == (void *)spl_syrk_cols_kernel;
        if (kp.func == (void *)spl_syrk_kblock_kernel || kp.func == (void *)spl_syrk256_kernel ||
            kp.func == (void *)spl_syrk_kernel)
            chain = kp.kernelParams && *static_cast<int *>(kp.kernelParams[7]) == 0;     // argument 7: `part`
        cudaKernelNodeAttrValue v;
        memset(&v, 0, sizeof(v));
        v.priority = chain ? greatest : least;
        if ((e = cudaGraphKernelNodeSetAttribute(nodes[k], cudaKernelNodeAttributePriority, &v)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// kernel-per-phase factor loop: two-level blocked (default) or one trailing update per panel (SPLPAK_B200_KBLOCK=1)
static cudaError_t enqueue_factor_phases(long long n, int bw, long long lda, double *d_AB, double *d_g, double *d_ysol,
                                         double *d_linv, int *d_fail, cudaStream_t st, cudaStream_t st_aux,
                                         size_t panel_smem, size_t syrk_smem, long long *nlaunch) {
    const int KB = spl_kblock();
    if (KB > 1)
        return enqueue_factor_blocked(n, bw, lda, d_AB, d_g, d_ysol, d_linv, d_fail, st, st_aux, panel_smem, syrk_smem, KB,
                                      nlaunch);
    return enqueue_factor(n, bw, lda, d_AB, d_g, d_ysol, d_linv, d_fail, st, st_aux, panel_smem, syrk_smem, nlaunch);
}

static cudaError_t enqueue_back(long long n, int bw, long long lda, const double *d_AB, const double *d_linv,
                                double *d_ysol, double *d_csol, const int *d_fail, cudaStream_t st,
                                long long *nlaunch) {
    const long long nblk = (n + SOLVE_NB - 1) / SOLVE_NB;
    long long count = 0;
    for (long long kb = nblk - 1; kb >= 0; --kb) {
        const long long j0 = kb * SOLVE_NB;
        const int nb = (int)((n - j0 < SOLVE_NB) ? n - j0 : SOLVE_NB);
        const long long span = (j0 < bw) ? j0 : bw;
        int blocks = (int)((span + BACK_THREADS - 1) / BACK_THREADS);
        if (blocks < 1) blocks = 1;
        spl_backsolve_kernel<<<blocks, BACK_THREADS, 0, st>>>(d_AB, lda, j0, nb, bw, d_linv + kb * 4096, d_ysol,
                                                              d_csol, d_fail);
        ++count;
    }
    *nlaunch = count;
    return cudaGetLastError();
}

int spl_solve_launch(const GridParams &gp, const double *d_S, double *d_AB, double *d_g, double *d_work,
                     double **d_coef_out, int *d_fail, cudaStream_t st, cudaStream_t st_aux, int nsm,
                     cudaEvent_t *ev, void **cache) {
    const long long n = gp.ncol;
    const int bw = spl_half_bandwidth(gp);
    const long long lda = spl_band_lda(bw);
    const long long nblk = (n + SOLVE_NB - 1) / SOLVE_NB;
    double *d_linv = d_work;
    double *d_ysol = d_work + nblk * 4096;
    double *d_csol = d_ysol + (n + 64);
    *d_coef_out = d_csol;

    const size_t syrk_smem = sizeof(double) * 2 * 64 * TILE_LD;
    const size_t panel_smem = sizeof(double) * (2 * 64 * TILE_LD + 128 + 64 + 64 + 32 * PANEL_LDT + 2);
    SPL_CUDA_TRY(cudaFuncSetAttribute(spl_syrk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)syrk_smem));
    SPL_CUDA_TRY(cudaFuncSetAttribute(spl_syrk256_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)syrk_smem));
    SPL_CUDA_TRY(cudaFuncSetAttribute(spl_syrk_cols_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)syrk_smem));
    SPL_CUDA_TRY(cudaFuncSetAttribute(spl_syrk_kblock_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)syrk_smem));
    SPL_CUDA_TRY(cudaFuncSetAttribute(spl_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)panel_smem));

    // The factor loop runs as ONE persistent cooperative kernel when the device can keep one CTA per SM resident
    // (SPLPAK_B200_SOLVER=graph selects the kernel-per-phase version: two streams, CUDA graph).
    const size_t pers_smem = panel_smem > syrk_smem ? panel_smem : syrk_smem;
    bool persistent = false;
    int pgrid = 0;
    {
        const char *mode = getenv("SPLPAK_B200_SOLVER");
        int dev = 0, coop = 0, per_sm = 0;
        if (!(mode && strcmp(mode, "graph") == 0) && cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) == cudaSuccess && coop) {
            if (cudaFuncSetAttribute(spl_factor_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)pers_smem) == cudaSuccess &&
                cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, spl_factor_persistent_kernel, PANEL_THREADS,
                                                              pers_smem) == cudaSuccess &&
                per_sm >= 1) {
                persistent = true;
                pgrid = nsm > 0 ? nsm : SPL_NSM_DEFAULT;
            }
        }
        cudaGetLastError();
    }
    // The persistent FACTOR kernel keeps one CTA per SM and gives the trailing update only the CTAs that are not on
    // the panel: right when the chain of panels dominates (cfg3: 29 tile rows, 406 update tiles per step for 119
    // helper CTAs), wrong when the update does (cfg4: 89 tile rows, 3,916 tiles for 59 helpers: 94 ms against 40 ms
    // for the kernel-per-phase version, which runs three update CTAs per SM on every SM).  Rule: the helpers must
    // get through a step's update in about four tiles each.
    bool persistent_factor = persistent;
    if (persistent) {
        const long long T = ((long long)bw + SYRK_TILE - 1) / SYRK_TILE;
        const long long helpers = (long long)pgrid - T;
        if (helpers <= 0 || (T - 1) * T / 2 > 4 * helpers) persistent_factor = false;
    }
    // Data-flow kernel (default) or the barrier-phased one (SPLPAK_B200_SOLVER=barrier) for the persistent factor loop
    const size_t df_smem = sizeof(double) * (4 * 64 * TILE_LD + 64 + 2);
    bool dataflow = false;
    int dfgrid = 1;
    if (persistent_factor) {
        const char *mode = getenv("SPLPAK_B200_SOLVER");
        int per_sm = 0;
        if (!(mode && strcmp(mode, "barrier") == 0) &&
            cudaFuncSetAttribute(spl_factor_dataflow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)df_smem) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, spl_factor_dataflow_kernel, DF_THREADS,
                                                          df_smem) == cudaSuccess &&
            per_sm >= 1) {
            const long long T = ((long long)bw + SYRK_TILE - 1) / SYRK_TILE;
            if (T >= 2) {
                const long long want = T + (T - 1) * T / 2;      // diagonal + panel workers + one helper per rest tile
                dfgrid = (int)(want < pgrid ? want : pgrid);
                dataflow = dfgrid >= T + 1;
            } else {
                dataflow = true;                                  // half bandwidth <= 64: the diagonal CTA alone
            }
        }
        cudaGetLastError();
    }
    const size_t back_smem = sizeof(double) * BACKP_SMEM_DOUBLES;
    int back_grid = 0;
    if (persistent) {
        const long long per_cta = (BACKP_THREADS / 32) * BACKP_NC;      // columns a CTA covers per step
        const long long need = ((long long)bw + SOLVE_NB + per_cta - 1) / per_cta;     // bw columns in front of a pair of blocks
        if (need >= 1 && need <= pgrid &&
            cudaFuncSetAttribute(spl_backsolve_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)back_smem) == cudaSuccess)
            back_grid = (int)need;
        cudaGetLastError();
    }
    (void)spl_panel_dbg_buffer();        // allocate (if asked for) outside stream capture
    // (re)build the graphs when the buffers or the problem changed
    SolveGraphs *sg = cache ? static_cast<SolveGraphs *>(*cache) : nullptr;
    if (cache && (!sg || sg->key_AB != d_AB || sg->key_g != d_g || sg->n != n || sg->bw != bw || sg->persistent != persistent_factor ||
                  sg->kblock != spl_kblock())) {
        spl_solve_cache_free(sg);
        sg = new (std::nothrow) SolveGraphs();
        *cache = sg;
        if (sg) {
            cudaGraph_t gr = nullptr;
            sg->persistent = persistent_factor;
            sg->kblock = spl_kblock();
            cudaError_t e = persistent_factor ? cudaSuccess : cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
            if (e == cudaSuccess && !persistent_factor) {
                const cudaError_t eq = enqueue_factor_phases(n, bw, lda, d_AB, d_g, d_ysol, d_linv, d_fail, st, st_aux,
                                                      panel_smem, syrk_smem, &sg->nfactor);
                e = cudaStreamEndCapture(st, &gr);
                if (eq != cudaSuccess) e = eq;
            }
            unsigned long long inst_flags = 0;
            if (e == cudaSuccess && !persistent_factor && spl_graph_priorities(gr) == cudaSuccess)
                inst_flags = cudaGraphInstantiateFlagUseNodePriority;
            if (e == cudaSuccess && !persistent_factor) e = cudaGraphInstantiateWithFlags(&sg->factor, gr, inst_flags);
            if (gr) cudaGraphDestroy(gr);
            gr = nullptr;
            if (e == cudaSuccess) e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
            if (e == cudaSuccess) {
                const cudaError_t eq = enqueue_back(n, bw, lda, d_AB, d_linv, d_ysol, d_csol, d_fail, st, &sg->nback);
                e = cudaStreamEndCapture(st, &gr);
                if (eq != cudaSuccess) e = eq;
            }
            if (e == cudaSuccess) e = cudaGraphInstantiate(&sg->back, gr, 0);
            if (gr) cudaGraphDestroy(gr);
            if (e != cudaSuccess) {
                fprintf(stderr, "splpak_b200: CUDA graph capture of the solve failed (%s); launching directly\n",
                        cudaGetErrorString(e));
                cudaGetLastError();
                spl_solve_cache_free(sg);
                sg = nullptr;
                *cache = nullptr;
            } else {
                sg->key_AB = d_AB;
                sg->key_g = d_g;
                sg->n = n;
                sg->bw = bw;
            }
        }
    }

    if (ev) cudaEventRecord(ev[0], st);
    {
        long long blocks = n;
        if (blocks > 148LL * 32) blocks = 148LL * 32;
        spl_expand_band_kernel<<<(unsigned)blocks, 256, 0, st>>>(gp, d_S, d_AB, lda, bw);
        ++g_spl_launches;
    }
    if (ev) cudaEventRecord(ev[1], st);
    long long nl = 0;
    bool df_done = false;
    if (persistent_factor && dataflow) {
        double *a_AB = d_AB, *a_g = d_g, *a_y = d_ysol, *a_li = d_linv;
        long long a_lda = lda, a_n = n;
        int a_bw = bw;
        int *a_fail = d_fail;
        long long *a_dbg = spl_panel_dbg_buffer();
        // flags behind the failure flag and the barrier counter of the other persistent kernels (SPL_FAIL_WORDS ints)
        unsigned *a_flags = reinterpret_cast<unsigned *>(d_fail) + DF_FLAG_STRIDE;
        SPL_CUDA_TRY(cudaMemsetAsync(a_flags, 0, sizeof(unsigned) * DF_NFLAGS * DF_FLAG_STRIDE, st));
        void *args[] = {&a_AB, &a_lda, &a_n, &a_bw, &a_g, &a_y, &a_li, &a_fail, &a_dbg, &a_flags};
        const cudaError_t ce = cudaLaunchCooperativeKernel((const void *)spl_factor_dataflow_kernel, dim3(dfgrid),
                                                           dim3(DF_THREADS), args, df_smem, st);
        if (ce == cudaSuccess) {
            nl = 1;
            df_done = true;
        } else {
            fprintf(stderr, "splpak_b200: cooperative launch of the data-flow factor kernel failed (%s)\n",
                    cudaGetErrorString(ce));
            cudaGetLastError();
        }
    }
    if (df_done) {
    } else if (persistent_factor) {
        double *a_AB = d_AB, *a_g = d_g, *a_y = d_ysol, *a_li = d_linv;
        long long a_lda = lda, a_n = n;
        int a_bw = bw;
        int *a_fail = d_fail;
        long long *a_dbg = spl_panel_dbg_buffer();
        // the barrier counter lives behind the failure flag (d_fail is allocated as two ints by the handle)
        unsigned *a_bar = reinterpret_cast<unsigned *>(d_fail + 1);
        SPL_CUDA_TRY(cudaMemsetAsync(a_bar, 0, sizeof(unsigned), st));
        void *args[] = {&a_AB, &a_lda, &a_n, &a_bw, &a_g, &a_y, &a_li, &a_fail, &a_dbg, &a_bar};
        const cudaError_t ce = cudaLaunchCooperativeKernel((const void *)spl_factor_persistent_kernel, dim3(pgrid),
                                                           dim3(PANEL_THREADS), args, pers_smem, st);
        if (ce == cudaSuccess) {
            nl = 1;
        } else {
            // e.g. the grid cannot be co-resident in this context: fall back to the kernel-per-phase loop
            fprintf(stderr, "splpak_b200: cooperative launch of the factor kernel failed (%s); launching per phase\n",
                    cudaGetErrorString(ce));
            cudaGetLastError();
            SPL_CUDA_TRY(enqueue_factor_phases(n, bw, lda, d_AB, d_g, d_ysol, d_linv, d_fail, st, st_aux, panel_smem, syrk_smem, &nl));
        }
    } else if (sg && sg->factor) {
        SPL_CUDA_TRY(cudaGraphLaunch(sg->factor, st));
        nl = sg->nfactor;
    } else {
        SPL_CUDA_TRY(enqueue_factor_phases(n, bw, lda, d_AB, d_g, d_ysol, d_linv, d_fail, st, st_aux, panel_smem, syrk_smem, &nl));
    }
    g_spl_launches += nl;
    if (spl_panel_dbg_buffer()) {
        long long hst[512];
        cudaStreamSynchronize(st);
        cudaMemcpy(hst, spl_panel_dbg_buffer(), sizeof(hst), cudaMemcpyDeviceToHost);
        if (df_done) {
            fprintf(stderr, "data-flow step (diagonal CTA, compute warps): chol %lld, inverse %lld, store Linv + operand wait %lld, y1 %lld, "
                            "L10 product %lld, diagonal update %lld, total %lld\n",
                    hst[1] - hst[0], hst[2] - hst[1], hst[3] - hst[2], hst[4] - hst[3], hst[5] - hst[4], hst[6] - hst[5],
                    hst[6] - hst[0]);
            fprintf(stderr, "  L10 product: MMA loop (warp 0) %lld, barrier %lld, transposition + barrier %lld, store %lld\n",
                    hst[40] - hst[4], hst[41] - hst[40], hst[42] - hst[41], hst[5] - hst[42]);
            fprintf(stderr, "  communication warp: wait T10/T11 %lld, arrive %lld, wait Linv %lld, post Linv %lld, "
                            "wait L10 %lld, post L10 + g share %lld\n",
                    hst[33] - hst[32], hst[34] - hst[33], hst[35] - hst[34], hst[36] - hst[35], hst[37] - hst[36],
                    hst[38] - hst[37]);
            fprintf(stderr, "  panel worker 1: wait Linv %lld, L21 gemm %lld, B1 %lld, column-0 tile %lld, B2 %lld (step start %+lld ns, B1 passed %+lld ns after the diagonal CTA's step start)\n",
                    hst[17] - hst[16], hst[18] - hst[17], hst[19] - hst[18], hst[20] - hst[19], hst[21] - hst[20],
                    hst[22] - hst[8], hst[23] - hst[8]);
            {
                // the five last arrivals at B1 of the stamped step (ns after the diagonal CTA's step start)
                int order[512], nw = 0;
                for (int c = 1; c < dfgrid && c < 448; ++c) order[nw++] = c;
                for (int a = 0; a < nw; ++a)
                    for (int b2 = a + 1; b2 < nw; ++b2)
                        if (hst[64 + order[b2]] > hst[64 + order[a]]) { const int t_ = order[a]; order[a] = order[b2]; order[b2] = t_; }
                fprintf(stderr, "  B1 arrivals (ns after the diagonal CTA's step start): last");
                for (int a = 0; a < 6 && a < nw; ++a) fprintf(stderr, " cta %d %+lld", order[a], hst[64 + order[a]] - hst[8]);
                fprintf(stderr, " .. median cta %d %+lld, first cta %d %+lld\n", order[nw / 2], hst[64 + order[nw / 2]] - hst[8],
                        order[nw - 1], hst[64 + order[nw - 1]] - hst[8]);
            }
            fprintf(stderr, "  helper 0: B1 %lld, first tile %lld, rest of its list %lld (B1 passed %+lld ns after the diagonal CTA's step start)\n",
                    hst[27] - hst[24], hst[28] - hst[27], hst[29] - hst[28], hst[31] - hst[8]);
        } else if (persistent_factor) {
            fprintf(stderr, "persistent step (CTA 0): panel body %lld, barrier 1 %lld, column-0 tile %lld, barrier 2 %lld\n",
                    hst[12] - hst[0], hst[13] - hst[12], hst[14] - hst[13], hst[15] - hst[14]);
        }
        if (!df_done)
            fprintf(stderr, "panel (mid) clocks: load %lld chol %lld inverse %lld wait %lld y1 %lld gemm+store %lld total %lld\n",
                    hst[1] - hst[0], hst[2] - hst[1], hst[3] - hst[2], hst[4] - hst[3], hst[5] - hst[4], hst[6] - hst[5],
                    hst[6] - hst[0]);
    }
    if (ev) cudaEventRecord(ev[2], st);
    if (persistent && back_grid > 0) {
        const double *a_AB = d_AB, *a_li = d_linv;
        double *a_y = d_ysol, *a_c = d_csol;
        long long a_lda = lda, a_n = n;
        int a_bw = bw;
        const int *a_fail = d_fail;
        unsigned *a_bar = reinterpret_cast<unsigned *>(d_fail + 1);
        SPL_CUDA_TRY(cudaMemsetAsync(a_bar, 0, sizeof(unsigned), st));
        void *args[] = {&a_AB, &a_lda, &a_n, &a_bw, &a_li, &a_y, &a_c, &a_fail, &a_bar};
        const cudaError_t ce = cudaLaunchCooperativeKernel((const void *)spl_backsolve_persistent_kernel, dim3(back_grid),
                                                           dim3(BACKP_THREADS), args, back_smem, st);
        if (ce == cudaSuccess) {
            nl = 1;
        } else {
            fprintf(stderr, "splpak_b200: cooperative launch of the back-substitution failed (%s); launching per block\n",
                    cudaGetErrorString(ce));
            cudaGetLastError();
            SPL_CUDA_TRY(enqueue_back(n, bw, lda, d_AB, d_linv, d_ysol, d_csol, d_fail, st, &nl));
        }
    } else if (sg && sg->back) {
        SPL_CUDA_TRY(cudaGraphLaunch(sg->back, st));
        nl = sg->nback;
    } else {
        SPL_CUDA_TRY(enqueue_back(n, bw, lda, d_AB, d_linv, d_ysol, d_csol, d_fail, st, &nl));
    }
    g_spl_launches += nl;
    if (ev) cudaEventRecord(ev[3], st);
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// Solve G c = g again with the factor left in d_AB / d_work by spl_solve_launch (same layout of d_work); g is
// destroyed.  Only the two persistent substitution kernels run: returns SPLPAK_ERR_HANDLE when they are not
// available for this shape (the caller then re-factors).
int spl_resolve_launch(const GridParams &gp, const double *d_AB, double *d_g, double *d_work, double **d_coef_out,
                       int *d_fail, cudaStream_t st, int nsm) {
    const long long n = gp.ncol;
    const int bw = spl_half_bandwidth(gp);
    const long long lda = spl_band_lda(bw);
    const long long nblk = (n + SOLVE_NB - 1) / SOLVE_NB;
    double *d_linv = d_work;
    double *d_ysol = d_work + nblk * 4096;
    double *d_csol = d_ysol + (n + 64);
    *d_coef_out = d_csol;
    const char *mode = getenv("SPLPAK_B200_SOLVER");
    if (mode && strcmp(mode, "graph") == 0) return SPLPAK_ERR_HANDLE;
    int dev = 0, coop = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) != cudaSuccess || !coop) {
        cudaGetLastError();
        return SPLPAK_ERR_HANDLE;
    }
    const int pgrid = nsm > 0 ? nsm : SPL_NSM_DEFAULT;
    const size_t back_smem = sizeof(double) * BACKP_SMEM_DOUBLES;
    const size_t fwd_smem = sizeof(double) * (2 * 64 * FWDP_LD + 128 + 8 * 32);
    const long long per_cta = (BACKP_THREADS / 32) * BACKP_NC;
    const long long back_grid = ((long long)bw + SOLVE_NB + per_cta - 1) / per_cta;
    long long fwd_grid = ((((long long)bw + 31) / 32) * 2 + FWDP_THREADS / 32 - 1) / (FWDP_THREADS / 32);
    if (fwd_grid < 1) fwd_grid = 1;
    if (back_grid < 1 || back_grid > pgrid || fwd_grid > pgrid) return SPLPAK_ERR_HANDLE;
    if (cudaFuncSetAttribute(spl_backsolve_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)back_smem) != cudaSuccess ||
        cudaFuncSetAttribute(spl_forwardsolve_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)fwd_smem) != cudaSuccess) {
        cudaGetLastError();
        return SPLPAK_ERR_HANDLE;
    }
    unsigned *a_bar = reinterpret_cast<unsigned *>(d_fail + 1);
    {
        const double *a_AB = d_AB, *a_li = d_linv;
        double *a_g = d_g, *a_y = d_ysol;
        long long a_lda = lda, a_n = n;
        int a_bw = bw;
        const int *a_fail = d_fail;
        SPL_CUDA_TRY(cudaMemsetAsync(a_bar, 0, sizeof(unsigned), st));
        void *args[] = {&a_AB, &a_lda, &a_n, &a_bw, &a_li, &a_g, &a_y, &a_fail, &a_bar};
        if (cudaLaunchCooperativeKernel((const void *)spl_forwardsolve_persistent_kernel, dim3((unsigned)fwd_grid),
                                        dim3(FWDP_THREADS), args, fwd_smem, st) != cudaSuccess) {
            cudaGetLastError();
            return SPLPAK_ERR_HANDLE;
        }
        ++g_spl_launches;
    }
    {
        const double *a_AB = d_AB, *a_li = d_linv;
        double *a_y = d_ysol, *a_c = d_csol;
        long long a_lda = lda, a_n = n;
        int a_bw = bw;
        const int *a_fail = d_fail;
        SPL_CUDA_TRY(cudaMemsetAsync(a_bar, 0, sizeof(unsigned), st));
        void *args[] = {&a_AB, &a_lda, &a_n, &a_bw, &a_li, &a_y, &a_c, &a_fail, &a_bar};
        SPL_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)spl_backsolve_persistent_kernel, dim3((unsigned)back_grid),
                                                 dim3(BACKP_THREADS), args, back_smem, st));
        ++g_spl_launches;
    }
    return SPLPAK_OK;
}

// min / max of diag(L) over all panels, from the stored block inverses (L_jj = 1 / Linv_jj): out2 = {min, max}
__global__ void __launch_bounds__(1024)
spl_pivot_range_kernel(const double *__restrict__ linv, long long n, double *__restrict__ out2) {
    __shared__ double s_mn[1024], s_mx[1024];
    double mn = 1e300, mx = 0.0;
    for (long long j = threadIdx.x; j < n; j += 1024) {
        const long long kb = j / SOLVE_NB;
        const int r = (int)(j % SOLVE_NB);
        const double li = fabs(linv[kb * 4096 + r * 64 + r]);
        if (li > 0.0) {
            const double l = 1.0 / li;
            mn = fmin(mn, l);
            mx = fmax(mx, l);
        } else {
            mn = 0.0;
        }
    }
    s_mn[threadIdx.x] = mn;
    s_mx[threadIdx.x] = mx;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            s_mn[threadIdx.x] = fmin(s_mn[threadIdx.x], s_mn[threadIdx.x + o]);
            s_mx[threadIdx.x] = fmax(s_mx[threadIdx.x], s_mx[threadIdx.x + o]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out2[0] = s_mn[0];
        out2[1] = s_mx[0];
    }
}
int spl_pivot_range_launch(const GridParams &gp, const double *d_work, double *d_out2, cudaStream_t st) {
    spl_pivot_range_kernel<<<1, 1024, 0, st>>>(d_work, gp.ncol, d_out2);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}
