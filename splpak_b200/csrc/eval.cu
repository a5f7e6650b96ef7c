// eval.cu -- batched splfe / splde (src/splpak.F90:1089-1275) for sm_100a.
//
// One persistent CTA per SM.  The whole coefficient table (<= 166 KB at the named configs) is staged
// once per CTA into shared memory with 1-D bulk async copies (cp.async.bulk -> SASS UBLKCP) signalled
// through an mbarrier.  After that there is no CTA-wide synchronisation: every warp claims chunks of
// 256 queries from a global atomic counter (dynamic scheduling), one query per lane, the coordinates
// of the next 32 queries in flight while the current 32 are evaluated.  Tables that do not fit in
// shared memory are gathered through the read-only path from L2 (same kernel, SMEM = false).
//
// Per query: four 1-D weights per dimension (basis.cuh: same formulas and index box as the
// reference), then the nested contraction  sum_k b3[k] sum_j b2[j] sum_i coef[..]*b1[i]  with
// dimension 1 innermost (4 contiguous coefficients).
//
// What binds the plain kernel for scattered queries is the GATHER of the 4^ndim coefficients: 64 8-byte
// shared-memory loads per 3-D query at random addresses, ~3 bank-conflict wavefronts per half-warp each (measured
// in round 1: 12.9 crossbar cycles per query per SM; 4 is the conflict-free floor).  Queries that arrive in
// coherent runs (raster order of an output grid) broadcast and are bound by instruction issue and the FP64 pipe.
//
// spl_eval_regroup_kernel (2-D..4-D, large batches) removes the conflicts by construction, without any CTA-wide
// barrier: the gather offsets i + s1 j + s2 k are the same for every query, so two queries whose BASE addresses
// differ mod 16 (8-byte banks per half-warp phase) never collide on any of the 4^ndim loads.  Lane l of a warp is
// DEDICATED to bank class l mod 16; every warp keeps 16 small per-class FIFOs in shared memory (its own, warp
// private: only __syncwarp), inserts the raw queries it streams (class from the window index; rank among same-class
// lanes from four ballots; the FIFO cursors live in registers of the dedicated lanes), and every round each lane
// pops one query of ITS class and evaluates it.  Queries whose FIFO is full stay pending in their lane and retry next
// round; coherent batches (raster order: all lanes in one class) bypass the FIFOs.  The table is padded to strides
// chosen so that the class distribution is uniform (24^3: s1 = 25, s2 = 603 -> within 1.4 %).
//
// Algorithmic HBM traffic: (ndim + 1) reals per query.
#include <stdlib.h>
#include <string.h>

#include "basis.cuh"

struct DerivParams {
    int nd[SPL_MAXDIM];
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *mbar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(mbar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *mbar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(mbar)), "r"(parity)
            : "memory");
    }
}
// global -> shared bulk copy (bytes: multiple of 16; src/dst 16-byte aligned), completion on mbar.
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *mbar) {
    const uint32_t chunk = 32768;
    for (uint32_t off = 0; off < bytes; off += chunk) {
        const uint32_t nb = min(chunk, bytes - off);
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                smem_u32((const char *)dst + off)),
            "l"((const char *)src + off), "r"(nb), "r"(smem_u32(mbar))
            : "memory");
    }
}

// Strides (in doubles) of the coefficient table the kernel reads: the caller's natural layout
// (s1 = nodes(1), s2 = nodes(1)*nodes(2), ...) or the padded shared-memory copy of the ring kernel.
struct TableLayout {
    int s1, s2;
    long long s3;
};

// Nested contraction over the 4^NDIM window starting at p0, dimension 1 innermost.
template <int NDIM, typename T = double>
__device__ __forceinline__ T spl_contract_at(const TableLayout &tl, const T *__restrict__ p0, const T (*b)[4]) {
    T sum = (T)0;
    if constexpr (NDIM == 1) {
#pragma unroll
        for (int i = 0; i < 4; ++i) sum = fma(p0[i], b[0][i], sum);
    } else if constexpr (NDIM == 2) {
        const int n0 = tl.s1;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const T *p = p0 + n0 * j;
            T sj = (T)0;
#pragma unroll
            for (int i = 0; i < 4; ++i) sj = fma(p[i], b[0][i], sj);
            sum = fma(sj, b[1][j], sum);
        }
    } else if constexpr (NDIM == 3) {
        const int n0 = tl.s1;
        const int n01 = tl.s2;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            T sk = (T)0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const T *p = p0 + n0 * j + n01 * k;
                T sj = (T)0;
#pragma unroll
                for (int i = 0; i < 4; ++i) sj = fma(p[i], b[0][i], sj);
                sk = fma(sj, b[1][j], sk);
            }
            sum = fma(sk, b[2][k], sum);
        }
    } else {
        const int n0 = tl.s1;
        const int n01 = tl.s2;
        const long long n012 = tl.s3;
#pragma unroll 1
        for (int l = 0; l < 4; ++l) {
            T sl = (T)0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                T sk = (T)0;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const T *p = p0 + n0 * j + n01 * k + n012 * l;
                    T sj = (T)0;
#pragma unroll
                    for (int i = 0; i < 4; ++i) sj = fma(p[i], b[0][i], sj);
                    sk = fma(sj, b[1][j], sk);
                }
                sl = fma(sk, b[2][k], sl);
            }
            sum = fma(sl, b[3][l], sum);
        }
    }
    return sum;
}

// window start from the per-dimension first nodes ws[]
template <int NDIM, typename T = double>
__device__ __forceinline__ T spl_contract(const TableLayout &tl, const T *__restrict__ cf,
                                          const int *ws, const T (*b)[4]) {
    const T *p0 = cf + ws[0];
    if constexpr (NDIM >= 2) p0 += tl.s1 * ws[1];
    if constexpr (NDIM >= 3) p0 += (long long)tl.s2 * ws[2];
    if constexpr (NDIM >= 4) p0 += tl.s3 * ws[3];
    return spl_contract_at<NDIM, T>(tl, p0, b);
}

// One query: weights of every dimension, then the contraction.  VALUE: every nderiv is 0 (splfe).
template <int NDIM, bool VALUE>
__device__ __forceinline__ double spl_eval_point(const GridParams &gp, const DerivParams &dp,
                                                 const TableLayout &tl, const double *__restrict__ cf,
                                                 const double *xv) {
    double b[NDIM][4];
    int ws[NDIM];
#pragma unroll
    for (int d = 0; d < NDIM; ++d) {
        if (VALUE)
            spl_window_weights_value<true>(xv[d], gp.xmin[d], gp.dx[d], gp.dxin[d], gp.nodes[d], ws[d], b[d]);   // 8 x
        else
            spl_window_weights(xv[d], gp.xmin[d], gp.dx[d], gp.dxin[d], gp.nodes[d], dp.nd[d], ws[d], b[d]);
    }
    double sum = spl_contract<NDIM>(tl, cf, ws, b);
    if (VALUE) {
        sum *= 1.0 / (double)spl_ipow(8, NDIM);      // the weights carry a factor 8 per dimension (exact scaling)
        // a NaN coordinate fails every comparison of bascmp, so every basis value stays 0 (:253-379)
        bool isnan_q = false;
#pragma unroll
        for (int d = 0; d < NDIM; ++d) isnan_q |= (xv[d] != xv[d]);
        if (isnan_q) sum = 0.0;
    }
    return sum;
}

// Uniform (phantom-node) form, basis.cuh: the same query against the EXTENDED table (nodes + 2 per dimension,
// spl_uni_table_kernel), window = extended entries cell .. cell+3 per dimension.
template <int NDIM>
__device__ __forceinline__ double spl_uni_scale(const GridParams &gp, const DerivParams &dp, bool value) {
    double sc = 1.0 / (double)spl_ipow(4, NDIM);
    if (!value) {
#pragma unroll
        for (int d = 0; d < NDIM; ++d) {
            if (dp.nd[d] >= 1) sc *= gp.dxin[d];
            if (dp.nd[d] >= 2) sc *= gp.dxin[d];
        }
    }
    return sc;
}
// from the fractional coordinates f[] and the window's base offset (flag SPL_UNI_OOB: some coordinate is out of range)
template <int NDIM, bool VALUE>
__device__ __forceinline__ double spl_eval_point_uni_at(const DerivParams &dp, const TableLayout &tl,
                                                        const double *__restrict__ cf, const double *f, unsigned base,
                                                        double scale) {
    double b[NDIM][4];
    const bool oob = (base & SPL_UNI_OOB) != 0u;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) spl_uni_weights<VALUE>(f[d], oob, VALUE ? 0 : dp.nd[d], b[d]);
    double sum = spl_contract_at<NDIM>(tl, cf + (base & ~SPL_UNI_OOB), b) * scale;
    // a NaN coordinate fails every comparison of bascmp, so every basis value stays 0 (:253-379)
    bool isnan_q = false;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) isnan_q |= (f[d] != f[d]);
    if (isnan_q) sum = 0.0;
    return sum;
}
template <int NDIM>
__device__ __forceinline__ unsigned spl_uni_locate(const GridParams &gp, const TableLayout &tl, const double *xv, double *f) {
    unsigned base = 0u;
    bool any = false;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) {
        int cell;
        bool oob;
        spl_uni_cell(xv[d], gp.xmin[d], gp.dxin[d], gp.nodes[d], cell, f[d], oob);
        any |= oob;
        const unsigned st = d == 0 ? 1u : (d == 1 ? (unsigned)tl.s1 : (d == 2 ? (unsigned)tl.s2 : (unsigned)tl.s3));
        base += (unsigned)cell * st;
    }
    return base | (any ? SPL_UNI_OOB : 0u);
}
template <int NDIM, bool VALUE>
__device__ __forceinline__ double spl_eval_point_uni(const GridParams &gp, const DerivParams &dp, const TableLayout &tl,
                                                     const double *__restrict__ cf, const double *xv, double scale) {
    double f[NDIM];
    const unsigned base = spl_uni_locate<NDIM>(gp, tl, xv, f);
    return spl_eval_point_uni_at<NDIM, VALUE>(dp, tl, cf, f, base, scale);
}

// ------------------------------------------------------------------------------------------
// Fused derivative sets (splpak_b200_eval_derivs): every partial derivative of total order <= ORDER of one query from
// ONE gather of its 4^ndim coefficients.  Output order: the value, d/dx1 .. d/dxn, then (ORDER 2) d2/dxi dxj for i <= j
// in row order.  Component k is bit-identical to the single-nderiv evaluation: each is the nested contraction of
// spl_contract_at with that component's weights per dimension, in the same fma order; what is shared is the gather
// and every partial sum over dimensions 1..m that components agree on (weight SET s of a dimension: derivative order
// s, and in the exact form set ORDER + 1 = the x8 value weights of spl_window_weights_value, which splfe uses and
// which only combine with each other).
// ------------------------------------------------------------------------------------------
__host__ __device__ constexpr int spl_ncomp(int ndim, int order) {
    return order == 1 ? ndim + 1 : (ndim + 1) * (ndim + 2) / 2;
}
// a prefix s[0..m-1] of weight sets that some output component extends
template <int ORDER>
__device__ constexpr bool spl_dprefix(int m, int s0, int s1 = 0, int s2 = 0, int s3 = 0) {
    const int s[4] = {s0, s1, s2, s3};
    int nv = 0, tot = 0;
    for (int i = 0; i < m; ++i) {
        nv += s[i] > ORDER;
        tot += s[i] > ORDER ? 0 : s[i];
    }
    return (nv == 0 || nv == m) && tot <= ORDER;
}
// output component of a full set of weight sets (-1: none; VSET: the exact form, whose value is the all-x8 set)
template <int NDIM, int ORDER, bool VSET>
__device__ constexpr int spl_dcomp(int s0, int s1 = 0, int s2 = 0, int s3 = 0) {
    const int s[4] = {s0, s1, s2, s3};
    if (!spl_dprefix<ORDER>(NDIM, s0, s1, s2, s3)) return -1;
    int tot = 0, i1 = -1, i2 = -1;
    for (int d = 0; d < NDIM; ++d) {
        if (s[d] > ORDER) return 0;
        tot += s[d];
        if (s[d] == 2) i1 = i2 = d;
        else if (s[d] == 1) (i1 < 0 ? i1 : i2) = d;
    }
    if (tot == 0) return VSET ? -1 : 0;
    if (tot == 1) return 1 + i1;
    return 1 + NDIM + i1 * NDIM - i1 * (i1 - 1) / 2 + (i2 - i1);
}
// derivative order of dimension d in component c (inverse of spl_dcomp)
__device__ __forceinline__ int spl_dorder(int ndim, int c, int d) {
    if (c == 0) return 0;
    if (c <= ndim) return c - 1 == d ? 1 : 0;
    int r = c - 1 - ndim, i = 0;
    while (r >= ndim - i) r -= ndim - i++;
    const int j = i + r;
    return (i == d) + (j == d);
}

// res[c] (NS weight sets per dimension, b[d][s][k]): the contraction of every component, dimension 1 innermost
template <int NDIM, int ORDER, int NS>
__device__ __forceinline__ void spl_contract_multi(const TableLayout &tl, const double *__restrict__ p0,
                                                   const double (*b)[NS][4], double *res) {
    constexpr bool VSET = NS > ORDER + 1;
#pragma unroll
    for (int c = 0; c < spl_ncomp(NDIM, ORDER); ++c) res[c] = 0.0;
    if constexpr (NDIM == 1) {
#pragma unroll
        for (int a = 0; a < NS; ++a) {
            const int c = spl_dcomp<1, ORDER, VSET>(a);
            if (c < 0) continue;
#pragma unroll
            for (int i = 0; i < 4; ++i) res[c] = fma(p0[i], b[0][a][i], res[c]);
        }
    } else if constexpr (NDIM == 2) {
        const int n0 = tl.s1;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double *p = p0 + n0 * j;
            double v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = p[i];
#pragma unroll
            for (int a = 0; a < NS; ++a) {
                if (!spl_dprefix<ORDER>(1, a)) continue;
                double sj = 0.0;
#pragma unroll
                for (int i = 0; i < 4; ++i) sj = fma(v[i], b[0][a][i], sj);
#pragma unroll
                for (int e = 0; e < NS; ++e) {
                    const int c = spl_dcomp<2, ORDER, VSET>(a, e);
                    if (c >= 0) res[c] = fma(sj, b[1][e][j], res[c]);
                }
            }
        }
    } else if constexpr (NDIM == 3) {
        const int n0 = tl.s1;
        const int n01 = tl.s2;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            double sk[NS][NS];
#pragma unroll
            for (int a = 0; a < NS; ++a)
#pragma unroll
                for (int e = 0; e < NS; ++e) sk[a][e] = 0.0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double *p = p0 + n0 * j + n01 * k;
                double v[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) v[i] = p[i];
#pragma unroll
                for (int a = 0; a < NS; ++a) {
                    if (!spl_dprefix<ORDER>(1, a)) continue;
                    double sj = 0.0;
#pragma unroll
                    for (int i = 0; i < 4; ++i) sj = fma(v[i], b[0][a][i], sj);
#pragma unroll
                    for (int e = 0; e < NS; ++e)
                        if (spl_dprefix<ORDER>(2, a, e)) sk[a][e] = fma(sj, b[1][e][j], sk[a][e]);
                }
            }
#pragma unroll
            for (int a = 0; a < NS; ++a)
#pragma unroll
                for (int e = 0; e < NS; ++e)
#pragma unroll
                    for (int g = 0; g < NS; ++g) {
                        const int c = spl_dcomp<3, ORDER, VSET>(a, e, g);
                        if (c >= 0) res[c] = fma(sk[a][e], b[2][g][k], res[c]);
                    }
        }
    } else {
        const int n0 = tl.s1;
        const int n01 = tl.s2;
        const long long n012 = tl.s3;
#pragma unroll
        for (int l = 0; l < 4; ++l) {
            double sl[NS][NS][NS];
#pragma unroll
            for (int a = 0; a < NS; ++a)
#pragma unroll
                for (int e = 0; e < NS; ++e)
#pragma unroll
                    for (int g = 0; g < NS; ++g) sl[a][e][g] = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                double sk[NS][NS];
#pragma unroll
                for (int a = 0; a < NS; ++a)
#pragma unroll
                    for (int e = 0; e < NS; ++e) sk[a][e] = 0.0;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const double *p = p0 + n0 * j + n01 * k + n012 * l;
                    double v[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) v[i] = p[i];
#pragma unroll
                    for (int a = 0; a < NS; ++a) {
                        if (!spl_dprefix<ORDER>(1, a)) continue;
                        double sj = 0.0;
#pragma unroll
                        for (int i = 0; i < 4; ++i) sj = fma(v[i], b[0][a][i], sj);
#pragma unroll
                        for (int e = 0; e < NS; ++e)
                            if (spl_dprefix<ORDER>(2, a, e)) sk[a][e] = fma(sj, b[1][e][j], sk[a][e]);
                    }
                }
#pragma unroll
                for (int a = 0; a < NS; ++a)
#pragma unroll
                    for (int e = 0; e < NS; ++e)
#pragma unroll
                        for (int g = 0; g < NS; ++g)
                            if (spl_dprefix<ORDER>(3, a, e, g)) sl[a][e][g] = fma(sk[a][e], b[2][g][k], sl[a][e][g]);
            }
#pragma unroll
            for (int a = 0; a < NS; ++a)
#pragma unroll
                for (int e = 0; e < NS; ++e)
#pragma unroll
                    for (int g = 0; g < NS; ++g)
#pragma unroll
                        for (int h = 0; h < NS; ++h) {
                            const int c = spl_dcomp<4, ORDER, VSET>(a, e, g, h);
                            if (c >= 0) res[c] = fma(sl[a][e][g], b[3][h][l], res[c]);
                        }
        }
    }
}

// one query, exact form (bascmp's node-by-node formulas): the ncomp results to o[0 .. ncomp-1]
template <int NDIM, int ORDER>
__device__ __forceinline__ void spl_eval_derivs_point(const GridParams &gp, const TableLayout &tl,
                                                      const double *__restrict__ cf, const double *xv,
                                                      real_t *__restrict__ o) {
    constexpr int NS = ORDER + 2;
    double b[NDIM][NS][4];
    int ws[NDIM];
#pragma unroll
    for (int d = 0; d < NDIM; ++d) {
#pragma unroll
        for (int s = 0; s <= ORDER; ++s)
            spl_window_weights(xv[d], gp.xmin[d], gp.dx[d], gp.dxin[d], gp.nodes[d], s, ws[d], b[d][s]);
        spl_window_weights_value<true>(xv[d], gp.xmin[d], gp.dx[d], gp.dxin[d], gp.nodes[d], ws[d], b[d][ORDER + 1]);
    }
    const double *p0 = cf + ws[0];
    if constexpr (NDIM >= 2) p0 += tl.s1 * ws[1];
    if constexpr (NDIM >= 3) p0 += (long long)tl.s2 * ws[2];
    if constexpr (NDIM >= 4) p0 += tl.s3 * ws[3];
    double res[spl_ncomp(NDIM, ORDER)];
    spl_contract_multi<NDIM, ORDER, NS>(tl, p0, b, res);
    // the value as spl_eval_point<VALUE = true>: 8^-ndim, and 0 for a NaN coordinate
    res[0] *= 1.0 / (double)spl_ipow(8, NDIM);
    bool isnan_q = false;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) isnan_q |= (xv[d] != xv[d]);
    if (isnan_q) res[0] = 0.0;
#pragma unroll
    for (int c = 0; c < spl_ncomp(NDIM, ORDER); ++c) o[c] = (real_t)res[c];
}
// one query, uniform form, from its fractional coordinates and window base (spl_uni_locate); scale[c]: the factor
// spl_uni_scale gives component c
template <int NDIM, int ORDER>
__device__ __forceinline__ void spl_eval_derivs_uni_at(const TableLayout &tl, const double *__restrict__ cf,
                                                       const double *f, unsigned base, const double *scale,
                                                       real_t *__restrict__ o) {
    constexpr int NS = ORDER + 1;
    double b[NDIM][NS][4];
    const bool oob = (base & SPL_UNI_OOB) != 0u;
#pragma unroll
    for (int d = 0; d < NDIM; ++d)
#pragma unroll
        for (int s = 0; s < NS; ++s) spl_uni_weights<false>(f[d], oob, s, b[d][s]);
    double res[spl_ncomp(NDIM, ORDER)];
    spl_contract_multi<NDIM, ORDER, NS>(tl, cf + (base & ~SPL_UNI_OOB), b, res);
    bool isnan_q = false;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) isnan_q |= (f[d] != f[d]);
#pragma unroll
    for (int c = 0; c < spl_ncomp(NDIM, ORDER); ++c) o[c] = (real_t)(isnan_q ? 0.0 : res[c] * scale[c]);
}
// spl_uni_scale of every component, same multiplication order (one entry per thread c < ncomp)
template <int NDIM, int ORDER>
__device__ __forceinline__ double spl_uni_dscale(const GridParams &gp, int c) {
    double sc = 1.0 / (double)spl_ipow(4, NDIM);
#pragma unroll
    for (int d = 0; d < NDIM; ++d) {
        const int nd = spl_dorder(NDIM, c, d);
        if (nd >= 1) sc *= gp.dxin[d];
        if (nd >= 2) sc *= gp.dxin[d];
    }
    return sc;
}

// threads per CTA of the plain kernel; ORDER > 0: the derivative sets, which carry (ORDER + 1..2) x 4 weights per dimension
// and up to 15 accumulators -- sized so that ptxas needs no spills (eval.ptxas.log)
template <int NDIM, int ORDER = 0> struct EvalCfg {
    static constexpr int THREADS = ORDER == 0 ? ((NDIM <= 3) ? 1024 : 512) : (NDIM <= 2 ? 512 : 256);
};

// ------------------------------------------------------------------------------------------
// kernel: one query per lane; every WARP claims its own chunks of queries from the global counter, so
// after the table is staged there is no CTA-wide barrier and the 32 warps of an SM drift out of phase
// (their FP64, shared-memory and issue demands interleave instead of peaking together).
// ------------------------------------------------------------------------------------------
#define EVAL_WCHUNK 256   // queries a warp claims per atomic (8 per lane)

// ORDER > 0: the derivative sets of spl_eval_derivs_point / spl_eval_derivs_uni_at, out(ncomp, nq); VALUE is false
template <int NDIM, bool SMEM, bool VALUE, bool UNI = false, int ORDER = 0>
__global__ void __launch_bounds__(EvalCfg<NDIM, ORDER>::THREADS, 1)
spl_eval_kernel(const __grid_constant__ GridParams gp, const DerivParams dp, const TableLayout tl,
                const real_t *__restrict__ x, int l1x, long long nq,
                const double *__restrict__ coef, long long ncol_padded, real_t *__restrict__ out,
                unsigned long long *__restrict__ chunk_counter, const int *__restrict__ order_flag) {
    constexpr int NC = ORDER > 0 ? spl_ncomp(NDIM, ORDER) : 1;
    extern __shared__ __align__(128) double s_dyn[];
    __shared__ __align__(8) uint64_t mbar;
    __shared__ unsigned long long s_chunk;
    __shared__ double s_dscale[NC];
    // order_flag (spl_eval_probe_kernel): 1 = the batch is scattered and the regrouping kernel evaluates it
    if (order_flag && *order_flag == 1) return;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    if (tid == 0) s_chunk = 0ULL;
    if constexpr (ORDER > 0 && UNI)
        if (tid < NC) s_dscale[tid] = spl_uni_dscale<NDIM, ORDER>(gp, tid);
    if (!SMEM) __syncthreads();
    const double *cf = coef;
    const double uscale = UNI ? spl_uni_scale<NDIM>(gp, dp, VALUE) : 1.0;
    if (SMEM) {
        if (tid == 0) {
            mbar_init(&mbar, 1);
            mbar_fence_init();
            mbar_expect_tx(&mbar, (uint32_t)(ncol_padded * sizeof(double)));
            bulk_g2s(s_dyn, coef, (uint32_t)(ncol_padded * sizeof(double)), &mbar);
        }
        __syncthreads();
        mbar_wait(&mbar, 0);
        cf = s_dyn;
    }
    if constexpr (NDIM <= 2 && UNI) {
        // 1-D / 2-D in the uniform form are bound by HBM, not by arithmetic: keep a whole chunk of coordinates per warp in
        // flight (KQ queries per lane, the NEXT chunk's loads issued before the current chunk is evaluated; 16-byte loads
        // for packed 2-D float64 points) -- one 8-byte load per lane in flight reaches only ~57 % of the HBM roof.
        constexpr int KQ = NDIM == 1 ? 8 : (VALUE ? 4 : 3);
        constexpr int CH = KQ * 32;
        const bool vec2 = NDIM == 2 && l1x == 2 && sizeof(real_t) == 8 && ((uintptr_t)x % 16 == 0);
        double cur[KQ][NDIM], nxt[KQ][NDIM];
        long long cbase = -1, nbase = -1;
        // static schedule (every query costs the same): CTA b owns a contiguous range, its warps take the chunks of that
        // range round robin -- no atomics (3.9e6 same-address atomics per 1e9 queries cost as much as the kernel itself)
        const long long q_lo = nq * (long long)blockIdx.x / (long long)gridDim.x;
        const long long q_hi = nq * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
        long long next_chunk = q_lo + (long long)(tid >> 5) * CH;
        auto claim = [&]() -> long long {
            const long long b = next_chunk;
            next_chunk += (long long)(blockDim.x >> 5) * CH;
            return b < q_hi ? b : -1;
        };
        auto issue = [&](long long b) {
            if (b < 0) return;
#pragma unroll
            for (int k = 0; k < KQ; ++k) {
                const long long q = b + k * 32 + lane;
                if (q < q_hi) {
                    if (NDIM == 2 && vec2) {
                        const double2 v = reinterpret_cast<const double2 *>(x)[q];
                        nxt[k][0] = v.x;
                        nxt[k][NDIM - 1] = v.y;
                    } else {
#pragma unroll
                        for (int d = 0; d < NDIM; ++d) nxt[k][d] = (double)x[q * (long long)l1x + d];
                    }
                } else {
#pragma unroll
                    for (int d = 0; d < NDIM; ++d) nxt[k][d] = 0.0;
                }
            }
        };
        nbase = claim();
        issue(nbase);
        while (nbase >= 0) {
            cbase = nbase;
#pragma unroll
            for (int k = 0; k < KQ; ++k)
#pragma unroll
                for (int d = 0; d < NDIM; ++d) cur[k][d] = nxt[k][d];
            nbase = claim();
            issue(nbase);
#pragma unroll
            for (int k = 0; k < KQ; ++k) {
                const long long q = cbase + k * 32 + lane;
                if constexpr (ORDER > 0) {
                    if (q < q_hi) {
                        double f[NDIM];
                        const unsigned base = spl_uni_locate<NDIM>(gp, tl, cur[k], f);
                        spl_eval_derivs_uni_at<NDIM, ORDER>(tl, cf, f, base, s_dscale, out + q * NC);
                    }
                } else if (q < q_hi) {
                    out[q] = (real_t)spl_eval_point_uni<NDIM, VALUE>(gp, dp, tl, cf, cur[k], uscale);
                }
            }
        }
        return;
    }
    // CTA b owns a contiguous range of the batch; its warps claim chunks of that range from a SHARED-memory counter
    // (one same-address global atomic per 256 queries, 3.9e6 per 1e9, serialises in L2 for milliseconds)
    const long long q_lo = nq * (long long)blockIdx.x / (long long)gridDim.x;
    const long long q_hi = nq * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
    for (;;) {
        unsigned long long c = 0;
        if (lane == 0) c = atomicAdd(&s_chunk, 1ULL);
        c = __shfl_sync(0xffffffffu, c, 0);
        const long long base = q_lo + (long long)c * EVAL_WCHUNK;
        if (base >= q_hi) break;
        // software pipeline: the coordinates of the next sub-step are in flight while this one is evaluated
        double xn[NDIM];
        {
            const long long q = base + lane;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) xn[d] = (q < q_hi) ? (double)x[q * (long long)l1x + d] : 0.0;
        }
#pragma unroll 1
        for (int sub = 0; sub < EVAL_WCHUNK / 32; ++sub) {
            const long long q = base + sub * 32 + lane;
            double xv[NDIM];
#pragma unroll
            for (int d = 0; d < NDIM; ++d) xv[d] = xn[d];
            const long long q2 = q + 32;
            if (sub + 1 < EVAL_WCHUNK / 32) {
#pragma unroll
                for (int d = 0; d < NDIM; ++d) xn[d] = (q2 < q_hi) ? (double)x[q2 * (long long)l1x + d] : 0.0;
            }
            if constexpr (ORDER > 0) {
                if (q < q_hi) {
                    if (UNI) {
                        double f[NDIM];
                        const unsigned base = spl_uni_locate<NDIM>(gp, tl, xv, f);
                        spl_eval_derivs_uni_at<NDIM, ORDER>(tl, cf, f, base, s_dscale, out + q * NC);
                    } else {
                        spl_eval_derivs_point<NDIM, ORDER>(gp, tl, cf, xv, out + q * NC);
                    }
                }
            } else if (q < q_hi) {
                out[q] = UNI ? (real_t)spl_eval_point_uni<NDIM, VALUE>(gp, dp, tl, cf, xv, uscale)
                             : (real_t)spl_eval_point<NDIM, VALUE>(gp, dp, tl, cf, xv);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// regrouping kernel: conflict-free gathers through warp-private per-bank-class FIFOs (see the file header)
// ------------------------------------------------------------------------------------------
#define RG_CHUNK 256u     // raw queries a warp claims from its CTA's range per shared-memory atomic

template <int NDIM, int ORDER = 0> struct RegroupCfg {
    // warps per CTA (one CTA per SM): the register budget per thread is 64 K / threads; the derivative sets (ORDER > 0)
    // need more registers than the value kernel, so fewer warps (and deeper FIFOs: regroup_plan)
    static constexpr int NWARPS = ORDER == 0 ? ((NDIM <= 2) ? 32 : (NDIM == 3 ? 24 : 16)) : (NDIM <= 2 ? 16 : 8);
};

// Order probe: are the queries scattered (regrouping kernel) or do they arrive in coherent runs, e.g. the raster order of
// an output grid (plain kernel: its gathers broadcast, and it runs 12 % faster than the regrouping kernel's bypass)?
// One CTA samples 32 groups of 32 CONSECUTIVE queries spread over the batch and counts the groups in which at least
// RG_BYPASS queries share one bank class.  Both evaluation kernels are launched; the one the flag rules out exits at once.
#define RG_BYPASS 12      // a batch with >= this many lanes in ONE class is coherent (raster order): evaluate it directly
template <int NDIM, bool UNI = false, int NCLS = 16>
__global__ void __launch_bounds__(1024)
spl_eval_probe_kernel(const __grid_constant__ GridParams gp, const TableLayout tl, const real_t *__restrict__ x, int l1x,
                      long long nq, int *__restrict__ order_flag) {
    __shared__ int s_coherent;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_coherent = 0;
    __syncthreads();
    const long long q = (nq / 32) * warp + lane;           // group `warp` starts at warp/32 of the batch
    int cls = 0;
    if (q < nq) {
        const long long st[4] = {1, tl.s1, tl.s2, tl.s3};
        int lin = 0;
#pragma unroll
        for (int d = 0; d < NDIM; ++d) {
            int ws;
            if (UNI) {
                double f;
                bool oob;
                spl_uni_cell((double)x[q * (long long)l1x + d], gp.xmin[d], gp.dxin[d], gp.nodes[d], ws, f, oob);
            } else {
                const double t = spl_mul(gp.dxin[d], spl_sub((double)x[q * (long long)l1x + d], gp.xmin[d]));
                const int it = max(__double2int_rz(t), -4);
                ws = min(max(it - 1, 0), gp.nodes[d] - 4);
            }
            lin += ws * (int)(st[d] & (NCLS - 1));
        }
        cls = lin & (NCLS - 1);
    }
    const unsigned peers = __match_any_sync(0xffffffffu, cls);
    const int big = __reduce_max_sync(0xffffffffu, __popc(peers));
    if (lane == 0 && big >= RG_BYPASS) atomicAdd(&s_coherent, 1);
    __syncthreads();
    if (threadIdx.x == 0) *order_flag = (s_coherent >= 16) ? 0 : 1;
}

// coefficient table -> padded image (strides tl.s1/s2/s3, zero-filled gaps), so that the CTAs can bulk-copy it
__global__ void spl_pad_table_kernel(const __grid_constant__ GridParams gp, const TableLayout tl,
                                     const double *__restrict__ coef, double *__restrict__ padded, long long total) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long st[4] = {1, tl.s1, tl.s2, tl.s3};
    long long mulv[4] = {1, 1, 1, 1};
    for (int d = 1; d < gp.ndim; ++d) mulv[d] = mulv[d - 1] * gp.nodes[d - 1];
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        // e = sum_d id_d st[d]: peel the indices off from the slowest dimension down (st[d+1] need not be a multiple of st[d])
        long long src = 0, rem = e;
        bool ok = true;
        for (int d = gp.ndim - 1; d >= 0; --d) {
            const long long id = rem / st[d];
            rem -= id * st[d];
            if (id >= gp.nodes[d]) ok = false;
            src += id * mulv[d];
        }
        padded[e] = ok ? coef[src] : 0.0;
    }
}

// coefficient table -> EXTENDED table of the uniform form (basis.cuh): nodes + 2 entries per dimension (extended index
// r = node + 1, r = 0 and r = nodes + 1 are the phantom nodes), strides tl.s1/s2/s3, zero-filled gaps.  Every entry is
// a fixed-order sum of <= 2^ndim coefficients with exact weights (1, 2, 4, 6 per dimension).
__device__ __forceinline__ void spl_uni_row(int r, int n, int &j0, double &w0, int &j1, double &w1) {
    const int j = r - 1;
    j1 = 0;
    w1 = 0.0;
    if (j == -1)          { j0 = 0; w0 = 4.0; j1 = 1; w1 = 6.0; }
    else if (j == 0)      { j0 = 0; w0 = 2.0; j1 = 1; w1 = 4.0; }
    else if (j == 1)      { j0 = 1; w0 = 2.0; }
    else if (j == n)      { j0 = n - 1; w0 = 4.0; j1 = n - 2; w1 = 6.0; }
    else if (j == n - 1)  { j0 = n - 1; w0 = 2.0; j1 = n - 2; w1 = 4.0; }
    else if (j == n - 2)  { j0 = n - 2; w0 = 2.0; }
    else                  { j0 = j; w0 = 1.0; }
}
template <typename TI, typename TO>
__global__ void spl_uni_table_kernel(const __grid_constant__ GridParams gp, const TableLayout tl,
                                     const TI *__restrict__ coef, TO *__restrict__ ext, long long total) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long st[4] = {1, tl.s1, tl.s2, tl.s3};
    long long mulv[4] = {1, 1, 1, 1};
    for (int d = 1; d < gp.ndim; ++d) mulv[d] = mulv[d - 1] * gp.nodes[d - 1];
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
        long long rem = e;
        bool ok = true;
        int j0[SPL_MAXDIM], j1[SPL_MAXDIM];
        double w0[SPL_MAXDIM], w1[SPL_MAXDIM];
        for (int d = gp.ndim - 1; d >= 0; --d) {
            const long long id = rem / st[d];
            rem -= id * st[d];
            if (id >= gp.nodes[d] + 2) ok = false;
            spl_uni_row((int)id, gp.nodes[d], j0[d], w0[d], j1[d], w1[d]);
        }
        double v = 0.0;
        if (ok) {
            for (int m = 0; m < (1 << gp.ndim); ++m) {
                double w = 1.0;
                long long src = 0;
                for (int d = 0; d < gp.ndim; ++d) {
                    const bool second = (m >> d) & 1;
                    w *= second ? w1[d] : w0[d];
                    src += (second ? j1[d] : j0[d]) * mulv[d];
                }
                if (w != 0.0) v = fma(w, (double)coef[src], v);
            }
        }
        ext[e] = (TO)v;
    }
}

// ORDER > 0: the derivative sets, out(ncomp, nq), as spl_eval_kernel
template <int NDIM, bool VALUE, int NWARPS = RegroupCfg<NDIM>::NWARPS, bool UNI = false, int ORDER = 0>
__global__ void __launch_bounds__(NWARPS * 32, 1)
spl_eval_regroup_kernel(const __grid_constant__ GridParams gp, const DerivParams dp, const TableLayout tl,
                        const real_t *__restrict__ x, int l1x, long long nq,
                        const double *__restrict__ coef_padded, unsigned table_doubles, int cap,
                        real_t *__restrict__ out, const int *__restrict__ order_flag) {
    constexpr int NC = ORDER > 0 ? spl_ncomp(NDIM, ORDER) : 1;
    extern __shared__ __align__(128) double s_dyn[];
    __shared__ __align__(8) uint64_t mbar;
    __shared__ unsigned s_chunk;
    __shared__ double s_dscale[NC];
    // order_flag (spl_eval_probe_kernel): 0 = the batch arrives in coherent runs and the plain kernel evaluates it
    if (order_flag && *order_flag == 0) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if constexpr (ORDER > 0 && UNI)
        if (tid < NC) s_dscale[tid] = spl_uni_dscale<NDIM, ORDER>(gp, tid);
    if (tid == 0) {
        s_chunk = 0;
        mbar_init(&mbar, 1);
        mbar_fence_init();
        mbar_expect_tx(&mbar, table_doubles * (unsigned)sizeof(double));
        bulk_g2s(s_dyn, coef_padded, table_doubles * (unsigned)sizeof(double), &mbar);
    }
    __syncthreads();
    mbar_wait(&mbar, 0);
    const double *cf = s_dyn;
    // warp-private FIFOs: fx[d][slot][class] (doubles: the coordinates, or their fractional parts in the uniform form),
    // then per (slot, class) the query's offset inside the CTA's range (exact form: 4 bytes) or the pair
    // (window base offset | out-of-range flag, query offset) (uniform form: 8 bytes)
    const int per_warp = cap * 16 * NDIM + (UNI ? cap * 16 : cap * 8);
    double *fx = s_dyn + table_doubles + (size_t)warp * per_warp;
    unsigned *ftag = reinterpret_cast<unsigned *>(fx + cap * 16 * NDIM);
    uint2 *fbt = reinterpret_cast<uint2 *>(fx + cap * 16 * NDIM);
    const double uscale = UNI ? spl_uni_scale<NDIM>(gp, dp, VALUE) : 1.0;

    // this CTA's contiguous range of queries (offsets inside it fit 32 bits: checked by the launcher)
    const long long q_lo = nq * (long long)blockIdx.x / (long long)gridDim.x;
    const long long q_hi = nq * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
    const unsigned range = (unsigned)(q_hi - q_lo);
    const real_t *xb = x + q_lo * (long long)l1x;
    real_t *ob = out + q_lo * NC;

    const unsigned full = 0xffffffffu, lt = (1u << lane) - 1u;
    const int dc = lane & 15, hf = lane >> 4;                        // dedicated class, half-warp
    int stride16[NDIM];                                              // table strides mod 16
    stride16[0] = 1;
    if (NDIM > 1) stride16[1] = tl.s1 & 15;
    if (NDIM > 2) stride16[2] = tl.s2 & 15;
    if (NDIM > 3) stride16[NDIM - 1] = (int)(tl.s3 & 15);
    int head = 0, cnt = 0;                                           // FIFO cursor of class dc (same in both halves)
    bool pend = false;                                               // this lane holds a raw query not yet in a FIFO
    double px[NDIM];
    unsigned ptag = 0;
    unsigned cpos = 0, cend = 0;                                     // warp-uniform: the warp's current chunk
    bool done = false;                                               // warp-uniform: the CTA's range is exhausted
#pragma unroll
    for (int d = 0; d < NDIM; ++d) px[d] = 0.0;

    // lanes without a pending query take the next raw queries of the warp's chunk (loads consumed one round later)
    auto refill = [&]() {
        const unsigned nm = __ballot_sync(full, !pend);
        if (done || nm == 0u) return;
        if (cpos == cend) {
            unsigned c = 0;
            if (lane == 0) c = atomicAdd(&s_chunk, 1u);
            c = __shfl_sync(full, c, 0);
            const unsigned long long b0 = (unsigned long long)c * RG_CHUNK;
            if (b0 >= (unsigned long long)range) {
                done = true;
                return;
            }
            cpos = (unsigned)b0;
            cend = (range - cpos < RG_CHUNK) ? range : cpos + RG_CHUNK;
        }
        const unsigned my = cpos + (unsigned)__popc(nm & lt);
        if (!pend && my < cend) {
            ptag = my;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) px[d] = (double)xb[(long long)my * l1x + d];
            pend = true;
        }
        const unsigned adv = cpos + (unsigned)__popc(nm);
        cpos = adv < cend ? adv : cend;
    };

    refill();
    for (;;) {
        // ---- insert: bank class of the pending query = its base address in the table mod 16 ----
        int cls = 0;
        unsigned pbase = 0u;                                         // uniform form: base offset | out-of-range flag
        double pf[NDIM];                                             // what goes into the FIFO
#pragma unroll
        for (int d = 0; d < NDIM; ++d) pf[d] = px[d];
        if (pend) {
            if (UNI) {
                pbase = spl_uni_locate<NDIM>(gp, tl, px, pf);
                cls = (int)(pbase & 15u);
            } else {
                int lin = 0;
#pragma unroll
                for (int d = 0; d < NDIM; ++d) {
                    const double t = spl_mul(gp.dxin[d], spl_sub(px[d], gp.xmin[d]));
                    const int it = max(__double2int_rz(t), -4);
                    const int ws = min(max(it - 1, 0), gp.nodes[d] - 4);
                    lin += ws * stride16[d];
                }
                cls = lin & 15;
            }
        }
        const unsigned bp = __ballot_sync(full, pend);
        const unsigned v0 = __ballot_sync(full, pend && (cls & 1));
        const unsigned v1 = __ballot_sync(full, pend && (cls & 2));
        const unsigned v2 = __ballot_sync(full, pend && (cls & 4));
        const unsigned v3 = __ballot_sync(full, pend && (cls & 8));
        const unsigned peers = bp & ((cls & 1) ? v0 : ~v0) & ((cls & 2) ? v1 : ~v1) & ((cls & 4) ? v2 : ~v2) &
                               ((cls & 8) ? v3 : ~v3);              // pending lanes of my query's class
        const unsigned arr = bp & ((dc & 1) ? v0 : ~v0) & ((dc & 2) ? v1 : ~v1) & ((dc & 4) ? v2 : ~v2) &
                             ((dc & 8) ? v3 : ~v3);                  // pending lanes of my DEDICATED class
        const int big = __reduce_max_sync(full, pend ? __popc(peers) : 0);
        bool take = false;
        double ex[NDIM];
        unsigned etag = 0, ebase = 0u;
#pragma unroll
        for (int d = 0; d < NDIM; ++d) ex[d] = 0.0;
        if (big >= RG_BYPASS) {
            // coherent batch (raster order): the lanes evaluate their own queries, the gathers broadcast
            take = pend;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) ex[d] = pf[d];
            etag = ptag;
            ebase = pbase;
            pend = false;
        } else {
            const int st = __shfl_sync(full, (head << 8) | cnt, cls);           // cursor of my query's class
            const int qh = st >> 8, qc = st & 255;
            const int rank = __popc(peers & lt);
            if (pend && qc + rank < cap) {
                int slot = qh + qc + rank;
                if (slot >= cap) slot -= cap;
#pragma unroll
                for (int d = 0; d < NDIM; ++d) fx[(d * cap + slot) * 16 + cls] = pf[d];
                if (UNI) fbt[slot * 16 + cls] = make_uint2(pbase, ptag);
                else ftag[slot * 16 + cls] = ptag;
                pend = false;
            }
            cnt += min(__popc(arr), cap - cnt);
            __syncwarp();
            // ---- pop: one query of my class (two per class and round: one per half-warp) ----
            take = cnt > hf;
            if (take) {
                int slot = head + hf;
                if (slot >= cap) slot -= cap;
#pragma unroll
                for (int d = 0; d < NDIM; ++d) ex[d] = fx[(d * cap + slot) * 16 + dc];
                if (UNI) {
                    const uint2 bt = fbt[slot * 16 + dc];
                    ebase = bt.x;
                    etag = bt.y;
                } else {
                    etag = ftag[slot * 16 + dc];
                }
            }
            const int n = min(cnt, 2);
            head += n;
            if (head >= cap) head -= cap;
            cnt -= n;
            __syncwarp();
        }
        refill();
        if constexpr (ORDER > 0) {
            if (take) {
                if (UNI) spl_eval_derivs_uni_at<NDIM, ORDER>(tl, cf, ex, ebase, s_dscale, ob + (size_t)etag * NC);
                else spl_eval_derivs_point<NDIM, ORDER>(gp, tl, cf, ex, ob + (size_t)etag * NC);
            }
        } else if (take) {
            if (UNI) ob[etag] = (real_t)spl_eval_point_uni_at<NDIM, VALUE>(dp, tl, cf, ex, ebase, uscale);
            else ob[etag] = (real_t)spl_eval_point<NDIM, VALUE>(gp, dp, tl, cf, ex);
        }
        if (done && !__any_sync(full, pend || cnt > 0)) break;
    }
}

// Padded table strides for the regrouping kernel: the class (base address mod 16) of a query must be uniformly
// distributed, or the dedicated lanes of the hot classes limit the throughput to 1 / (16 p_max).  For window starts
// distributed as for uniformly scattered data, the class distribution is the cyclic convolution of the per-dimension
// ones; a small search over the paddings picks the flattest.  Cached for the last grid seen.
struct RegroupPlan {
    bool ok = false;
    TableLayout tl;
    long long table_doubles = 0;
    int cap = 0, nwarps = 0;
    size_t smem = 0;
    int key_ndim = 0, key_nodes[SPL_MAXDIM] = {0, 0, 0, 0}, key_warps = 0;
    size_t key_smem = 0;
};
// uni: the table is the extended one of the uniform form (nodes + 2 per dimension, window base = cell index)
static double class_pmax(const GridParams &gp, const long long *st, bool uni, int ncls = 16) {
    double dist[32] = {1.0};
    for (int c = 1; c < 32; ++c) dist[c] = 0.0;
    const int msk = ncls - 1;
    for (int d = 0; d < gp.ndim; ++d) {
        double pd[32] = {0.0};
        const int nod = gp.nodes[d];
        for (int it = 0; it < nod - 1; ++it) {
            int ws = uni ? it : it - 1;
            if (!uni) {
                if (ws < 0) ws = 0;
                if (ws > nod - 4) ws = nod - 4;
            }
            pd[(int)((ws * (st[d] & msk)) & msk)] += 1.0 / (double)(nod - 1);
        }
        double nx[32] = {0.0};
        for (int a = 0; a < ncls; ++a)
            for (int b = 0; b < ncls; ++b) nx[(a + b) & msk] += dist[a] * pd[b];
        for (int c = 0; c < ncls; ++c) dist[c] = nx[c];
    }
    double m = 0.0;
    for (int c = 0; c < ncls; ++c) m = dist[c] > m ? dist[c] : m;
    return m;
}
// warps per CTA of the regrouping kernel (SPLPAK_B200_RG_WARPS = 16 | 24 | 32 overrides the default for experiments)
static int regroup_warps(int ndim, bool uni, int order) {
    if (order == 1) return ndim == 2 ? RegroupCfg<2, 1>::NWARPS : (ndim == 3 ? RegroupCfg<3, 1>::NWARPS : RegroupCfg<4, 1>::NWARPS);
    if (order == 2) return ndim == 2 ? RegroupCfg<2, 2>::NWARPS : (ndim == 3 ? RegroupCfg<3, 2>::NWARPS : RegroupCfg<4, 2>::NWARPS);
    int nw = ndim == 2 ? RegroupCfg<2>::NWARPS : (ndim == 3 ? RegroupCfg<3>::NWARPS : RegroupCfg<4>::NWARPS);
    // uniform form, 3-D: the larger extended table leaves less room for the FIFOs; 16 warps keep them 9 deep
    // (measured 8 / 12 / 16 / 24 / 32 warps: 28.4 / 24.2 / 22.9 / 24.3 / 24.1 ms per 1e9 scattered queries)
    if (ndim == 3 && uni) nw = 16;
    if (const char *e = getenv("SPLPAK_B200_RG_WARPS")) {
        const int v = atoi(e);
        if (ndim == 3 && (v == 8 || v == 12 || v == 16 || v == 24 || v == 32)) nw = v;
    }
    return nw;
}
// f32: the float kernel of the REAL32 library (uniform form only): 4-byte table entries, 32 bank classes, one FIFO
// column per lane.  order: 0 = single-component evaluation, 1 / 2 = the derivative-set kernels (their own warp counts,
// so a plan per order is cached and alternating value and derivative calls do not redo the search)
static const RegroupPlan &regroup_plan(const GridParams &gp, size_t smem_optin, bool uni, bool f32 = false, int order = 0) {
    static thread_local RegroupPlan plans[7];
    RegroupPlan &plan = plans[f32 ? 6 : 2 * order + (uni ? 1 : 0)];
    const int nwarps = f32 ? 16 : regroup_warps(gp.ndim, uni, order);
    bool same = plan.key_ndim == gp.ndim && plan.key_smem == smem_optin && plan.key_warps == nwarps;
    for (int d = 0; d < SPL_MAXDIM && same; ++d) same = plan.key_nodes[d] == gp.nodes[d];
    if (same) return plan;
    plan = RegroupPlan();
    plan.key_ndim = gp.ndim;
    plan.key_smem = smem_optin;
    plan.key_warps = nwarps;
    for (int d = 0; d < SPL_MAXDIM; ++d) plan.key_nodes[d] = gp.nodes[d];
    if (gp.ndim < 2) return plan;
    const int ext = uni ? 2 : 0;
    const long long n0 = gp.nodes[0] + ext, n1 = gp.nodes[1] + ext, n2 = gp.ndim > 2 ? gp.nodes[2] + ext : 1,
                    n3 = gp.ndim > 3 ? gp.nodes[3] + ext : 1;
    const size_t reserve = 1024;                                       // static shared memory + alignment
    const int ncls = f32 ? 32 : 16;
    const size_t esz = f32 ? sizeof(float) : sizeof(double);
    const size_t per_slot = f32 ? (size_t)nwarps * 32 * (4 * gp.ndim + 8)
                                : (size_t)nwarps * 16 * (8 * gp.ndim + (uni ? 8 : 4));   // bytes of FIFO per unit of cap
    double best = 1e30;
    const int r1 = gp.ndim == 4 ? 4 : 8, r2 = f32 ? (gp.ndim == 4 ? 16 : 32) : (gp.ndim == 4 ? 8 : 16);
    for (long long s1 = n0; s1 < n0 + r1; ++s1)
        for (long long s2 = s1 * n1; s2 < s1 * n1 + (gp.ndim > 2 ? r2 : 1); ++s2)
            for (long long s3 = s2 * n2; s3 < s2 * n2 + (gp.ndim > 3 ? (f32 ? 32 : 16) : 1); ++s3) {
                long long total = gp.ndim == 2 ? s1 * n1 : (gp.ndim == 3 ? s2 * n2 : s3 * n3);
                total = f32 ? ((total + 3) & ~3LL) : ((total + 1) & ~1LL);
                const size_t tbytes = (size_t)total * esz;
                if (tbytes + reserve + 4 * per_slot > smem_optin || total >= (1LL << 28)) continue;
                const long long st[4] = {1, s1, s2, s3};
                const double pm = class_pmax(gp, st, uni, ncls);
                long long cap = (long long)((smem_optin - reserve - tbytes) / per_slot);
                if (cap > 24) cap = 24;
                // estimated lane efficiency: the hottest class bounds it; short FIFOs lose a little more
                const double eff = (1.0 / ((double)ncls * pm)) * (1.0 - 0.6 / (double)cap);
                const double score = -eff;
                if (score < best) {
                    best = score;
                    plan.ok = true;
                    plan.tl.s1 = (int)s1;
                    plan.tl.s2 = (int)s2;
                    plan.tl.s3 = s3;
                    plan.table_doubles = total;
                    plan.cap = (int)cap;
                    plan.nwarps = nwarps;
                    plan.smem = tbytes + (size_t)cap * per_slot;
                }
            }
    return plan;
}

static TableLayout natural_layout(const GridParams &gp, int ext) {
    TableLayout tl;
    tl.s1 = gp.nodes[0] + ext;
    tl.s2 = tl.s1 * (gp.ndim > 1 ? gp.nodes[1] + ext : 1);
    tl.s3 = (long long)tl.s2 * (gp.ndim > 2 ? gp.nodes[2] + ext : 1);
    return tl;
}
static long long natural_doubles(const GridParams &gp, int ext) {
    long long t = 1;
    for (int d = 0; d < gp.ndim; ++d) t *= gp.nodes[d] + ext;
    return (t + 1) & ~1LL;
}

// How a batch is evaluated (decided once on the host, the same way by the scratch sizing and by the launcher):
//   uni      uniform (phantom-node) form: extended table in shared memory, 9-operation basis (basis.cuh).  Chosen for
//            every batch large enough to pay for the table transform whose extended table fits in shared memory and
//            whose nderiv is valid (0..2); SPLPAK_B200_BASIS=exact forces the node-by-node formulas of bascmp.
//   regroup  scattered-order kernel with warp-private bank-class FIFOs (+ order probe unless forced)
struct EvalRoute {
    bool uni = false, regroup = false, force_regroup = false;
    TableLayout tl;                 // layout of the table the kernels read (extended and/or padded)
    long long table_doubles = 0;    // its size; 0: the caller's table is read directly
};
static EvalRoute eval_route(const GridParams &gp, const int *nderiv, long long nq, int nsm, size_t smem_optin) {
    EvalRoute r;
    r.tl = natural_layout(gp, 0);
    const char *mode = getenv("SPLPAK_B200_EVAL");
    const char *basis = getenv("SPLPAK_B200_BASIS");
    const bool plain_only = mode && strcmp(mode, "plain") == 0;
    r.force_regroup = mode && strcmp(mode, "regroup") == 0;
    bool valid = true;
    for (int d = 0; d < gp.ndim; ++d)
        if (nderiv && (nderiv[d] < 0 || nderiv[d] > 2)) valid = false;
    const long long ext_doubles = natural_doubles(gp, 2);
    const bool force_uni = basis && strcmp(basis, "uniform") == 0;
    bool uni = valid && !(basis && strcmp(basis, "exact") == 0) && (size_t)ext_doubles * 8 + 2048 <= smem_optin &&
               (force_uni || nq * (long long)spl_ipow(4, gp.ndim) * 16 > ext_doubles);
    // measured (profiles/r02_eval_ab.md): 3-D 45.5 -> 30.0 ms and 4-D 201 -> 84 ms per 1e9 random queries; 2-D gathers only
    // 16 values per query and is faster in the plain kernel (12.1 vs 17.2 ms), so it regroups only when forced
    // uniform form (profiles/r02_eval_uniform.md): 2-D scattered 10.2 (regrouped) vs 11.9 ms (plain), so 2-D regroups as well
    bool rg = !plain_only && gp.ndim >= 2 && (r.force_regroup || ((gp.ndim >= 3 || uni) && nq >= (1LL << 18))) &&
              nq / (nsm > 0 ? nsm : 1) < (1LL << 32) - 1024;
    if (rg) {
        const RegroupPlan &pl = regroup_plan(gp, smem_optin, uni);
        if (pl.ok) {
            r.regroup = true;
            r.tl = pl.tl;
            r.table_doubles = pl.table_doubles;
        } else if (uni) {
            // the extended table leaves no room for the FIFOs: scattered batches keep the exact form if that regroups
            const RegroupPlan &pe = regroup_plan(gp, smem_optin, false);
            if (pe.ok) {
                uni = false;
                r.regroup = true;
                r.tl = pe.tl;
                r.table_doubles = pe.table_doubles;
            }
        }
    }
    r.uni = uni;
    if (uni && !r.regroup) {
        r.tl = natural_layout(gp, 2);
        r.table_doubles = ext_doubles;
    }
    return r;
}
// derivative sets of order 1 / 2: the same decisions as a single-component batch -- in particular the same basis form,
// so that every component is bit-identical to it -- with the regrouping plan of the derivative kernels; when that plan
// does not fit, the plain kernel in the SAME form
static EvalRoute eval_route_derivs(const GridParams &gp, int order, long long nq, int nsm, size_t smem_optin) {
    EvalRoute r = eval_route(gp, nullptr, nq, nsm, smem_optin);
    if (!r.regroup) return r;
    const RegroupPlan &pl = regroup_plan(gp, smem_optin, r.uni, false, order);
    if (pl.ok) {
        r.tl = pl.tl;
        r.table_doubles = pl.table_doubles;
        return r;
    }
    r.regroup = r.force_regroup = false;
    r.tl = natural_layout(gp, r.uni ? 2 : 0);
    r.table_doubles = r.uni ? natural_doubles(gp, 2) : 0;
    return r;
}

// doubles of device scratch the evaluation of this batch needs behind the caller's table (+ 2 for the order flag): the
// extended and/or padded copy of the table.  0: none.  order 1 / 2: the derivative sets (nderiv unused)
long long spl_eval_scratch_elems(const GridParams &gp, const int *nderiv, int order, long long nq, int nsm,
                                 size_t smem_optin) {
    if (order > 0) return eval_route_derivs(gp, order, nq, nsm, smem_optin).table_doubles;
    return eval_route(gp, nderiv, nq, nsm, smem_optin).table_doubles;
}
// the exact-form regrouping kernel alone (REAL32 library, 4-D): 0 or the number of doubles of its padded table
long long spl_eval_regroup_elems(const GridParams &gp, long long nq, int nsm, size_t smem_optin) {
    const char *mode = getenv("SPLPAK_B200_EVAL");
    if (mode && strcmp(mode, "plain") == 0) return 0;
    const bool force = mode && strcmp(mode, "regroup") == 0;
    if (gp.ndim < 2 || (!force && (gp.ndim < 3 || nq < (1LL << 18)))) return 0;
    if (nq / (nsm > 0 ? nsm : 1) >= (1LL << 32) - 1024) return 0;
    const RegroupPlan &pl = regroup_plan(gp, smem_optin, false);
    return pl.ok ? pl.table_doubles : 0;
}

// table image for the kernels: padded copy (exact form) or extended table (uniform form)
static void launch_table(const GridParams &gp, const TableLayout &tl, long long total, bool uni, const double *d_coef,
                         double *d_tab, cudaStream_t stream) {
    long long blocks = (total + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    if (uni) spl_uni_table_kernel<double, double><<<(unsigned)blocks, 256, 0, stream>>>(gp, tl, d_coef, d_tab, total);
    else spl_pad_table_kernel<<<(unsigned)blocks, 256, 0, stream>>>(gp, tl, d_coef, d_tab, total);
    ++g_spl_launches;
}

// d_tab: the table image launch_table() made for this plan
template <int NDIM, bool VALUE, bool UNI, int ORDER = 0>
static int launch_eval_regroup(const GridParams &gp, const DerivParams &dp, const real_t *d_x, int l1x, long long nq,
                               const double *d_tab, real_t *d_out, cudaStream_t stream, int nsm,
                               size_t smem_optin, int *d_flag) {
    const RegroupPlan &pl = regroup_plan(gp, smem_optin, UNI, false, ORDER);
    if (d_flag) {
        spl_eval_probe_kernel<NDIM, UNI><<<1, 1024, 0, stream>>>(gp, pl.tl, d_x, l1x, nq, d_flag);
        ++g_spl_launches;
    }
    void (*kern)(GridParams, DerivParams, TableLayout, const real_t *, int, long long, const double *, unsigned, int,
                 real_t *, const int *) = spl_eval_regroup_kernel<NDIM, VALUE, RegroupCfg<NDIM, ORDER>::NWARPS, UNI, ORDER>;
    if constexpr (ORDER == 0) {
        if (NDIM == 3 && pl.nwarps == 8) kern = spl_eval_regroup_kernel<NDIM, VALUE, (NDIM == 3 ? 8 : RegroupCfg<NDIM>::NWARPS), UNI>;
        if (NDIM == 3 && pl.nwarps == 12) kern = spl_eval_regroup_kernel<NDIM, VALUE, (NDIM == 3 ? 12 : RegroupCfg<NDIM>::NWARPS), UNI>;
        if (NDIM == 3 && pl.nwarps == 16) kern = spl_eval_regroup_kernel<NDIM, VALUE, (NDIM == 3 ? 16 : RegroupCfg<NDIM>::NWARPS), UNI>;
        if (NDIM == 3 && pl.nwarps == 32) kern = spl_eval_regroup_kernel<NDIM, VALUE, (NDIM == 3 ? 32 : RegroupCfg<NDIM>::NWARPS), UNI>;
    }
    SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    long long grid = nsm;
    const long long per_cta_min = 4096;                 // tiny batches: fewer CTAs, each with a useful range
    if (grid > (nq + per_cta_min - 1) / per_cta_min) grid = (nq + per_cta_min - 1) / per_cta_min;
    if (grid < 1) grid = 1;
    kern<<<(unsigned)grid, pl.nwarps * 32, pl.smem, stream>>>(gp, dp, pl.tl, d_x, l1x, nq, d_tab,
                                                                             (unsigned)pl.table_doubles, pl.cap, d_out, d_flag);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

#ifdef SPLPAK_REAL32
// ------------------------------------------------------------------------------------------
// REAL32 library, splfe: the reference built with -DREAL32 computes in float, so this path does too -- float
// coordinates, float basis (spl_window_weights_value_f32, unfused: bit-identical 1-D values), float table in shared
// memory (half the bytes and half the crossbar wavefronts of the real64 gather), FFMA contraction on the FP32 pipe.
// Derivatives (splde) and the fit keep float I/O with float64 arithmetic.
// ------------------------------------------------------------------------------------------
template <int NDIM, bool SMEM>
__global__ void __launch_bounds__(1024, 1)
spl_eval_f32_kernel(const __grid_constant__ GridParams gp, const float *__restrict__ x, int l1x, long long nq,
                    const float *__restrict__ coef, long long ncol, float *__restrict__ out,
                    unsigned long long *__restrict__ chunk_counter, const int *__restrict__ order_flag) {
    extern __shared__ __align__(16) float s_tab[];
    // order_flag (spl_eval_probe_kernel, 4-D only): 1 = scattered batch, the float64 regrouping kernel evaluates it
    if (order_flag && *order_flag == 1) return;
    const int lane = threadIdx.x & 31;
    const float *cf = coef;
    if (SMEM) {
        for (long long e = threadIdx.x; e < ncol; e += blockDim.x) s_tab[e] = coef[e];
        __syncthreads();
        cf = s_tab;
    }
    TableLayout tl;
    tl.s1 = gp.nodes[0];
    tl.s2 = gp.nodes[0] * gp.nodes[1];
    tl.s3 = (long long)tl.s2 * gp.nodes[2];
    float xmin[NDIM], dx[NDIM], dxin[NDIM];
#pragma unroll
    for (int d = 0; d < NDIM; ++d) {
        xmin[d] = (float)gp.xmin[d];          // exact: GridParams holds the widened working-precision values
        dx[d] = (float)gp.dx[d];
        dxin[d] = (float)gp.dxin[d];
    }
    for (;;) {
        unsigned long long c = 0;
        if (lane == 0) c = atomicAdd(chunk_counter, 1ULL);
        c = __shfl_sync(0xffffffffu, c, 0);
        const long long base = (long long)c * EVAL_WCHUNK;
        if (base >= nq) break;
        float xn[NDIM];
        {
            const long long q = base + lane;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) xn[d] = (q < nq) ? x[q * (long long)l1x + d] : 0.0f;
        }
#pragma unroll 1
        for (int sub = 0; sub < EVAL_WCHUNK / 32; ++sub) {
            const long long q = base + sub * 32 + lane;
            float xv[NDIM];
#pragma unroll
            for (int d = 0; d < NDIM; ++d) xv[d] = xn[d];
            const long long q2 = q + 32;
            if (sub + 1 < EVAL_WCHUNK / 32) {
#pragma unroll
                for (int d = 0; d < NDIM; ++d) xn[d] = (q2 < nq) ? x[q2 * (long long)l1x + d] : 0.0f;
            }
            if (q < nq) {
                float b[NDIM][4];
                int ws[NDIM];
                bool isnan_q = false;
#pragma unroll
                for (int d = 0; d < NDIM; ++d) {
                    spl_window_weights_value_f32<true>(xv[d], xmin[d], dx[d], dxin[d], gp.nodes[d], ws[d], b[d]);
                    isnan_q |= (xv[d] != xv[d]);
                }
                float sum = spl_contract<NDIM, float>(tl, cf, ws, b) * (1.0f / (float)spl_ipow(8, NDIM));
                out[q] = isnan_q ? 0.0f : sum;
            }
        }
    }
}

template <int NDIM>
static int launch_eval_f32(const GridParams &gp, const float *d_x, int l1x, long long nq, const float *d_coef,
                           float *d_out, cudaStream_t stream, int nsm, size_t smem_optin, unsigned long long *d_counter,
                           const int *d_flag = nullptr) {
    SPL_CUDA_TRY(cudaMemsetAsync(d_counter, 0, sizeof(unsigned long long), stream));
    const size_t bytes = (size_t)gp.ncol * sizeof(float);
    const bool use_smem = bytes + 2048 <= smem_optin && nq * (long long)spl_ipow(4, NDIM) * 64 > gp.ncol;
    long long chunks = (nq + EVAL_WCHUNK - 1) / EVAL_WCHUNK;
    long long ctas = (chunks + 31) / 32;
    if (ctas < 1) ctas = 1;
    if (use_smem) {
        auto kern = spl_eval_f32_kernel<NDIM, true>;
        SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        // small tables leave room for two CTAs per SM
        long long grid = (long long)nsm * (bytes <= 100 * 1024 ? 2 : 1);
        if (grid > ctas) grid = ctas;
        kern<<<(unsigned)grid, 1024, bytes, stream>>>(gp, d_x, l1x, nq, d_coef, gp.ncol, d_out, d_counter, d_flag);
    } else {
        auto kern = spl_eval_f32_kernel<NDIM, false>;
        long long grid = (long long)nsm * 2;
        if (grid > ctas) grid = ctas;
        kern<<<(unsigned)grid, 1024, 0, stream>>>(gp, d_x, l1x, nq, d_coef, gp.ncol, d_out, d_counter, d_flag);
    }
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// splfe in working precision real32 (nderiv all zero).  d_coef: the caller's float table, ncol entries.
int spl_eval_f32_launch(const GridParams &gp, const real_t *d_x, int l1x, long long nq, const real_t *d_coef,
                        real_t *d_out, cudaStream_t stream, int nsm, size_t smem_optin, unsigned long long *d_counter) {
    if (nq <= 0) return SPLPAK_OK;
    switch (gp.ndim) {
    case 1: return launch_eval_f32<1>(gp, d_x, l1x, nq, d_coef, d_out, stream, nsm, smem_optin, d_counter);
    case 2: return launch_eval_f32<2>(gp, d_x, l1x, nq, d_coef, d_out, stream, nsm, smem_optin, d_counter);
    case 3: return launch_eval_f32<3>(gp, d_x, l1x, nq, d_coef, d_out, stream, nsm, smem_optin, d_counter);
    case 4: return launch_eval_f32<4>(gp, d_x, l1x, nq, d_coef, d_out, stream, nsm, smem_optin, d_counter);
    }
    return SPLPAK_ERR_NDIM;
}

// splfe of the REAL32 library in the uniform (phantom-node) form: extended FLOAT table in shared memory, float weights
// (9 FP32 operations per dimension) and FFMA contraction; only the cell index / fractional coordinate are formed in
// float64 from the float inputs (3 operations per dimension), so f carries no eps32 * node-index error.  CTA-static
// ranges, a whole chunk of coordinates per warp in flight (as spl_eval_kernel's 1-D / 2-D uniform loop).
template <int NDIM>
__global__ void __launch_bounds__(1024, 1)
spl_eval_uni_f32_kernel(const __grid_constant__ GridParams gp, const TableLayout tl, const float *__restrict__ x, int l1x,
                        long long nq, const float *__restrict__ ext, unsigned table_floats, float *__restrict__ out,
                        const int *__restrict__ order_flag) {
    extern __shared__ __align__(128) float s_ext[];
    __shared__ __align__(8) uint64_t mbar;
    if (order_flag && *order_flag == 1) return;
    const int tid = threadIdx.x, lane = tid & 31;
    if (tid == 0) {
        mbar_init(&mbar, 1);
        mbar_fence_init();
        mbar_expect_tx(&mbar, table_floats * (unsigned)sizeof(float));
        bulk_g2s(s_ext, ext, table_floats * (unsigned)sizeof(float), &mbar);
    }
    __syncthreads();
    mbar_wait(&mbar, 0);
    const float *cf = s_ext;
    constexpr int KQ = NDIM == 1 ? 8 : (NDIM == 2 ? 4 : 2);
    constexpr int CH = KQ * 32;
    const bool vec2 = NDIM == 2 && l1x == 2 && ((uintptr_t)x % 8 == 0);
    float cur[KQ][NDIM], nxt[KQ][NDIM];
    const long long q_lo = nq * (long long)blockIdx.x / (long long)gridDim.x;
    const long long q_hi = nq * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
    long long next_chunk = q_lo + (long long)(tid >> 5) * CH;
    auto claim = [&]() -> long long {
        const long long b = next_chunk;
        next_chunk += (long long)(blockDim.x >> 5) * CH;
        return b < q_hi ? b : -1;
    };
    auto issue = [&](long long b) {
        if (b < 0) return;
#pragma unroll
        for (int k = 0; k < KQ; ++k) {
            const long long q = b + k * 32 + lane;
            if (q < q_hi) {
                if (NDIM == 2 && vec2) {
                    const float2 v = reinterpret_cast<const float2 *>(x)[q];
                    nxt[k][0] = v.x;
                    nxt[k][NDIM - 1] = v.y;
                } else {
#pragma unroll
                    for (int d = 0; d < NDIM; ++d) nxt[k][d] = x[q * (long long)l1x + d];
                }
            } else {
#pragma unroll
                for (int d = 0; d < NDIM; ++d) nxt[k][d] = 0.0f;
            }
        }
    };
    const float scale = 1.0f / (float)spl_ipow(4, NDIM);
    long long nbase = claim();
    issue(nbase);
    while (nbase >= 0) {
        const long long cbase = nbase;
#pragma unroll
        for (int k = 0; k < KQ; ++k)
#pragma unroll
            for (int d = 0; d < NDIM; ++d) cur[k][d] = nxt[k][d];
        nbase = claim();
        issue(nbase);
#pragma unroll
        for (int k = 0; k < KQ; ++k) {
            const long long q = cbase + k * 32 + lane;
            if (q < q_hi) {
                float b[NDIM][4];
                unsigned base = 0u;
                bool isnan_q = false;
#pragma unroll
                for (int d = 0; d < NDIM; ++d) {
                    int cell;
                    double fd;
                    bool oob;
                    spl_uni_cell((double)cur[k][d], gp.xmin[d], gp.dxin[d], gp.nodes[d], cell, fd, oob);
                    spl_uni_weights_f32((float)fd, oob, b[d]);
                    isnan_q |= (cur[k][d] != cur[k][d]);
                    const unsigned st = d == 0 ? 1u : (d == 1 ? (unsigned)tl.s1 : (d == 2 ? (unsigned)tl.s2 : (unsigned)tl.s3));
                    base += (unsigned)cell * st;
                }
                const float sum = spl_contract_at<NDIM, float>(tl, cf + base, b) * scale;
                out[q] = isnan_q ? 0.0f : sum;
            }
        }
    }
}

// Regrouping kernel of the REAL32 library (uniform form, splfe): the float table has 4-byte entries, so a WARP-wide
// LDS.32 is conflict-free when its 32 lanes read 32 distinct banks -- 32 bank classes (window base mod 32), lane l
// DEDICATED to class l, one FIFO column per lane, one pop per lane and round.  Otherwise the scheme of
// spl_eval_regroup_kernel: warp-private FIFOs, ranks from ballots, cursors in registers, coherent batches bypass.
// Half the crossbar wavefronts per query of the float64 kernel (64 x 4 B = 2 instead of 4).
template <int NDIM, int NWARPS>
__global__ void __launch_bounds__(NWARPS * 32, 1)
spl_eval_regroup_f32_kernel(const __grid_constant__ GridParams gp, const TableLayout tl, const float *__restrict__ x, int l1x,
                            long long nq, const float *__restrict__ ext_padded, unsigned table_floats, int cap,
                            float *__restrict__ out, const int *__restrict__ order_flag) {
    extern __shared__ __align__(128) float s_ext[];
    __shared__ __align__(8) uint64_t mbar;
    __shared__ unsigned s_chunk;
    if (order_flag && *order_flag == 0) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        s_chunk = 0;
        mbar_init(&mbar, 1);
        mbar_fence_init();
        mbar_expect_tx(&mbar, table_floats * (unsigned)sizeof(float));
        bulk_g2s(s_ext, ext_padded, table_floats * (unsigned)sizeof(float), &mbar);
    }
    __syncthreads();
    mbar_wait(&mbar, 0);
    const float *cf = s_ext;
    // warp-private FIFOs: fbt[slot][class] = (window base | out-of-range flag, query offset) (8 bytes), then
    // ff[d][slot][class] = fractional coordinates (floats)
    const int per_warp = cap * 32 * (NDIM + 2);                     // floats
    float *wbase = s_ext + table_floats + (size_t)warp * per_warp;
    uint2 *fbt = reinterpret_cast<uint2 *>(wbase);
    float *ff = wbase + cap * 64;
    const float scale = 1.0f / (float)spl_ipow(4, NDIM);

    const long long q_lo = nq * (long long)blockIdx.x / (long long)gridDim.x;
    const long long q_hi = nq * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
    const unsigned range = (unsigned)(q_hi - q_lo);
    const float *xb = x + q_lo * (long long)l1x;
    float *ob = out + q_lo;

    const unsigned full = 0xffffffffu, lt = (1u << lane) - 1u;
    int head = 0, cnt = 0;                                           // FIFO cursor of class `lane`
    bool pend = false;
    float px[NDIM];
    unsigned ptag = 0;
    unsigned cpos = 0, cend = 0;
    bool done = false;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) px[d] = 0.0f;

    auto refill = [&]() {
        const unsigned nm = __ballot_sync(full, !pend);
        if (done || nm == 0u) return;
        if (cpos == cend) {
            unsigned c = 0;
            if (lane == 0) c = atomicAdd(&s_chunk, 1u);
            c = __shfl_sync(full, c, 0);
            const unsigned long long b0 = (unsigned long long)c * RG_CHUNK;
            if (b0 >= (unsigned long long)range) {
                done = true;
                return;
            }
            cpos = (unsigned)b0;
            cend = (range - cpos < RG_CHUNK) ? range : cpos + RG_CHUNK;
        }
        const unsigned my = cpos + (unsigned)__popc(nm & lt);
        if (!pend && my < cend) {
            ptag = my;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) px[d] = xb[(long long)my * l1x + d];
            pend = true;
        }
        const unsigned adv = cpos + (unsigned)__popc(nm);
        cpos = adv < cend ? adv : cend;
    };

    refill();
    for (;;) {
        int cls = 0;
        unsigned pbase = 0u;
        float pf[NDIM];
#pragma unroll
        for (int d = 0; d < NDIM; ++d) pf[d] = 0.0f;
        if (pend) {
            bool any = false;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) {
                int cell;
                double fd;
                bool oob;
                spl_uni_cell((double)px[d], gp.xmin[d], gp.dxin[d], gp.nodes[d], cell, fd, oob);
                pf[d] = (px[d] != px[d]) ? px[d] : (float)fd;        // NaN stays NaN
                any |= oob;
                const unsigned st = d == 0 ? 1u : (d == 1 ? (unsigned)tl.s1 : (d == 2 ? (unsigned)tl.s2 : (unsigned)tl.s3));
                pbase += (unsigned)cell * st;
            }
            cls = (int)(pbase & 31u);
            if (any) pbase |= SPL_UNI_OOB;
        }
        const unsigned bp = __ballot_sync(full, pend);
        const unsigned v0 = __ballot_sync(full, pend && (cls & 1));
        const unsigned v1 = __ballot_sync(full, pend && (cls & 2));
        const unsigned v2 = __ballot_sync(full, pend && (cls & 4));
        const unsigned v3 = __ballot_sync(full, pend && (cls & 8));
        const unsigned v4 = __ballot_sync(full, pend && (cls & 16));
        const unsigned peers = bp & ((cls & 1) ? v0 : ~v0) & ((cls & 2) ? v1 : ~v1) & ((cls & 4) ? v2 : ~v2) &
                               ((cls & 8) ? v3 : ~v3) & ((cls & 16) ? v4 : ~v4);
        const unsigned arr = bp & ((lane & 1) ? v0 : ~v0) & ((lane & 2) ? v1 : ~v1) & ((lane & 4) ? v2 : ~v2) &
                             ((lane & 8) ? v3 : ~v3) & ((lane & 16) ? v4 : ~v4);
        const int big = __reduce_max_sync(full, pend ? __popc(peers) : 0);
        bool take = false;
        float ex[NDIM];
        unsigned etag = 0, ebase = 0u;
#pragma unroll
        for (int d = 0; d < NDIM; ++d) ex[d] = 0.0f;
        if (big >= RG_BYPASS) {
            take = pend;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) ex[d] = pf[d];
            etag = ptag;
            ebase = pbase;
            pend = false;
        } else {
            const int st = __shfl_sync(full, (head << 8) | cnt, cls);
            const int qh = st >> 8, qc = st & 255;
            const int rank = __popc(peers & lt);
            if (pend && qc + rank < cap) {
                int slot = qh + qc + rank;
                if (slot >= cap) slot -= cap;
#pragma unroll
                for (int d = 0; d < NDIM; ++d) ff[(d * cap + slot) * 32 + cls] = pf[d];
                fbt[slot * 32 + cls] = make_uint2(pbase, ptag);
                pend = false;
            }
            cnt += min(__popc(arr), cap - cnt);
            __syncwarp();
            take = cnt > 0;
            if (take) {
#pragma unroll
                for (int d = 0; d < NDIM; ++d) ex[d] = ff[(d * cap + head) * 32 + lane];
                const uint2 bt = fbt[head * 32 + lane];
                ebase = bt.x;
                etag = bt.y;
                head = (head + 1 >= cap) ? 0 : head + 1;
                --cnt;
            }
            __syncwarp();
        }
        refill();
        if (take) {
            float b[NDIM][4];
            bool isnan_q = false;
            const bool oob = (ebase & SPL_UNI_OOB) != 0u;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) {
                spl_uni_weights_f32(ex[d], oob, b[d]);
                isnan_q |= (ex[d] != ex[d]);
            }
            const float sum = spl_contract_at<NDIM, float>(tl, cf + (ebase & ~SPL_UNI_OOB), b) * scale;
            ob[etag] = isnan_q ? 0.0f : sum;
        }
        if (done && !__any_sync(full, pend || cnt > 0)) break;
    }
}

// How the REAL32 library evaluates a splfe batch in the uniform form (decided the same way by the scratch sizing and
// by the launcher): extended float table in natural layout (plain kernel alone), or padded for the 32-class regrouping
// kernel (order probe + both kernels, as the float64 path; SPLPAK_B200_EVAL=plain|regroup overrides).
struct EvalRouteF32 {
    bool ok = false, regroup = false, force_regroup = false;
    TableLayout tl;
    long long table_floats = 0;
};
static EvalRouteF32 eval_route_f32(const GridParams &gp, long long nq, int nsm, size_t smem_optin) {
    EvalRouteF32 r;
    const char *basis = getenv("SPLPAK_B200_BASIS");
    const char *mode = getenv("SPLPAK_B200_EVAL");
    if (basis && strcmp(basis, "exact") == 0) return r;
    const long long ext = natural_doubles(gp, 2);                  // entries (rounded up to even)
    const long long ext4 = (ext + 3) & ~3LL;                       // bulk copies move multiples of 16 bytes
    if ((size_t)ext4 * sizeof(float) + 2048 > smem_optin) return r;
    if (!(basis && strcmp(basis, "uniform") == 0) && nq * (long long)spl_ipow(4, gp.ndim) * 16 <= ext) return r;
    r.ok = true;
    r.tl = natural_layout(gp, 2);
    r.table_floats = ext4;
    const bool plain_only = mode && strcmp(mode, "plain") == 0;
    r.force_regroup = mode && strcmp(mode, "regroup") == 0;
    // measured per 1e9 scattered float queries, plain vs regrouped: 2-D 6.6 vs 13.5 ms (regroups only when forced),
    // 3-D 25.2 vs 17.8 ms, 4-D 82.7 (float64 regrouping kernel) vs 46.4 ms
    if (!plain_only && gp.ndim >= 2 && (r.force_regroup || (gp.ndim >= 3 && nq >= (1LL << 18))) &&
        nq / (nsm > 0 ? nsm : 1) < (1LL << 32) - 1024) {
        const RegroupPlan &pl = regroup_plan(gp, smem_optin, true, true);
        if (pl.ok) {
            r.regroup = true;
            r.tl = pl.tl;
            r.table_floats = pl.table_doubles;
        }
    }
    return r;
}
// floats of scratch the uniform float path needs for this batch (table image + 4 for the order flag); 0: not applicable
long long spl_eval_uni_f32_elems(const GridParams &gp, long long nq, int nsm, size_t smem_optin) {
    const EvalRouteF32 r = eval_route_f32(gp, nq, nsm, smem_optin);
    return r.ok ? r.table_floats + 4 : 0;
}

template <int NDIM>
static int launch_eval_uni_f32(const GridParams &gp, const EvalRouteF32 &rt, const float *d_x, int l1x, long long nq,
                               const float *d_coef, float *d_ext, float *d_out, cudaStream_t stream, int nsm,
                               size_t smem_optin) {
    {
        long long blocks = (rt.table_floats + 255) / 256;
        if (blocks > 1024) blocks = 1024;
        spl_uni_table_kernel<float, float><<<(unsigned)blocks, 256, 0, stream>>>(gp, rt.tl, d_coef, d_ext, rt.table_floats);
        ++g_spl_launches;
    }
    int *d_flag = nullptr;
    if (rt.regroup) {
        if constexpr (NDIM >= 2) {
            const RegroupPlan &pl = regroup_plan(gp, smem_optin, true, true);
            if (!rt.force_regroup) {
                d_flag = reinterpret_cast<int *>(d_ext + rt.table_floats);
                spl_eval_probe_kernel<NDIM, true, 32><<<1, 1024, 0, stream>>>(gp, pl.tl, d_x, l1x, nq, d_flag);
                ++g_spl_launches;
            }
            auto kern = spl_eval_regroup_f32_kernel<NDIM, 16>;
            SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
            long long grid = nsm;
            const long long per_cta_min = 4096;
            if (grid > (nq + per_cta_min - 1) / per_cta_min) grid = (nq + per_cta_min - 1) / per_cta_min;
            if (grid < 1) grid = 1;
            kern<<<(unsigned)grid, 16 * 32, pl.smem, stream>>>(gp, pl.tl, d_x, l1x, nq, d_ext, (unsigned)pl.table_doubles, pl.cap,
                                                               d_out, d_flag);
            ++g_spl_launches;
            SPL_CUDA_TRY(cudaGetLastError());
            if (rt.force_regroup) return SPLPAK_OK;
        }
    }
    auto kern = spl_eval_uni_f32_kernel<NDIM>;
    const size_t bytes = (size_t)rt.table_floats * sizeof(float);
    SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    long long grid = nsm;
    const long long per_cta_min = 8192;
    if (grid > (nq + per_cta_min - 1) / per_cta_min) grid = (nq + per_cta_min - 1) / per_cta_min;
    if (grid < 1) grid = 1;
    kern<<<(unsigned)grid, 1024, bytes, stream>>>(gp, rt.tl, d_x, l1x, nq, d_ext, (unsigned)rt.table_floats, d_out, d_flag);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// d_ext: scratch of spl_eval_uni_f32_elems() floats
int spl_eval_uni_f32_launch(const GridParams &gp, const real_t *d_x, int l1x, long long nq, const real_t *d_coef,
                            real_t *d_ext, real_t *d_out, cudaStream_t stream, int nsm, size_t smem_optin) {
    if (nq <= 0) return SPLPAK_OK;
    const EvalRouteF32 rt = eval_route_f32(gp, nq, nsm, smem_optin);
    if (!rt.ok) return SPLPAK_ERR_HANDLE;
    switch (gp.ndim) {
    case 1: return launch_eval_uni_f32<1>(gp, rt, d_x, l1x, nq, d_coef, d_ext, d_out, stream, nsm, smem_optin);
    case 2: return launch_eval_uni_f32<2>(gp, rt, d_x, l1x, nq, d_coef, d_ext, d_out, stream, nsm, smem_optin);
    case 3: return launch_eval_uni_f32<3>(gp, rt, d_x, l1x, nq, d_coef, d_ext, d_out, stream, nsm, smem_optin);
    case 4: return launch_eval_uni_f32<4>(gp, rt, d_x, l1x, nq, d_coef, d_ext, d_out, stream, nsm, smem_optin);
    }
    return SPLPAK_ERR_NDIM;
}

// 4-D splfe of the REAL32 library, large batches: the float table has no regrouping variant, and for SCATTERED queries
// the float64 regrouping kernel is faster than the float plain kernel (83.8 vs 117 ms per 1e9), while coherent batches
// are faster in float (35.6 vs 56.9 ms).  So: order probe, then both -- the flag makes the wrong one exit at once.
// d_coef64 / d_pad: the table widened to float64 and the padded-table scratch (+ 2 doubles for the flag).
int spl_eval_f32_mixed4_launch(const GridParams &gp, const real_t *d_x, int l1x, long long nq, const real_t *d_coef,
                               const double *d_coef64, double *d_pad, real_t *d_out, cudaStream_t stream, int nsm,
                               size_t smem_optin, unsigned long long *d_counter) {
    const long long pad_elems = spl_eval_regroup_elems(gp, nq, nsm, smem_optin);
    if (gp.ndim != 4 || pad_elems <= 0 || !d_pad)
        return spl_eval_f32_launch(gp, d_x, l1x, nq, d_coef, d_out, stream, nsm, smem_optin, d_counter);
    DerivParams dp;
    for (int d = 0; d < SPL_MAXDIM; ++d) dp.nd[d] = 0;
    int *d_flag = reinterpret_cast<int *>(d_pad + pad_elems);
    const RegroupPlan &pl = regroup_plan(gp, smem_optin, false);
    launch_table(gp, pl.tl, pl.table_doubles, false, d_coef64, d_pad, stream);
    int rc = launch_eval_regroup<4, true, false>(gp, dp, d_x, l1x, nq, d_pad, d_out, stream, nsm, smem_optin, d_flag);
    if (rc != SPLPAK_OK) return rc;
    return launch_eval_f32<4>(gp, d_x, l1x, nq, d_coef, d_out, stream, nsm, smem_optin, d_counter, d_flag);
}
#endif   // SPLPAK_REAL32

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// d_tab: the table the kernel reads, tab_doubles (even) entries laid out as tl
template <int NDIM, bool VALUE, bool UNI, int ORDER = 0>
static int launch_eval(const GridParams &gp, const DerivParams &dp, const TableLayout &tl, const real_t *d_x, int l1x,
                       long long nq, const double *d_tab, long long tab_doubles, real_t *d_out,
                       cudaStream_t stream, int nsm, size_t smem_optin, unsigned long long *d_counter,
                       const int *d_flag = nullptr) {
    constexpr int THREADS = EvalCfg<NDIM, ORDER>::THREADS;
    const size_t coef_bytes = (size_t)tab_doubles * sizeof(double);
    const size_t static_reserve = 2048;
    SPL_CUDA_TRY(cudaMemsetAsync(d_counter, 0, sizeof(unsigned long long), stream));
    // a handful of queries (scalar splfe / splde calls): gathering 4^ndim values from L2 is cheaper than staging the table
    const bool use_smem = coef_bytes + static_reserve <= smem_optin && coef_bytes < (1u << 20) &&
                          (UNI || nq * (long long)spl_ipow(4, NDIM) * 64 > (long long)coef_bytes / 8);
    long long chunks = (nq + EVAL_WCHUNK - 1) / EVAL_WCHUNK;
    long long ctas = (chunks + THREADS / 32 - 1) / (THREADS / 32);
    if (ctas < 1) ctas = 1;
    if (use_smem) {
        auto kern = spl_eval_kernel<NDIM, true, VALUE, UNI, ORDER>;
        SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coef_bytes));
        long long grid = nsm;
        if (grid > ctas) grid = ctas;
        kern<<<(unsigned)grid, THREADS, coef_bytes, stream>>>(gp, dp, tl, d_x, l1x, nq, d_tab, tab_doubles, d_out,
                                                              d_counter, d_flag);
    } else {
        auto kern = spl_eval_kernel<NDIM, false, VALUE, UNI, ORDER>;
        long long grid = (long long)nsm * (2048 / THREADS);
        if (grid > ctas) grid = ctas;
        kern<<<(unsigned)grid, THREADS, 0, stream>>>(gp, dp, tl, d_x, l1x, nq, d_tab, tab_doubles, d_out, d_counter, d_flag);
    }
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

template <int NDIM, bool VALUE, bool UNI, int ORDER = 0>
static int eval_dispatch(const GridParams &gp, const DerivParams &dp, const EvalRoute &rt, const real_t *d_x, int l1x,
                         long long nq, const double *d_coef, long long ncol_padded, real_t *d_out, cudaStream_t stream,
                         int nsm, size_t smem_optin, unsigned long long *d_counter, double *d_scratch) {
    const double *tab = d_coef;
    long long tab_doubles = ncol_padded;
    if (rt.table_doubles > 0) {
        launch_table(gp, rt.tl, rt.table_doubles, UNI, d_coef, d_scratch, stream);
        tab = d_scratch;
        tab_doubles = rt.table_doubles;
    }
    if (rt.regroup) {
        if constexpr (NDIM >= 2) {
            // forced ("regroup"): the regrouping kernel alone.  Default: order probe, then BOTH kernels -- the probe's flag
            // (behind the table image in d_scratch) makes the wrong one exit immediately.
            int *d_flag = rt.force_regroup ? nullptr : reinterpret_cast<int *>(d_scratch + rt.table_doubles);
            int rc = launch_eval_regroup<NDIM, VALUE, UNI, ORDER>(gp, dp, d_x, l1x, nq, tab, d_out, stream, nsm, smem_optin, d_flag);
            if (rc != SPLPAK_OK || !d_flag) return rc;
            // the plain kernel reads the same (padded) image when it is the extended table; the exact form reads the caller's
            if (UNI) return launch_eval<NDIM, VALUE, UNI, ORDER>(gp, dp, rt.tl, d_x, l1x, nq, tab, tab_doubles, d_out, stream,
                                                                 nsm, smem_optin, d_counter, d_flag);
            return launch_eval<NDIM, VALUE, false, ORDER>(gp, dp, natural_layout(gp, 0), d_x, l1x, nq, d_coef, ncol_padded,
                                                          d_out, stream, nsm, smem_optin, d_counter, d_flag);
        }
    }
    return launch_eval<NDIM, VALUE, UNI, ORDER>(gp, dp, rt.tl, d_x, l1x, nq, tab, tab_doubles, d_out, stream, nsm,
                                                smem_optin, d_counter);
}

// d_coef: float64 device table with ncol_padded (even, >= ncol) entries; d_counter: 8-byte scratch; d_scratch: scratch of
// spl_eval_scratch_elems() + 2 doubles (or NULL when that is 0, or when the allocation failed: exact plain kernel).
// order 0: one output per query, the derivative nderiv (NULL: splfe); order 1 / 2: the derivative sets, out(ncomp, nq).
int spl_eval_launch(const GridParams &gp, const int *nderiv, int order, const real_t *d_x, int l1x, long long nq,
                    const double *d_coef, long long ncol_padded, real_t *d_out, cudaStream_t stream,
                    int nsm, size_t smem_optin, unsigned long long *d_counter, double *d_scratch) {
    DerivParams dp;
    bool value = true;
    for (int d = 0; d < SPL_MAXDIM; ++d) {
        dp.nd[d] = (nderiv && d < gp.ndim && order == 0) ? nderiv[d] : 0;
        if (dp.nd[d] != 0) value = false;
    }
    if (nq <= 0) return SPLPAK_OK;
    if (order < 0 || order > 2) return SPLPAK_ERR_NDERIV;
    EvalRoute rt = order > 0 ? eval_route_derivs(gp, order, nq, nsm, smem_optin) : eval_route(gp, nderiv, nq, nsm, smem_optin);
    if (!d_scratch && rt.table_doubles > 0) {
        rt = EvalRoute();                         // no scratch: the exact plain kernel on the caller's table
        rt.tl = natural_layout(gp, 0);
    }
#define SPL_EVAL_ARGS gp, dp, rt, d_x, l1x, nq, d_coef, ncol_padded, d_out, stream, nsm, smem_optin, d_counter, d_scratch
#define SPL_EVAL_CASE(N)                                                                                              \
    case N:                                                                                                           \
        if (order == 1)                                                                                               \
            return rt.uni ? eval_dispatch<N, false, true, 1>(SPL_EVAL_ARGS) : eval_dispatch<N, false, false, 1>(SPL_EVAL_ARGS); \
        if (order == 2)                                                                                               \
            return rt.uni ? eval_dispatch<N, false, true, 2>(SPL_EVAL_ARGS) : eval_dispatch<N, false, false, 2>(SPL_EVAL_ARGS); \
        if (rt.uni)                                                                                                   \
            return value ? eval_dispatch<N, true, true>(SPL_EVAL_ARGS) : eval_dispatch<N, false, true>(SPL_EVAL_ARGS);    \
        return value ? eval_dispatch<N, true, false>(SPL_EVAL_ARGS) : eval_dispatch<N, false, false>(SPL_EVAL_ARGS);
    switch (gp.ndim) {
        SPL_EVAL_CASE(1)
        SPL_EVAL_CASE(2)
        SPL_EVAL_CASE(3)
        SPL_EVAL_CASE(4)
    }
#undef SPL_EVAL_CASE
#undef SPL_EVAL_ARGS
    return SPLPAK_ERR_NDIM;
}
