// common.cuh -- shared definitions for the sm_100a kernels of splpak_b200.
//
// Data layout in HBM (see DESIGN.md):
//   points      AoS as Fortran passes them: x(l1x, n) + y(n) [+ w(n)], splpak_real
//   records     window-sorted AoS scratch: (ndim+2) float64 per point = x[0..ndim-1], y, w
//   S           "orthant stencil" storage of the Gram matrix G = sum (w phi)(w phi)^T:
//               S[node * 4^ndim + sum_d delta_d 4^d], delta_d = |col_d - row_d| in 0..3, node_d =
//               min(row_d, col_d).  G is symmetric under swapping row_d <-> col_d in every
//               dimension separately (tensor-product basis), so 4^ndim values per node hold all of it.
//   AB          lower band storage of G for the Cholesky: element (i, j), i >= j, at AB[i + j*lda]
//   coef        float64 on the device, dimension 1 fastest (src/splpak.F90:661-666)
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/splpak_b200.h"

typedef splpak_real real_t;

#define SPL_MAXDIM 4
#define SPL_NSM_DEFAULT 148
#define SPL_FAIL_WORDS 256      // ints behind a handle's failure flag: [0] flag, [1] barrier counter, [32..] data-flow flags

struct GridParams {
    int ndim;
    int nodes[SPL_MAXDIM];
    int nwin[SPL_MAXDIM];          // windows per dimension = nodes - 3
    double xmin[SPL_MAXDIM];
    double dx[SPL_MAXDIM];         // (xmax-xmin)/(nodes-1), src/splpak.F90:747
    double dxin[SPL_MAXDIM];       // 1/dx, :748
    long long ncol;                // product of nodes
    long long nwindows;            // product of nwin
    int nsten;                     // 4^ndim
    // Deterministic accumulation (opt-in, SPLPAK_B200_DETERMINISTIC=1; null otherwise): every partial sum that several
    // CTAs add to the same entry of S / g goes into three 40-bit fixed-point limbs with INTEGER atomics (integer addition
    // commutes, so the sums do not depend on the order in which the CTAs arrive), scaled by 2^(fxe - 116):
    //   fxS [3 * ncol * nsten], fxg [3 * ncol], fxe[0] / fxe[1] = exponent bound of any S / g partial sum of the pass.
    // A pass runs twice: fxpass = 1 records the largest |partial sum| (bit pattern, atomicMax) in fxmax[0] / fxmax[1], from
    // which the scale is taken; fxpass = 0 adds.  Both passes compute the same values (sorted permutation, fixed item order).
    unsigned long long *fxS, *fxg, *fxmax;
    const int *fxe;
    int fxpass;
};

// ---- deterministic accumulation: 120-bit fixed point in three int64 limbs (see GridParams) ----
// v = t * 2^(e - 116), |t| < 2^116 (+ 23 bits of head-room in the top limb); limbs hold bits [0, 40), [40, 80), [80, ..)
// of trunc(t); the splits are exact in double arithmetic (each remainder is a suffix of t's 53-bit mantissa), bits below
// 2^(e - 116) are dropped -- 60 binary digits below the rounding of any entry within 2^-60 of the bound.
__device__ __forceinline__ void spl_fx_add(unsigned long long *limb, double v, int e) {
    const double t = scalbn(v, 116 - e);
    const double h2 = trunc(t * 0x1p-80);
    const double r1 = fma(-h2, 0x1p80, t);
    const double h1 = trunc(r1 * 0x1p-40);
    const double h0 = trunc(fma(-h1, 0x1p40, r1));
    if (h2 != 0.0) atomicAdd(limb + 2, (unsigned long long)(long long)h2);
    if (h1 != 0.0) atomicAdd(limb + 1, (unsigned long long)(long long)h1);
    if (h0 != 0.0) atomicAdd(limb, (unsigned long long)(long long)h0);
}
__device__ __forceinline__ double spl_fx_value(const unsigned long long *limb, int e) {
    const __int128 tot = ((__int128)(long long)limb[2] << 80) + ((__int128)(long long)limb[1] << 40) + (__int128)(long long)limb[0];
    const long long hi = (long long)(tot >> 64);
    const unsigned long long lo = (unsigned long long)tot;
    return scalbn(fma((double)hi, 0x1p64, (double)lo), e - 116);
}
// scale-finding pass: largest |v| as a bit pattern.  The current maximum is read first -- almost every value is below it,
// and one atomicMax per value on a single address serialised the pass (cfg4: 1.5e8 values, 70 ms)
__device__ __forceinline__ void spl_fx_max(unsigned long long *m, double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(fabs(v));
    if (b > *reinterpret_cast<volatile unsigned long long *>(m)) atomicMax(m, b);
}
// one contribution to S[idx] / g[idx]
__device__ __forceinline__ void spl_add_S(const GridParams &gp, double *S, long long idx, double v) {
    if (!gp.fxS) atomicAdd(S + idx, v);
    else if (gp.fxpass) spl_fx_max(gp.fxmax, v);
    else spl_fx_add(gp.fxS + 3 * idx, v, gp.fxe[0]);
}
__device__ __forceinline__ void spl_add_g(const GridParams &gp, double *g, long long idx, double v) {
    if (!gp.fxS) atomicAdd(g + idx, v);
    else if (gp.fxpass) spl_fx_max(gp.fxmax + 1, v);
    else spl_fx_add(gp.fxg + 3 * idx, v, gp.fxe[1]);
}

// 10 symmetric pairs (i <= j) of the 4 window-local node indices of one dimension.
__host__ __device__ __forceinline__ void spl_pair(int a, int &i, int &j) {
    // a: 0..9 -> (0,0)(0,1)(0,2)(0,3)(1,1)(1,2)(1,3)(2,2)(2,3)(3,3)
    const int pi = (a >= 4) + (a >= 7) + (a >= 9);
    const int start = (pi == 0) ? 0 : (pi == 1) ? 4 : (pi == 2) ? 7 : 9;
    i = pi;
    j = pi + (a - start);
}

__host__ __device__ constexpr int spl_ipow(int b, int e) { return e <= 0 ? 1 : b * spl_ipow(b, e - 1); }

// Fixed-point nearest-node histogram (assemble.cu: spl_classify_kernel): two int64 limbs per node (+ one pair for
// totlwt), the chunk's scale (qscale, lsb exponent) and the bit pattern of its largest |w|.
struct HistScratch {
    unsigned long long *hq = nullptr;
    double *qparams = nullptr;
    unsigned long long *wmax = nullptr;
};

// Scratch of the chunk pipeline of assemble.cu (owned by a fit handle, sized by spl_assemble_scratch_*).
struct AssembleScratch {
    unsigned *wincount, *winstart, *wincursor, *itemstart, *item_win, *item_seg, *meta;
    unsigned *perm;
    long long cap;        // points the chunk-sized arrays hold (perm, perm2, yw, pairs, keys, item_win, item_seg)
    long long max_items;
    long long nbins;      // bins of the counting sort: windows (direct path) or cells (moment path)
    int moments;          // 1: 3-D assembly by cell moments (moments.cuh)
    double *celltab;      // moment path: per-(dimension, cell) coefficient tables
    double *cellmom;      // moment path: per-cell moment sums of the chunk in flight (kept zero between chunks)
    int cursor_stride;    // 4-byte words between the per-bin cursors of the second binning pass
    HistScratch hist;     // fixed-point histogram scratch
    double *yw;           // moment path: interleaved (y, w) copy of the chunk, 2 doubles per point (sized with perm)
    // deterministic mode (GridParams::fxS): limb arrays, exponents, bound scratch, second permutation buffer of the sort
    int deterministic;
    unsigned long long *fxS, *fxg, *fxmax;   // fxS and fxg are one allocation (3 (ncol nsten + ncol) limbs), fxmax 2 words
    int *fxe;
    unsigned *perm2;
    // two-level partition of the cell path (spl_part1_kernel / spl_part2_kernel): bucket-sorted (key, index) pairs of the
    // chunk (8 bytes per point, sized with perm) and the <= 64 bucket cursors
    unsigned long long *pairs;
    unsigned *cursor1;
    unsigned *keys;       // bin key per point of the chunk, written by the classify pass (4 bytes per point)
};

// Scratch of the orthogonal fit path (ortho.cuh), owned by a fit handle.
struct OrthoScratch {
    unsigned *wincount = nullptr, *winstart = nullptr, *wincursor = nullptr, *itemstart = nullptr, *meta = nullptr;
    unsigned *perm = nullptr;
    long long perm_cap = 0;
    HistScratch hist;              // fixed-point histogram scratch
    double *Rw = nullptr;          // nwindows x ncw x (ncw + 1)
    unsigned *blist = nullptr;     // non-zero stage-2 blocks, in order; meta2[0] = their number
    unsigned *meta2 = nullptr;
    double *Rb = nullptr;          // ncol x (bw + 2): band row + transformed rhs
    long long *progress = nullptr; // pipeline flags, one per block
    double *csol = nullptr;        // ncol
    int ncw = 0, nrb = 0, nblk_win = 0, bw = 0;
    long long max_blocks = 0;
    int ready = 0;
};

// Scratch of one robust fit call (robust.cu): per point the |residual| keys, the spline values and the row weights;
// the selection's histogram + state, the weight kernel's partial sums, the previous coefficients and the small results.
struct RobustScratch {
    long long n;
    int nparts;                           // CTAs of the weight kernel (one partial sum each)
    unsigned long long *key;              // n
    real_t *s;                            // n: s(x_i), then the keys are formed from it
    real_t *rw;                           // n: row weights w_i sqrt(u_i) of the next assembly
    unsigned long long *hist, *state, *nzero;   // one allocation: bins, 4 state words, the rejected count
    // one allocation: [cprev (ncol) | change {max |dc|, max |c|} | stats {sum u, rejected} | tot0 | part (nparts)];
    // tot0: [totlwt, nrows] of the first assembly, restored before every solve so that the constraint rows stay fixed
    double *small, *cprev, *change, *stats, *tot0, *part;
};

// Scratch of one GLM fit call (glm.cu): per point the spline values, the working response and the row weights; the
// domain-check counts, the previous and the final coefficients, the deviance and the working kernel's partial sums.
struct GlmScratch {
    long long n;
    int nparts;                           // CTAs of the working kernel (three partial sums each)
    real_t *s;                            // n: s(x_i) of the coefficients being evaluated
    real_t *z, *rw;                       // n: working response z_i and row weight sqrt(W_i) of the next assembly
    unsigned long long *count;            // {y outside the family's domain where w > 0, m = points with w > 0}
    // one allocation: [cprev (ncol) | cfin (ncol) | dev {D, X^2, ywy} | tot0 | part (3 nparts)]; tot0 as in RobustScratch
    double *small, *cprev, *cfin, *dev, *tot0, *part;
};

extern unsigned long long g_spl_launches;   // host-side launch counter (capi.cu)

#define SPL_CUDA_TRY(expr)                                                              \
    do {                                                                                \
        cudaError_t _e = (expr);                                                        \
        if (_e != cudaSuccess) {                                                        \
            fprintf(stderr, "splpak_b200: CUDA error %s at %s:%d (%s)\n",               \
                    cudaGetErrorString(_e), __FILE__, __LINE__, #expr);                 \
            return SPLPAK_ERR_CUDA;                                                     \
        }                                                                               \
    } while (0)

static inline int spl_div_up(long long a, long long b) { return (int)((a + b - 1) / b); }
