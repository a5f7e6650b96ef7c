// assemble.cu -- point-sharded assembly of the weighted normal equations for sm_100a.
//
// Replaces the data-row loop of splcw (src/splpak.F90:788-855) and the row accumulation of
// suprls (:1468-1549): instead of one dense ncol-wide row per point pushed through a streaming
// Householder QR (2*ncol^2 flops per point), each point contributes its <= 4^ndim non-zeros to
//   G = sum_i (w_i phi_i)(w_i phi_i)^T,   g = sum_i (w_i phi_i)(w_i y_i)
// and, when xtrap != 0, to the nearest-node weight histogram of :885-907.
//
// Pipeline per chunk of points (all on one stream):
//   1. spl_classify_kernel   one pass over the raw AoS points: window id -> per-window counts,
//                            nearest-node histogram (with the :899 quirk), totlwt, row count
//   2. spl_scan_kernel       exclusive scan of the counts -> window segment starts + work items
//   3. spl_perm_kernel       second pass: counting sort of the point INDICES by window (4 bytes per
//                            point; scattering 40-byte records instead was LSU-bound, see DESIGN.md);
//      spl_part1/2_kernel    cell path, large chunks: two-level partition (buckets of cells, then cells), every tile
//                            sorted locally in shared memory and written in position order -- one global reservation
//                            per (tile, bucket) / (tile, cell) instead of one returning L2 atomic per point
//      spl_segsort_kernel    SPLPAK_B200_DETERMINISTIC=1 only: every bin's segment of the permutation sorted
//   4. spl_items_kernel      work-item table (window, segment of <= CH points)
//   5. accumulate            3-D / 4-D: spl_moments[4]_kernel + spl_cell_transform[4]_kernel (moments.cuh: per-cell
//                            Legendre moments as an FP64 tensor-core GEMM over the points, then one change of basis
//                            per cell); 1-D / 2-D (and 3-D / 4-D under SPLPAK_B200_ASSEMBLY=direct):
//      spl_accumulate_kernel persistent CTAs; per work item the points are gathered through the
//                            permutation (prefetched two batches ahead, hidden under the FP64 work),
//                            the window-local block of G is accumulated in REGISTERS and flushed once
//                            with red.global.add.f64 (deterministic mode: fixed-point limbs, integer atomics)
//
// The per-point outer product of a tensor-product basis has only 10^ndim distinct entries
// (10 symmetric pairs per dimension), not 4^ndim(4^ndim+1)/2: G is symmetric under swapping the row
// and column index of any single dimension.  The accumulator of a window is therefore the
// 10 x ... x 10 tensor  M[a_N]..[a_1] = sum_p w^2 prod_d s_d[a_d],  s_d[(i,j)] = b_d[i] b_d[j],
// which is exactly the "orthant stencil" storage S (common.cuh).  This halves the FP64 work of a
// plain symmetric rank-1 update (1000 vs 2080 FMAs per point in 3-D).
//
// Thread mapping inside a CTA: a "group" of LPG lanes owns the whole accumulator tensor of the
// window; lane u of the group owns R "outer" index tuples (a_N..a_2) x all 10 a_1, i.e. R*10
// accumulators, and different groups take different points (K-split), reduced at the end of the
// work item with warp shuffles + one shared-memory pass.  The right-hand side g rides along as
// 4^(ndim-1) extra outer tuples whose inner vector is b_1[0..3] instead of s_1[0..9].
#include <stdlib.h>
#include <string.h>

#include "basis.cuh"

// ------------------------------------------------------------------------------------------
// window id / nearest node
// ------------------------------------------------------------------------------------------
template <int NDIM>
__device__ __forceinline__ unsigned spl_window_key(const GridParams &gp, const real_t *xp) {
    unsigned key = 0;
#pragma unroll
    for (int dd = 0; dd < NDIM; ++dd) {
        const int d = NDIM - 1 - dd;
        int ws, ibmn, ibmx;
        spl_box((double)xp[d], gp.xmin[d], gp.dxin[d], gp.nodes[d], ws, ibmn, ibmx);
        key = key * (unsigned)gp.nwin[d] + (unsigned)ws;
    }
    return key;
}

// Cell id (moment path): every dimension has nodes+1 cells -- the nodes-1 node intervals plus the two
// exterior half-lines, on which the basis continues linearly (bascmp's s >= 2 branch, :342-379).  Inside
// one cell every 1-D basis function is a single polynomial of degree <= 3.
__device__ __forceinline__ int spl_cell_of(double x, double xmin, double dxin, int nod) {
    const double t = spl_mul(dxin, spl_sub(x, xmin));
    const int it = min(__double2int_rz(t), nod - 1);         // saturating; NaN -> 0
    return (t < 0.0) ? 0 : it + 1;
}
template <int NDIM>
__device__ __forceinline__ unsigned spl_cell_key(const GridParams &gp, const real_t *xp) {
    unsigned key = 0;
#pragma unroll
    for (int dd = 0; dd < NDIM; ++dd) {
        const int d = NDIM - 1 - dd;
        key = key * (unsigned)(gp.nodes[d] + 1) + (unsigned)spl_cell_of((double)xp[d], gp.xmin[d], gp.dxin[d], gp.nodes[d]);
    }
    return key;
}
template <int NDIM, bool CELL>
__device__ __forceinline__ unsigned spl_bin_key(const GridParams &gp, const real_t *xp) {
    return CELL ? spl_cell_key<NDIM>(gp, xp) : spl_window_key<NDIM>(gp, xp);
}

// Nearest-node address of :893-902, including the quirk at :899 (a dimension whose index is out of
// range is skipped in the Horner recurrence instead of discarding the point).
template <int NDIM>
__device__ __forceinline__ long long spl_nearest_node(const GridParams &gp, const real_t *xp) {
    long long iin = 0;
#pragma unroll
    for (int dd = 0; dd < NDIM; ++dd) {
        const int d = NDIM - 1 - dd;
        const int inmx = gp.nodes[d] - 1;
        double t = spl_add(spl_mul(gp.dxin[d], spl_sub((double)xp[d], gp.xmin[d])), 0.5);
        t = fmin(fmax(t, -4.0), (double)inmx + 4.0);
        const int inidim = __double2int_rz(t);     // Fortran int(): truncation toward zero
        if (inidim < 0 || inidim > inmx) continue;
        iin = (long long)(inmx + 1) * iin + inidim;
    }
    return iin;
}

// Both binning passes are latency-bound (one dependent global round trip per point), so every thread
// handles BIN_U points per iteration with all their loads -- and, in the second pass, all their
// returning atomics -- in flight together.  Counts use fire-and-forget RED (no warp aggregation:
// MATCH.ANY costs more than the reds it saves on scattered data).
#define BIN_U 4

// SMEMH: the per-window counts are first accumulated in a shared-memory histogram (native 32-bit
// ATOMS) and flushed once per CTA -- the L2 atomic units, not HBM, bound this pass when every point
// issues two global reductions.  Used when the window table fits (launcher decides).
// SMEMC (with SMEMH): the nearest-node weight histogram is privatised per CTA in shared memory as well (one
// 1024-thread CTA per SM, shared-memory f64 atomic adds, one flush of the non-zero entries per CTA): with one
// red.global.add.f64 per point the pass was bound by the L2 atomic units (1.45 ms per 1e8 points for 0.5 ms of HBM
// traffic).  Used when both tables fit (launcher decides).
template <int NDIM, bool SMEMH, bool CELL, bool SMEMC = false, bool KEYS = false>
__global__ void __launch_bounds__(SMEMC ? 1024 : 512, SMEMC ? 1 : 2)
spl_classify_kernel(const __grid_constant__ GridParams gp, const real_t *__restrict__ x, int l1x,
                    const real_t *__restrict__ w, int weighted, long long n, int nbins,
                    unsigned *__restrict__ wincount, int do_hist, unsigned long long *__restrict__ hq,
                    const double *__restrict__ qparams, double *__restrict__ totals, const real_t *__restrict__ y,
                    double2 *__restrict__ yw, unsigned *__restrict__ keys = nullptr) {
    // keys (two-level partition): the bin key of every point (0xffffffff for a zero-weight point), so that the partition
    // pass reads 4 bytes per point instead of the coordinates and the weight again
    extern __shared__ __align__(8) unsigned s_hist[];
    unsigned long long *s_cnt = reinterpret_cast<unsigned long long *>(s_hist + ((nbins + 1) & ~1));   // SMEMC: gp.ncol x 8 bytes
    if (SMEMH) {
        for (int e = threadIdx.x; e < nbins; e += blockDim.x) s_hist[e] = 0u;
        if (SMEMC)
            for (long long e = threadIdx.x; e < gp.ncol; e += blockDim.x) s_cnt[e] = 0ULL;
        __syncthreads();
    }
    // nearest-node histogram in FIXED POINT: q = rn(w * qscale) with qscale a power of two chosen from the chunk's
    // largest |w| (spl_hist_prepare), accumulated with INTEGER atomics -- exact, hence independent of the order in which
    // the atomics land: the sparse-node decision of :936 is reproducible run to run (a float64 atomic sum is not)
    const double qscale = do_hist ? qparams[0] : 0.0;
    long long totq = 0;
    double rows = 0.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < n; i0 += stride * BIN_U) {
        double wv[BIN_U];
        real_t xp[BIN_U][NDIM];
#pragma unroll
        for (int u = 0; u < BIN_U; ++u) {
            const long long i = i0 + u * stride;
            wv[u] = 0.0;
            if (i < n) {
                wv[u] = weighted ? (double)w[i] : 1.0;
#pragma unroll
                for (int d = 0; d < NDIM; ++d) xp[u][d] = x[i * (long long)l1x + d];
                // moment path, weighted: interleaved (y, w) copy, so the cell-sorted gather of the moment
                // kernel pulls ONE 128-byte line for the pair instead of one each (streaming 16 B/point here
                // against 128 B/point of gather traffic there)
                if (CELL && yw) yw[i] = make_double2((double)y[i], wv[u]);
            } else {
#pragma unroll
                for (int d = 0; d < NDIM; ++d) xp[u][d] = (real_t)0;
            }
        }
#pragma unroll
        for (int u = 0; u < BIN_U; ++u) {
            if (KEYS && wv[u] == 0.0 && i0 + u * stride < n) __stcs(keys + i0 + u * stride, 0xffffffffu);
            if (wv[u] != 0.0) {                                  // zero-weight points are skipped (:796-800)
                const unsigned key = spl_bin_key<NDIM, CELL>(gp, xp[u]);
                if (KEYS) __stcs(keys + i0 + u * stride, key);
                if (SMEMH) atomicAdd(s_hist + key, 1u);
                else atomicAdd(wincount + key, 1u);
                rows += 1.0;
                if (do_hist) {
                    const long long q = __double2ll_rn(wv[u] * qscale);
                    const long long node = spl_nearest_node<NDIM>(gp, xp[u]);
                    if (SMEMC) {
                        atomicAdd(s_cnt + node, (unsigned long long)q);
                    } else {
                        atomicAdd(hq + 2 * node, (unsigned long long)(q & 0x7fffffffLL));
                        atomicAdd(hq + 2 * node + 1, (unsigned long long)(q >> 31));
                    }
                    totq += q;
                }
            }
        }
    }
    if (SMEMH) {
        __syncthreads();
        for (int e = threadIdx.x; e < nbins; e += blockDim.x) {
            const unsigned c = s_hist[e];
            if (c) atomicAdd(wincount + e, c);
        }
        if (SMEMC && do_hist)
            for (long long e = threadIdx.x; e < gp.ncol; e += blockDim.x) {
                const long long c = (long long)s_cnt[e];             // this CTA's exact sum: two limbs into the global table
                if (c != 0) {
                    atomicAdd(hq + 2 * e, (unsigned long long)(c & 0x7fffffffLL));
                    atomicAdd(hq + 2 * e + 1, (unsigned long long)(c >> 31));
                }
            }
    }
    // block reduction of totlwt (fixed point, exact) and the row count (integer-valued, exact)
    __shared__ long long s_tot[32];
    __shared__ double s_rows[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        totq += __shfl_xor_sync(0xffffffffu, totq, o);
        rows += __shfl_xor_sync(0xffffffffu, rows, o);
    }
    if ((threadIdx.x & 31) == 0) {
        s_tot[threadIdx.x >> 5] = totq;
        s_rows[threadIdx.x >> 5] = rows;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long t = 0;
        double r = 0.0;
        for (int k = 0; k < (int)(blockDim.x >> 5); ++k) {
            t += s_tot[k];
            r += s_rows[k];
        }
        if (do_hist && t != 0) {
            atomicAdd(hq + 2 * gp.ncol, (unsigned long long)(t & 0x7fffffffLL));
            atomicAdd(hq + 2 * gp.ncol + 1, (unsigned long long)(t >> 31));
        }
        if (r != 0.0) atomicAdd(totals + 1, r);
    }
}

// ---- fixed-point histogram: scale selection before, conversion to float64 after the classify pass ----
// largest finite |w| of the chunk (bit pattern: non-negative doubles order like integers)
__global__ void __launch_bounds__(1024)
spl_wmax_kernel(const real_t *__restrict__ w, long long n, unsigned long long *__restrict__ wmax_bits) {
    unsigned long long m = 0ULL;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long b = (unsigned long long)__double_as_longlong(fabs((double)w[i]));
        if (b < 0x7ff0000000000000ULL && b > m) m = b;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long v = __shfl_xor_sync(0xffffffffu, m, o);
        m = v > m ? v : m;
    }
    __shared__ unsigned long long s_m[32];
    if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 0; k < (int)(blockDim.x >> 5); ++k) m = s_m[k] > m ? s_m[k] : m;
        if (m) atomicMax(wmax_bits, m);
    }
}
// qparams[0] = qscale = 2^-lsb_exp, qparams[1] = lsb_exp: |w| < 2^e  ->  |q| = |w| qscale < 2^bits
__global__ void spl_qparams_kernel(const unsigned long long *__restrict__ wmax_bits, int bits, double *__restrict__ qparams) {
    const double wmax = wmax_bits ? __longlong_as_double((long long)*wmax_bits) : 1.0;
    int e = 0;
    if (wmax > 0.0) frexp(wmax, &e);                     // wmax = m 2^e, 0.5 <= m < 1
    int lsb_exp = e - bits;
    lsb_exp = max(min(lsb_exp, 1000), -1000);
    qparams[0] = ldexp(1.0, -lsb_exp);
    qparams[1] = (double)lsb_exp;
}
// cnt[node] += exact chunk sum (two limbs) * lsb; totals[0] += the same for totlwt; the limbs are zeroed for the next chunk
__global__ void __launch_bounds__(256)
spl_hist_finalize_kernel(unsigned long long *__restrict__ hq, const double *__restrict__ qparams, long long ncol,
                         double *__restrict__ cnt, double *__restrict__ totals) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e > ncol) return;
    const int lsb_exp = (int)qparams[1];
    const long long lo = (long long)hq[2 * e], hi = (long long)hq[2 * e + 1];
    hq[2 * e] = 0ULL;
    hq[2 * e + 1] = 0ULL;
    if (lo == 0 && hi == 0) return;
    const double v = ldexp((double)hi, 31 + lsb_exp) + ldexp((double)lo, lsb_exp);
    if (e < ncol) cnt[e] += v;
    else totals[0] += v;
}

int spl_hist_scratch_init(const GridParams &gp, HistScratch &hs, cudaStream_t st) {
    if (hs.hq) return SPLPAK_OK;
    SPL_CUDA_TRY(cudaMalloc((void **)&hs.hq, sizeof(unsigned long long) * (size_t)(2 * gp.ncol + 2)));
    SPL_CUDA_TRY(cudaMalloc((void **)&hs.qparams, sizeof(double) * 2));
    SPL_CUDA_TRY(cudaMalloc((void **)&hs.wmax, sizeof(unsigned long long)));
    SPL_CUDA_TRY(cudaMemsetAsync(hs.hq, 0, sizeof(unsigned long long) * (size_t)(2 * gp.ncol + 2), st));
    return SPLPAK_OK;
}
void spl_hist_scratch_free(HistScratch &hs) {
    if (hs.hq) cudaFree(hs.hq);
    if (hs.qparams) cudaFree(hs.qparams);
    if (hs.wmax) cudaFree(hs.wmax);
    hs.hq = nullptr;
    hs.qparams = nullptr;
    hs.wmax = nullptr;
}
// before the classify pass of a chunk: per_acc = the largest number of points one integer accumulator can receive
static int spl_hist_prepare(const HistScratch &hs, const real_t *d_w, int weighted, long long n, long long per_acc,
                            cudaStream_t st, int nsm) {
    int bits = 42;
    while (bits > 8 && (per_acc >> (62 - bits)) != 0) --bits;         // per_acc * 2^bits < 2^62
    if (weighted) {
        SPL_CUDA_TRY(cudaMemsetAsync(hs.wmax, 0, sizeof(unsigned long long), st));
        long long blocks = (n + 4095) / 4096;
        if (blocks > 4LL * nsm) blocks = 4LL * nsm;
        spl_wmax_kernel<<<(unsigned)(blocks < 1 ? 1 : blocks), 1024, 0, st>>>(d_w, n, hs.wmax);
        spl_qparams_kernel<<<1, 1, 0, st>>>(hs.wmax, bits, hs.qparams);
        g_spl_launches += 2;
    } else {
        spl_qparams_kernel<<<1, 1, 0, st>>>(nullptr, bits, hs.qparams);
        ++g_spl_launches;
    }
    return SPLPAK_OK;
}
static void spl_hist_finalize(const HistScratch &hs, const GridParams &gp, double *d_cnt, double *d_totals, cudaStream_t st) {
    spl_hist_finalize_kernel<<<spl_div_up(gp.ncol + 1, 256), 256, 0, st>>>(hs.hq, hs.qparams, gp.ncol, d_cnt, d_totals);
    ++g_spl_launches;
}


// Exclusive scan of the window counts (single CTA; nwindows is at most a few 10^5 in practice).
// winstart[k] = first record of window k, itemstart[k] = first work item of window k,
// meta[0] = number of work items, meta[1] = number of records; also resets the work counter.
__global__ void __launch_bounds__(1024)
spl_scan_kernel(const unsigned *__restrict__ wincount, long long nwindows, unsigned ch,
                unsigned *__restrict__ winstart, unsigned *__restrict__ itemstart,
                unsigned *__restrict__ meta) {
    __shared__ unsigned s_a[1024], s_b[1024];
    const int t = threadIdx.x;
    const long long per = (nwindows + 1023) / 1024;
    const long long lo = (long long)t * per;
    const long long hi = (lo + per < nwindows) ? lo + per : nwindows;
    unsigned sa = 0, sb = 0;
    for (long long k = lo; k < hi; ++k) {
        const unsigned c = wincount[k];
        sa += c;
        sb += (c + ch - 1) / ch;
    }
    s_a[t] = sa;
    s_b[t] = sb;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
        unsigned va = 0, vb = 0;
        if (t >= off) {
            va = s_a[t - off];
            vb = s_b[t - off];
        }
        __syncthreads();
        s_a[t] += va;
        s_b[t] += vb;
        __syncthreads();
    }
    unsigned ra = s_a[t] - sa, rb = s_b[t] - sb;   // exclusive prefix of this strip
    for (long long k = lo; k < hi; ++k) {
        const unsigned c = wincount[k];
        winstart[k] = ra;
        itemstart[k] = rb;
        ra += c;
        rb += (c + ch - 1) / ch;
    }
    if (t == 1023) {
        meta[0] = s_b[1023];
        meta[1] = s_a[1023];
        meta[2] = 0;   // work counter for the accumulate kernel
    }
}

template <int NDIM, bool CELL>
__global__ void __launch_bounds__(256)
spl_perm_kernel(const __grid_constant__ GridParams gp, const real_t *__restrict__ x, int l1x,
                const real_t *__restrict__ w, int weighted, long long n,
                const unsigned *__restrict__ winstart, unsigned *__restrict__ wincursor, int cstride,
                unsigned *__restrict__ perm) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < n; i0 += stride * BIN_U) {
        double wv[BIN_U];
        real_t xp[BIN_U][NDIM];
#pragma unroll
        for (int u = 0; u < BIN_U; ++u) {
            const long long i = i0 + u * stride;
            wv[u] = 0.0;
            if (i < n) {
                wv[u] = weighted ? (double)w[i] : 1.0;
#pragma unroll
                for (int d = 0; d < NDIM; ++d) xp[u][d] = x[i * (long long)l1x + d];
            } else {
#pragma unroll
                for (int d = 0; d < NDIM; ++d) xp[u][d] = (real_t)0;
            }
        }
        unsigned key[BIN_U], pos[BIN_U], ws0[BIN_U];
#pragma unroll
        for (int u = 0; u < BIN_U; ++u) {
            key[u] = 0xffffffffu;
            pos[u] = 0;
            ws0[u] = 0;
            if (wv[u] != 0.0) {
                key[u] = spl_bin_key<NDIM, CELL>(gp, xp[u]);
                ws0[u] = winstart[key[u]];
                pos[u] = atomicAdd(wincursor + (size_t)key[u] * cstride, 1u);
            }
        }
#pragma unroll
        for (int u = 0; u < BIN_U; ++u)
            if (key[u] != 0xffffffffu) perm[(long long)ws0[u] + pos[u]] = (unsigned)(i0 + u * stride);
    }
}

// ------------------------------------------------------------------------------------------
// Two-level partition (round 2; cell path, large chunks) in place of spl_perm_kernel's one returning L2 atomic per point
// (1e8 atomics in 1.9 ms: bound by the L2 atomic units, not by HBM).  The bins are grouped into <= 64 BUCKETS of 2^shift
// consecutive cells.
//   pass 1 (spl_part1_kernel)  tiles of 8,192 points: bin key, rank inside (tile, bucket) from a shared-memory counter, ONE
//                              global reservation per (tile, bucket); (key, index) pairs land bucket-sorted in `pairs`,
//                              each tile writing <= 64 contiguous runs;
//   pass 2 (spl_part2_kernel)  tiles of 8,192 pairs (a tile spans few buckets): rank inside (tile, cell) from a shared-memory
//                              histogram over the tile's key range, one global reservation per (tile, non-empty cell) --
//                              ~13 points per reservation at cfg3 -- then the point indices go to their cell's segment.
// The write frontiers of pass 2 are the cells of the buckets in flight (a few MB), which stay in L2; ranking whole chunks
// per CTA without the bucket level kept 148 x 15,625 partly written sectors alive and lost (experiments/ranked_binning_r02).
// The order of the points inside a cell is as arbitrary as before.
// ------------------------------------------------------------------------------------------
#ifndef PART2_NT
#define PART2_NT 1024                  // pass 2: threads per CTA (2048 / PART2_NT CTAs per SM)
#endif
#define PART_U 8
#define PART_TILE (PART2_NT * PART_U)  // pairs per tile of pass 2
#define PART1_NT 512                   // pass 1: 512 threads x 8 points, several CTAs per SM
#define PART1_U 8
#define PART1_TILE (PART1_NT * PART1_U)

// exclusive scan of s[0..n) in place (n <= 2 * blockDim.x, blockDim.x = 32 * nw <= 1024), total returned to every thread;
// s_w: nw + 1 words of scratch.  Contains barriers: all threads of the CTA call it.
__device__ __forceinline__ unsigned spl_block_exscan2(unsigned *s, int n, unsigned *s_w) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    const unsigned v0 = (2 * tid < n) ? s[2 * tid] : 0u, v1 = (2 * tid + 1 < n) ? s[2 * tid + 1] : 0u;
    unsigned incl = v0 + v1;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned o = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += o;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned t = (lane < nw) ? s_w[lane] : 0u, ti = t;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const unsigned o = __shfl_up_sync(0xffffffffu, ti, off);
            if (lane >= off) ti += o;
        }
        if (lane < nw) s_w[lane] = ti - t;
        if (lane == 31) s_w[nw] = ti;
    }
    __syncthreads();
    const unsigned ex = s_w[warp] + incl - v0 - v1;
    if (2 * tid < n) s[2 * tid] = ex;
    if (2 * tid + 1 < n) s[2 * tid + 1] = ex + v0;
    const unsigned total = s_w[nw];
    __syncthreads();
    return total;
}

// Both passes sort their tile LOCALLY in shared memory first and write it out in position order, so that the lanes of a
// warp store to consecutive addresses inside a run: storing every pair straight to its run (32 lanes, 32 runs) made
// 1e8 partial-sector writes, which the L2 handles no faster than the 1e8 atomics they were meant to replace (1.2 ms).
__global__ void __launch_bounds__(PART1_NT, 3)
spl_part1_kernel(const unsigned *__restrict__ keys, long long n, const unsigned *__restrict__ winstart,
                 int shift, int nbuckets, unsigned *__restrict__ cursor1, uint2 *__restrict__ pairs) {
    // per-WARP bucket counters (the 512 threads of a CTA hitting <= 64 shared counters serialised on them), turned into
    // the warps' offsets inside the tile's run of every bucket by one scan over the warps per bucket
    __shared__ unsigned s_cnt[PART1_NT / 32][64];
    __shared__ unsigned s_base[64], s_toff[64], s_w[PART1_NT / 32 + 1];
    __shared__ uint2 s_stage[PART1_TILE];
    const int tid = threadIdx.x, warp = tid >> 5;
    const long long ntiles = (n + PART1_TILE - 1) / PART1_TILE;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int e = tid; e < (PART1_NT / 32) * 64; e += PART1_NT) (&s_cnt[0][0])[e] = 0;
        __syncthreads();
        unsigned key[PART1_U], rank[PART1_U];
#pragma unroll
        for (int u = 0; u < PART1_U; ++u) {
            const long long i = tile * PART1_TILE + u * PART1_NT + tid;
            key[u] = (i < n) ? __ldcs(keys + i) : 0xffffffffu;     // written by spl_classify_kernel
            rank[u] = 0;
        }
#pragma unroll
        for (int u = 0; u < PART1_U; ++u)
            if (key[u] != 0xffffffffu) rank[u] = atomicAdd(&s_cnt[warp][key[u] >> shift], 1u);
        __syncthreads();
        if (tid < 64) {
            unsigned run = 0;
#pragma unroll
            for (int q = 0; q < PART1_NT / 32; ++q) {
                const unsigned c = s_cnt[q][tid];
                s_cnt[q][tid] = run;
                run += c;
            }
            s_toff[tid] = run;
            s_base[tid] = (run && tid < nbuckets) ? winstart[(unsigned)tid << shift] + atomicAdd(cursor1 + tid, run) : 0u;
        }
        __syncthreads();
        const unsigned count = spl_block_exscan2(s_toff, 64, s_w);          // tile-local start of every bucket's run
#pragma unroll
        for (int u = 0; u < PART1_U; ++u)
            if (key[u] != 0xffffffffu) {
                const unsigned b = key[u] >> shift;
                s_stage[s_toff[b] + s_cnt[warp][b] + rank[u]] =
                    make_uint2(key[u], (unsigned)(tile * PART1_TILE + u * PART1_NT + tid));
            }
        __syncthreads();
        for (unsigned p = tid; p < count; p += PART1_NT) {
            const uint2 pr = s_stage[p];
            const unsigned b = pr.x >> shift;
            pairs[s_base[b] + (p - s_toff[b])] = pr;
        }
        __syncthreads();
    }
}

// span: cells per group (a multiple of the bucket size, <= 2048: spl_block_exscan2); meta[1] = number of pairs.
// Shared memory: [span] counts -> tile-local offsets | [span] global bases | [PART_TILE] staged (cell - g0, index).
__global__ void __launch_bounds__(PART2_NT, 2048 / PART2_NT)
spl_part2_kernel(const uint2 *__restrict__ pairs, const unsigned *__restrict__ meta, const unsigned *__restrict__ winstart,
                 unsigned *__restrict__ wincursor, int cstride, int shift, int span, long long nbins,
                 unsigned *__restrict__ perm) {
    extern __shared__ unsigned s_part[];
    __shared__ unsigned s_lo, s_hi, s_w[33];
    unsigned *s_h = s_part, *s_b = s_part + span;
    uint2 *s_stage = reinterpret_cast<uint2 *>(s_part + 2 * span);
    const int tid = threadIdx.x;
    const long long nrec = meta[1];
    const long long ntiles = (nrec + PART_TILE - 1) / PART_TILE;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long t0 = tile * PART_TILE;
        const long long tend = (t0 + PART_TILE < nrec) ? t0 + PART_TILE : nrec;
        // the pairs are bucket-sorted: the tile's keys lie between the bucket of its first and of its last pair
        if (tid == 0) {
            s_lo = (pairs[t0].x >> shift) << shift;
            s_hi = pairs[tend - 1].x | ((1u << shift) - 1u);
        }
        __syncthreads();
        const unsigned klo = s_lo, khi = s_hi;
        for (unsigned g0 = klo; g0 <= khi; g0 += (unsigned)span) {
            for (int e = tid; e < span; e += PART2_NT) s_h[e] = 0;
            __syncthreads();
            // (the pairs are read twice, the second time from L2, instead of being held in registers: two CTAs per SM)
            unsigned rank[PART_U];
#pragma unroll
            for (int u = 0; u < PART_U; ++u) {
                const long long pos = t0 + u * PART2_NT + tid;
                const unsigned k = (pos < tend) ? __ldcg(&pairs[pos].x) : 0xffffffffu;
                rank[u] = 0;
                if (k - g0 < (unsigned)span) rank[u] = atomicAdd(&s_h[k - g0], 1u);
            }
            __syncthreads();
            for (int e = tid; e < span; e += PART2_NT) {
                const unsigned c = s_h[e];
                if (c && (long long)g0 + e < nbins)
                    s_b[e] = winstart[g0 + e] + atomicAdd(wincursor + (size_t)(g0 + e) * cstride, c);
            }
            const unsigned count = spl_block_exscan2(s_h, span, s_w);        // counts -> tile-local offsets
#pragma unroll
            for (int u = 0; u < PART_U; ++u) {
                const long long pos = t0 + u * PART2_NT + tid;
                if (pos < tend) {
                    const uint2 pr = __ldcg(pairs + pos);
                    if (pr.x - g0 < (unsigned)span) s_stage[s_h[pr.x - g0] + rank[u]] = make_uint2(pr.x - g0, pr.y);
                }
            }
            __syncthreads();
            for (unsigned p = tid; p < count; p += PART2_NT) {
                const uint2 st = s_stage[p];
                perm[(long long)s_b[st.x] + (p - s_h[st.x])] = st.y;
            }
            __syncthreads();
        }
    }
}

__global__ void __launch_bounds__(256)
spl_items_kernel(const unsigned *__restrict__ wincount, const unsigned *__restrict__ itemstart,
                 long long nwindows, unsigned ch, unsigned *__restrict__ item_win,
                 unsigned *__restrict__ item_seg) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nwindows) return;
    const unsigned c = wincount[k];
    const unsigned ni = (c + ch - 1) / ch;
    const unsigned s0 = itemstart[k];
    for (unsigned s = 0; s < ni; ++s) {
        item_win[s0 + s] = (unsigned)k;
        item_seg[s0 + s] = s;
    }
}

// ------------------------------------------------------------------------------------------
// accumulate
// ------------------------------------------------------------------------------------------

template <int NDIM> struct AccTraits;
// R   outer tuples per lane (x 10 inner = accumulators per lane)
// LPG lanes per group (a group owns one point at a time); NT threads per CTA
// PB  points staged per batch (double buffered); CH max points per work item
// RS  doubles per staged point: even (16-byte aligned 128-bit loads) with RS/2 odd, so consecutive
//     points start 4 banks apart and the staging stores of neighbouring points do not collide.
template <> struct AccTraits<1> { static constexpr int R = 1, LPG = 1,   NT = 256, PB = 256, CH = 16384, RS = 18;  };
template <> struct AccTraits<2> { static constexpr int R = 4, LPG = 4,   NT = 256, PB = 256, CH = 8192,  RS = 34;  };
template <> struct AccTraits<3> { static constexpr int R = 4, LPG = 32,  NT = 256, PB = 256, CH = 16384, RS = 46;  };
template <> struct AccTraits<4> { static constexpr int R = 4, LPG = 256, NT = 256, PB = 72,  CH = 4096,  RS = 150; };

template <int NDIM> struct AccDerived {
    using T = AccTraits<NDIM>;
    static constexpr int NOUT = spl_ipow(10, NDIM - 1);          // G outer tuples (a_N..a_2)
    static constexpr int NGT = (NOUT + T::R - 1) / T::R;         // lanes of a group holding G tuples
    static constexpr int NG = T::NT / T::LPG;                    // groups per CTA
    static constexpr int NW = T::NT / 32;                        // warps per CTA
    static constexpr int LPGW = T::LPG < 32 ? T::LPG : 32;       // lanes of a group inside one warp
    static constexpr int NRACC = spl_ipow(4, NDIM);              // rhs accumulators of a window
    static constexpr int APL = NRACC / T::LPG;                   // rhs accumulators per lane (4,4,2,1)
    // staged record of one point (doubles):
    static constexpr int OFF_I = 0;                              // s_1[10], b_1[4], 2 pad
    static constexpr int OFF_T2 = 16;                            // s_2[10], s_2[0], s_2[1] (cyclic), b_2[4]
    static constexpr int OFF_H = (NDIM >= 2) ? 32 : 16;          // outer table
    static constexpr int NH = (NDIM <= 2) ? 2 : (NDIM == 3 ? 14 : 116);
    static constexpr int HRHS = (NDIM <= 2) ? 1 : NOUT / 10;     // first rhs entry of H
    // staging tasks per point: one per dimension; in 4-D dimensions 3 and 4 share a task (it also
    // forms their 116 products, so no second staging phase is needed)
    static constexpr int NTASK = (NDIM == 4) ? 3 : NDIM;
    static constexpr int NP = 128;                               // producer (gather + staging) threads
    static constexpr int TPT = (T::PB * NTASK + NP - 1) / NP;    // staging tasks per producer thread
    static_assert(NGT <= T::LPG, "group too small");
    static_assert(APL * T::LPG == NRACC && APL >= 1 && APL <= 4, "rhs split");
    static_assert(OFF_H + NH <= T::RS, "record stride too small");
    static_assert(T::RS % 2 == 0 && (T::RS / 2) % 2 == 1, "record stride must be 2*odd");
};

// G accumulator (outer tuple o = u*R + r, inner pair a) -> S
template <int NDIM>
__device__ __forceinline__ void spl_flush_g(const GridParams &gp, const int *ws, int u, int r, int a,
                                            double v, double *__restrict__ S) {
    using D = AccDerived<NDIM>;
    using T = AccTraits<NDIM>;
    if (v == 0.0 || u >= D::NGT) return;
    int o = u * T::R + r;
    if (o >= D::NOUT) return;
    long long node = 0, nstride = 1;
    int sten = 0, sstride = 1;
    int ad = a;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) {
        int i, j;
        spl_pair(ad, i, j);
        node += (long long)(ws[d] + i) * nstride;
        sten += (j - i) * sstride;
        nstride *= gp.nodes[d];
        sstride *= 4;
        ad = o % 10;
        o /= 10;
    }
    spl_add_S(gp, S, node * gp.nsten + sten, v);
}

// rhs accumulator e = (i_N..i_1) in base 4, i_1 fastest -> g
template <int NDIM>
__device__ __forceinline__ void spl_flush_rhs(const GridParams &gp, const int *ws, int e, double v,
                                              double *__restrict__ g) {
    if (v == 0.0) return;
    long long node = 0, nstride = 1;
#pragma unroll
    for (int d = 0; d < NDIM; ++d) {
        node += (long long)(ws[d] + (e & 3)) * nstride;
        nstride *= gp.nodes[d];
        e >>= 2;
    }
    spl_add_g(gp, g, node, v);
}

// named barriers (id 0 is __syncthreads): FULL/EMPTY per staging buffer, one for the consumer warps
#define ACC_BAR_FULL 1
#define ACC_BAR_EMPTY 3
#define ACC_BAR_CONS 5
__device__ __forceinline__ void spl_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void spl_bar_arrive(int id, int nthreads) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Warp-specialised: threads [0, NT) are CONSUMERS (pure register-tiled DFMA stream over staged
// points), threads [NT, NT + NP) are PRODUCERS (gather through the permutation, 1-D bases, per-point
// factor tables into the double-buffered staging area).  The two meet only at named barriers
// (producer: bar.arrive FULL / bar.sync EMPTY; consumer: bar.sync FULL / bar.arrive EMPTY), so the
// latency-bound staging never stalls the FP64 stream.
// RHS_ONLY: only g = sum (w phi)(w y) is accumulated (the refinement pass of capi.cu re-assembles the
// right-hand side from residuals; G is already there).
template <int NDIM, bool RHS_ONLY>
__global__ void __launch_bounds__(AccTraits<NDIM>::NT + AccDerived<NDIM>::NP, 1)
spl_accumulate_kernel(const __grid_constant__ GridParams gp, const real_t *__restrict__ x, int l1x,
                      const real_t *__restrict__ y, const real_t *__restrict__ w, int weighted,
                      const unsigned *__restrict__ perm, const unsigned *__restrict__ wincount,
                      const unsigned *__restrict__ winstart, const unsigned *__restrict__ item_win,
                      const unsigned *__restrict__ item_seg, unsigned *__restrict__ meta,
                      double *__restrict__ S, double *__restrict__ g) {
    using T = AccTraits<NDIM>;
    using D = AccDerived<NDIM>;
    constexpr int R = T::R, RS = T::RS, PB = T::PB, NT = T::NT, NP = D::NP, TPT = D::TPT, APL = D::APL;
    constexpr int NALL = NT + NP;
    constexpr int NTASK = D::NTASK;
    extern __shared__ __align__(16) double smem[];
    double *s_pts = smem;                       // 2 x PB x RS (double buffered)
    double *s_red = smem + 2 * PB * RS;         // LPGW * (R * 10 + APL)   (unused for 4-D)
    __shared__ unsigned s_item;

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int grp = tid / T::LPG;
    const int u = tid % T::LPG;
    const bool is_prod = tid >= NT;
    const int ptid = tid - NT;                  // producer thread index

    // per-lane constant offsets into a staged record.  The lane's R = 4 outer tuples o = 4u + r use
    // T2[(4u) % 10 .. +1], T2[(4u+2) % 10 .. +1] (two aligned 128-bit loads thanks to the cyclic copy)
    // and H[(4u)/10], H[(4u+2)/10] (a multiple of 10 can only fall between r = 1 and r = 2).
    const int uo = min(u, D::NGT - 1) * R;
    const int offT = D::OFF_T2 + (uo % 10);
    const int offHa = D::OFF_H + (NDIM == 1 ? 0 : uo / 10);
    const int offHb = D::OFF_H + (NDIM == 1 ? 0 : (uo + 2) / 10);
    // rhs: accumulators e = u*APL + j share (i_N..i_2); i_1 = (u*APL) % 4 + j
    const int e0 = u * APL;
    const int offRI = D::OFF_I + 10 + (e0 & 3);
    const int offRT = D::OFF_T2 + 12 + ((e0 >> 2) & 3);
    const int offRH = D::OFF_H + D::HRHS + (NDIM >= 3 ? (e0 >> 4) : 0);
    const unsigned nitems = meta[0];

    // staging task j of this thread: point tp[j] of the batch, task type tt[j]
    int tp[TPT], tt[TPT];
#pragma unroll
    for (int j = 0; j < TPT; ++j) {
        const int idx = (is_prod ? ptid : 0) + j * NP;
        tp[j] = idx / NTASK;
        tt[j] = idx - tp[j] * NTASK;
    }

    for (;;) {
        __syncthreads();                        // protects s_item, s_pts and s_red reuse
        if (tid == 0) s_item = atomicAdd(meta + 2, 1u);
        __syncthreads();
        const unsigned item = s_item;
        if (item >= nitems) break;
        const unsigned win = item_win[item];
        const unsigned seg = item_seg[item];
        const unsigned wc = wincount[win];
        const long long first = (long long)winstart[win] + (long long)seg * T::CH;
        const int npts = (int)min((unsigned)T::CH, wc - seg * (unsigned)T::CH);
        const int nbatch = (npts + PB - 1) / PB;
        int ws[NDIM];
        {
            unsigned k = win;
#pragma unroll
            for (int d = 0; d < NDIM; ++d) {
                ws[d] = (int)(k % (unsigned)gp.nwin[d]);
                k /= (unsigned)gp.nwin[d];
            }
        }

        // ---- software pipeline registers: permutation entries and gathered point data ----
        unsigned pi[TPT];
        double dx_[TPT], dx2_[NDIM == 4 ? TPT : 1], dy_[TPT], dw_[TPT];
        auto load_perm = [&](int b) {           // permutation entries of batch b
#pragma unroll
            for (int j = 0; j < TPT; ++j) {
                const int p = b * PB + tp[j];
                pi[j] = (tp[j] < PB && p < npts) ? perm[first + p] : 0xffffffffu;
            }
        };
        auto load_data = [&]() {                // gather the points named by pi[]
#pragma unroll
            for (int j = 0; j < TPT; ++j) {
                dx_[j] = 0.0;
                dy_[j] = 0.0;
                dw_[j] = 0.0;
                if (NDIM == 4) dx2_[j] = 0.0;
                if (pi[j] != 0xffffffffu) {
                    const long long i = pi[j];
                    const int d = (NDIM == 4 && tt[j] == 2) ? 2 : tt[j];
                    dx_[j] = (double)x[i * (long long)l1x + d];
                    if (NDIM == 4 && tt[j] == 2) dx2_[j] = (double)x[i * (long long)l1x + 3];
                    if (tt[j] == NTASK - 1) {
                        dy_[j] = (double)y[i];
                        dw_[j] = weighted ? (double)w[i] : 1.0;
                    }
                }
            }
        };
        // ---- stage batch b (held in dx_/dy_/dw_) into its shared-memory buffer ----
        auto stage = [&](int b) {
            const int nb = min(PB, npts - b * PB);
            double *buf = s_pts + (b & 1) * (PB * RS);
#pragma unroll
            for (int j = 0; j < TPT; ++j) {
                const int p = tp[j], t = tt[j];
                if (p < nb) {
                    const int d = (NDIM == 4 && t == 2) ? 2 : t;
                    double bb[4], s[10];
                    int wsd;
                    spl_window_weights_value(dx_[j], gp.xmin[d], gp.dx[d], gp.dxin[d], gp.nodes[d], wsd, bb);
                    {
                        int a = 0;
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int jj = i; jj < 4; ++jj) s[a++] = bb[i] * bb[jj];
                    }
                    double *out = buf + p * RS;
                    if (t == 0) {
#pragma unroll
                        for (int a = 0; a < 10; ++a) out[D::OFF_I + a] = s[a];
#pragma unroll
                        for (int i = 0; i < 4; ++i) out[D::OFF_I + 10 + i] = bb[i];
                    }
                    if (NDIM >= 2 && t == 1) {
#pragma unroll
                        for (int a = 0; a < 10; ++a) out[D::OFF_T2 + a] = s[a];
                        out[D::OFF_T2 + 10] = s[0];
                        out[D::OFF_T2 + 11] = s[1];
#pragma unroll
                        for (int i = 0; i < 4; ++i) out[D::OFF_T2 + 12 + i] = bb[i];
                    }
                    if (t == NTASK - 1) {
                        const double w2 = dw_[j] * dw_[j];      // row = w*phi, rhs = w*y (:806, :837)
                        const double w2y = w2 * dy_[j];
                        if (NDIM <= 2) {
                            out[D::OFF_H + 0] = w2;
                            out[D::OFF_H + 1] = w2y;
                        } else if (NDIM == 3) {
#pragma unroll
                            for (int a = 0; a < 10; ++a) out[D::OFF_H + a] = w2 * s[a];
#pragma unroll
                            for (int i = 0; i < 4; ++i) out[D::OFF_H + 10 + i] = w2y * bb[i];
                        } else {
                            // 4-D: this task owns dimensions 3 (in bb/s) and 4:
                            // H[a4*10+a3] = w2 s4[a4] s3[a3];  H[100 + i4*4+i3] = w2y b4[i4] b3[i3]
                            double b4[4];
                            int ws4;
                            spl_window_weights_value(dx2_[j], gp.xmin[3], gp.dx[3], gp.dxin[3], gp.nodes[3], ws4, b4);
                            int a4 = 0;
#pragma unroll
                            for (int i = 0; i < 4; ++i)
#pragma unroll
                                for (int jj = i; jj < 4; ++jj) {
                                    const double s4 = w2 * (b4[i] * b4[jj]);
#pragma unroll
                                    for (int a3 = 0; a3 < 10; ++a3) out[D::OFF_H + a4 * 10 + a3] = s4 * s[a3];
                                    ++a4;
                                }
#pragma unroll
                            for (int i4 = 0; i4 < 4; ++i4) {
                                const double t4 = w2y * b4[i4];
#pragma unroll
                                for (int i3 = 0; i3 < 4; ++i3) out[D::OFF_H + 100 + i4 * 4 + i3] = t4 * bb[i3];
                            }
                        }
                    }
                }
            }
        };
        if (is_prod) {
            // ================= producers =================
            load_perm(0);
            load_data();
            load_perm(1);
            for (int b = 0; b < nbatch; ++b) {
                if (b >= 2) spl_bar_sync(ACC_BAR_EMPTY + (b & 1), NALL);     // consumers are done with this buffer
                stage(b);
                spl_bar_arrive(ACC_BAR_FULL + (b & 1), NALL);
                if (b + 1 < nbatch) load_data();                            // gathers one batch ahead
                if (b + 2 < nbatch) load_perm(b + 2);                       // permutation two ahead
            }
        } else {
            // ================= consumers =================
            double acc[R][10];
            double racc[APL];
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int a = 0; a < 10; ++a) acc[r][a] = 0.0;
#pragma unroll
            for (int j = 0; j < APL; ++j) racc[j] = 0.0;
            // group grp takes points grp, grp+NG, ... of the batch
            for (int b = 0; b < nbatch; ++b) {
                spl_bar_sync(ACC_BAR_FULL + (b & 1), NALL);
                const int nb = min(PB, npts - b * PB);
                const double *buf = s_pts + (b & 1) * (PB * RS);
#pragma unroll 2
                for (int p = grp; p < nb; p += D::NG) {
                    const double *rec = buf + p * RS;
                    double in[10];
#pragma unroll
                    for (int a = 0; a < 10; a += 2) {
                        const double2 v = *reinterpret_cast<const double2 *>(rec + D::OFF_I + a);
                        in[a] = v.x;
                        in[a + 1] = v.y;
                    }
                    double P[R];
                    if constexpr (NDIM == 1) {
                        P[0] = rec[D::OFF_H];
                    } else {
                        const double2 ta = *reinterpret_cast<const double2 *>(rec + offT);
                        const double2 tb = *reinterpret_cast<const double2 *>(rec + offT + 2);
                        const double ha = rec[offHa], hb = rec[offHb];
                        P[0] = ha * ta.x;
                        P[1] = ha * ta.y;
                        P[2] = hb * tb.x;
                        P[3] = hb * tb.y;
                    }
                    // right-hand side of the same point: APL accumulators per lane
                    double t = rec[offRH];
                    if (NDIM >= 2) t *= rec[offRT];
#pragma unroll
                    for (int j = 0; j < APL; ++j) racc[j] = fma(t, rec[offRI + j], racc[j]);
                    if (!RHS_ONLY) {
#pragma unroll
                        for (int r = 0; r < R; ++r)
#pragma unroll
                            for (int a = 0; a < 10; ++a) acc[r][a] = fma(P[r], in[a], acc[r][a]);
                    }
                }
                if (b + 2 < nbatch) spl_bar_arrive(ACC_BAR_EMPTY + (b & 1), NALL);
            }

            // ---- reduce the K-split groups and flush once per work item ----
            if (T::LPG < 32) {
#pragma unroll
                for (int off = T::LPG; off < 32; off <<= 1) {
#pragma unroll
                    for (int r = 0; r < R; ++r)
#pragma unroll
                        for (int a = 0; a < 10; ++a)
                            acc[r][a] += __shfl_xor_sync(0xffffffffu, acc[r][a], off);
#pragma unroll
                    for (int j = 0; j < APL; ++j) racc[j] += __shfl_xor_sync(0xffffffffu, racc[j], off);
                }
            }
            if (D::NG > 1) {
                constexpr int PER = R * 10 + APL;   // values per lane
                for (int w2_ = 0; w2_ < D::NW; ++w2_) {
                    if (warp == w2_ && lane < D::LPGW) {
                        double *dst = s_red + lane * PER;       // lane == u for the first group of the warp
#pragma unroll
                        for (int r = 0; r < R; ++r)
#pragma unroll
                            for (int a = 0; a < 10; ++a)
                                dst[r * 10 + a] = (w2_ == 0 ? 0.0 : dst[r * 10 + a]) + acc[r][a];
#pragma unroll
                        for (int j = 0; j < APL; ++j)
                            dst[R * 10 + j] = (w2_ == 0 ? 0.0 : dst[R * 10 + j]) + racc[j];
                    }
                    spl_bar_sync(ACC_BAR_CONS, NT);
                }
                for (int idx = tid; idx < D::LPGW * PER; idx += NT) {
                    const int ul = idx / PER;
                    const int k = idx - ul * PER;
                    const double v = s_red[idx];
                    if (k < R * 10) {
                        if (!RHS_ONLY) spl_flush_g<NDIM>(gp, ws, ul, k / 10, k % 10, v, S);
                    } else spl_flush_rhs<NDIM>(gp, ws, ul * APL + (k - R * 10), v, g);
                }
            } else {
                if (!RHS_ONLY) {
#pragma unroll
                    for (int r = 0; r < R; ++r)
#pragma unroll
                        for (int a = 0; a < 10; ++a) spl_flush_g<NDIM>(gp, ws, u, r, a, acc[r][a], S);
                }
#pragma unroll
                for (int j = 0; j < APL; ++j) spl_flush_rhs<NDIM>(gp, ws, u * APL + j, racc[j], g);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// deterministic mode (opt-in; GridParams::fxS): the reference is a serial program and gives the same coefficients every run;
// here the order of the points inside a bin (returning atomics of spl_perm_kernel) and the order in which work items and
// cells add their sums into S / g (FP64 atomics) change from run to run, and the coefficients with them at the level of
// eps * cond(G).  With SPLPAK_B200_DETERMINISTIC=1
//   * every bin's segment of the permutation is sorted (spl_segsort_kernel), so a work item always holds the same points in
//     the same order; on the moment path a work item is a whole cell, so every moment receives exactly one addition;
//   * the sums that several CTAs add to one entry of S / g go through fixed-point limbs with integer atomics
//     (common.cuh: spl_add_S / spl_add_g), in two passes: the first finds the largest |partial sum| (the scale), the
//     second adds; spl_fx_finalize_kernel then adds the exact limb sums to S / g, one rounding per entry and chunk.
// Integer addition commutes, so S, g and -- with the solver's single add per row and panel -- the coefficients are
// bit-for-bit reproducible (tests/test_gpu_fit.py::test_deterministic_mode_is_bit_reproducible).
// ------------------------------------------------------------------------------------------
// In-place ascending sort of every bin's segment of perm (distinct point indices < 2^(8 passes)): LSD radix sort, 8-bit
// digits, one CTA per bin (grid-stride), tiles of 1024 elements ranked stably: match.any inside the warp, per-warp digit
// counts, one scan over the warps per digit.
__global__ void __launch_bounds__(1024)
spl_segsort_kernel(unsigned *__restrict__ perm, unsigned *__restrict__ tmp, const unsigned *__restrict__ binstart,
                   const unsigned *__restrict__ bincount, long long nbins, int passes) {
    __shared__ unsigned s_base[256];
    __shared__ unsigned s_wc[32][256];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (long long bin = blockIdx.x; bin < nbins; bin += gridDim.x) {
        const unsigned c = bincount[bin];
        if (c < 2) continue;
        unsigned *src = perm + binstart[bin], *dst = tmp + binstart[bin];
        for (int pass = 0; pass < passes; ++pass) {
            const int shift = 8 * pass;
            __syncthreads();
            if (tid < 256) s_base[tid] = 0;
            __syncthreads();
            for (unsigned i = tid; i < c; i += 1024) atomicAdd(&s_base[(src[i] >> shift) & 255u], 1u);
            __syncthreads();
            if (warp == 0) {                                    // exclusive scan of the 256 digit counts
                unsigned v[8], sum = 0;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    v[q] = s_base[lane * 8 + q];
                    sum += v[q];
                }
                unsigned incl = sum;
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const unsigned o = __shfl_up_sync(0xffffffffu, incl, off);
                    if (lane >= off) incl += o;
                }
                unsigned run = incl - sum;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    s_base[lane * 8 + q] = run;
                    run += v[q];
                }
            }
            __syncthreads();
            for (unsigned t0 = 0; t0 < c; t0 += 1024) {
                const unsigned i = t0 + tid;
                const bool valid = i < c;
                const unsigned key = valid ? src[i] : 0u;
                const unsigned d = valid ? ((key >> shift) & 255u) : 256u;
                for (int e = tid; e < 32 * 256; e += 1024) (&s_wc[0][0])[e] = 0;
                __syncthreads();
                const unsigned mask = __match_any_sync(0xffffffffu, d);
                const unsigned rank = __popc(mask & ((1u << lane) - 1u));
                if (valid && rank == 0) s_wc[warp][d] = __popc(mask);
                __syncthreads();
                if (tid < 256) {
                    unsigned run = s_base[tid];
#pragma unroll 8
                    for (int w = 0; w < 32; ++w) {
                        const unsigned cnt = s_wc[w][tid];
                        s_wc[w][tid] = run;
                        run += cnt;
                    }
                    s_base[tid] = run;
                }
                __syncthreads();
                if (valid) dst[s_wc[warp][d] + rank] = key;
                __syncthreads();
            }
            unsigned *sw = src;
            src = dst;
            dst = sw;
        }
        if (passes & 1) {                                        // the sorted segment is in tmp
            __syncthreads();
            for (unsigned i = tid; i < c; i += 1024) dst[i] = src[i];
        }
    }
}

// fxe[k] = exponent bound of the pass's partial sums: |v| < 2^fxe for every v recorded in fxmax[k]
__global__ void spl_fx_exponent_kernel(const unsigned long long *__restrict__ fxmax, int *__restrict__ fxe) {
    const int k = threadIdx.x;
    if (k < 2) {
        const double m = __longlong_as_double((long long)fxmax[k]);
        fxe[k] = (m > 0.0 && m < 1.7e308) ? ilogb(m) + 1 : 0;     // inf / NaN sums: any scale, they are dropped as zeros
    }
}

// dst[i] += exact limb sum (one rounding), limbs cleared for the next pass
__global__ void __launch_bounds__(256)
spl_fx_finalize_kernel(double *__restrict__ dst, unsigned long long *__restrict__ limbs, long long n,
                       const int *__restrict__ fxe, int which) {
    const int e = fxe[which];
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        unsigned long long *l = limbs + 3 * i;
        if (l[0] | l[1] | l[2]) {
            dst[i] += spl_fx_value(l, e);
            l[0] = l[1] = l[2] = 0ull;
        }
    }
}

// zero limbs + maxima before a deterministic pass pair; exponent between the passes; finalize after them
int spl_fx_begin(const GridParams &gp, cudaStream_t st) {
    SPL_CUDA_TRY(cudaMemsetAsync(gp.fxmax, 0, 2 * sizeof(unsigned long long), st));
    return SPLPAK_OK;
}
int spl_fx_scale(const GridParams &gp, int *fxe, cudaStream_t st) {
    spl_fx_exponent_kernel<<<1, 32, 0, st>>>(gp.fxmax, fxe);
    ++g_spl_launches;
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}
int spl_fx_finish(const GridParams &gp, double *d_S, double *d_g, cudaStream_t st) {
    if (d_S) {
        const long long n = gp.ncol * gp.nsten;
        spl_fx_finalize_kernel<<<(unsigned)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16), 256, 0, st>>>(d_S, gp.fxS, n, gp.fxe, 0);
        ++g_spl_launches;
    }
    if (d_g) {
        const long long n = gp.ncol;
        spl_fx_finalize_kernel<<<(unsigned)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16), 256, 0, st>>>(d_g, gp.fxg, n, gp.fxe, 1);
        ++g_spl_launches;
    }
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

// ------------------------------------------------------------------------------------------
// host-side launch of the chunk pipeline
// ------------------------------------------------------------------------------------------
#include "moments.cuh"

#define TWOLEVEL_MIN_POINTS (1LL << 21)   // smallest chunk of the two-level partition (pairs and keys are sized for it)

static int spl_acc_chunk_points(int ndim, int moments) {
    if (moments) return MOM_CH;
    switch (ndim) {
    case 1: return AccTraits<1>::CH;
    case 2: return AccTraits<2>::CH;
    case 3: return AccTraits<3>::CH;
    default: return AccTraits<4>::CH;
    }
}

// Bin tables, work counter and (moment path) the per-cell coefficient tables and moment sums.
// SPLPAK_B200_ASSEMBLY=direct keeps 3-D on the direct orthant-stencil accumulation (A/B tests).
int spl_assemble_scratch_init(const GridParams &gp, AssembleScratch &sc, cudaStream_t st) {
    const char *mode = getenv("SPLPAK_B200_ASSEMBLY");
    sc.moments = ((gp.ndim == 3 || gp.ndim == 4) && !(mode && strcmp(mode, "direct") == 0)) ? 1 : 0;
    sc.nbins = gp.nwindows;
    if (sc.moments) {
        long long ncell = 1, ntab = 0;
        for (int d = 0; d < gp.ndim; ++d) {
            ncell *= gp.nodes[d] + 1;
            ntab += gp.nodes[d] + 1;
        }
        // 4-D: 21 KB of moments per cell; beyond 2^31 cells-bytes / 16 GB the direct accumulation is used instead
        const size_t per_cell = gp.ndim == 4 ? MOM4_MG : MOM_MG;
        if (ncell > 0x7fffffffLL || (double)ncell * per_cell * sizeof(double) > 16e9) sc.moments = 0;
        if (sc.moments) sc.nbins = ncell;
    }
    if (sc.moments) {
        long long ntab = 0;
        for (int d = 0; d < gp.ndim; ++d) ntab += gp.nodes[d] + 1;
        const size_t per_cell = gp.ndim == 4 ? MOM4_MG : MOM_MG;
        SPL_CUDA_TRY(cudaMalloc((void **)&sc.celltab, sizeof(double) * (size_t)ntab * MOM_CW));
        SPL_CUDA_TRY(cudaMalloc((void **)&sc.cellmom, sizeof(double) * (size_t)sc.nbins * per_cell));
        SPL_CUDA_TRY(cudaMemsetAsync(sc.cellmom, 0, sizeof(double) * (size_t)sc.nbins * per_cell, st));
        spl_cell_tables_kernel<<<spl_div_up(ntab, 128), 128, 0, st>>>(gp, sc.celltab);
        ++g_spl_launches;
        SPL_CUDA_TRY(cudaGetLastError());
    }
    SPL_CUDA_TRY(cudaMalloc((void **)&sc.wincount, sizeof(unsigned) * (size_t)sc.nbins));
    SPL_CUDA_TRY(cudaMalloc((void **)&sc.winstart, sizeof(unsigned) * (size_t)sc.nbins));
    // one cursor per 32-byte sector when that stays small: packed cursors made neighbouring bins contend in the L2
    // atomic units (measured per 1e8 points: stride 1: 2.33 ms, 8: 2.10 ms, 32: 2.19 ms; SPLPAK_B200_CURSOR_STRIDE
    // overrides, in 4-byte words)
    {
        const char *e = getenv("SPLPAK_B200_CURSOR_STRIDE");
        sc.cursor_stride = e ? atoi(e) : 8;
        if (sc.cursor_stride < 1 || (size_t)sc.nbins * sc.cursor_stride * sizeof(unsigned) > (64u << 20)) sc.cursor_stride = 1;
    }
    SPL_CUDA_TRY(cudaMalloc((void **)&sc.wincursor, sizeof(unsigned) * (size_t)sc.nbins * sc.cursor_stride));
    SPL_CUDA_TRY(cudaMalloc((void **)&sc.itemstart, sizeof(unsigned) * (size_t)sc.nbins));
    SPL_CUDA_TRY(cudaMalloc((void **)&sc.meta, sizeof(unsigned) * 4));
    if (sc.moments) SPL_CUDA_TRY(cudaMalloc((void **)&sc.cursor1, sizeof(unsigned) * 64));
    {
        // limb arrays for S and g, exponents, maxima: always for the constraint rows, for the assembly in the opt-in
        // deterministic mode (see spl_segsort_kernel)
        const char *e = getenv("SPLPAK_B200_DETERMINISTIC");
        sc.deterministic = (e && atoi(e) != 0) ? 1 : 0;
        {
            const size_t nl = 3 * (size_t)(gp.ncol * gp.nsten + gp.ncol);
            SPL_CUDA_TRY(cudaMalloc((void **)&sc.fxS, sizeof(unsigned long long) * nl));
            SPL_CUDA_TRY(cudaMemsetAsync(sc.fxS, 0, sizeof(unsigned long long) * nl, st));
            sc.fxg = sc.fxS + 3 * (size_t)(gp.ncol * gp.nsten);
            SPL_CUDA_TRY(cudaMalloc((void **)&sc.fxmax, sizeof(unsigned long long) * 2));
            SPL_CUDA_TRY(cudaMalloc((void **)&sc.fxe, sizeof(int) * 2));
            SPL_CUDA_TRY(cudaMemsetAsync(sc.fxe, 0, sizeof(int) * 2, st));
        }
    }
    return spl_hist_scratch_init(gp, sc.hist, st);
}

static void free_chunk_arrays(AssembleScratch &sc) {
    unsigned *u[] = {sc.perm, sc.perm2, sc.keys, sc.item_win, sc.item_seg};
    for (unsigned *p : u)
        if (p) cudaFree(p);
    if (sc.yw) cudaFree(sc.yw);
    if (sc.pairs) cudaFree(sc.pairs);
    sc.perm = sc.perm2 = sc.keys = sc.item_win = sc.item_seg = nullptr;
    sc.yw = nullptr;
    sc.pairs = nullptr;
    sc.cap = 0;
}

// Grow-only: the chunk-sized arrays for chunks of up to n points.  The old arrays are released with the synchronising
// cudaFree: the kernels of an earlier chunk may still be reading them.
int spl_assemble_scratch_reserve(const GridParams &gp, AssembleScratch &sc, long long n) {
    if (n <= sc.cap) return SPLPAK_OK;
    free_chunk_arrays(sc);
    sc.max_items = sc.nbins + n / spl_acc_chunk_points(gp.ndim, sc.moments) + 2;
    SPL_CUDA_TRY(cudaMalloc((void **)&sc.perm, sizeof(unsigned) * (size_t)n));
    // deterministic mode: second permutation buffer of the per-bin sort
    if (sc.deterministic) SPL_CUDA_TRY(cudaMalloc((void **)&sc.perm2, sizeof(unsigned) * (size_t)n));
    if (sc.moments) SPL_CUDA_TRY(cudaMalloc((void **)&sc.yw, 2 * sizeof(double) * (size_t)n));
    if (sc.moments && n >= TWOLEVEL_MIN_POINTS) {
        SPL_CUDA_TRY(cudaMalloc((void **)&sc.pairs, sizeof(unsigned long long) * (size_t)n));
        SPL_CUDA_TRY(cudaMalloc((void **)&sc.keys, sizeof(unsigned) * (size_t)n));
    }
    SPL_CUDA_TRY(cudaMalloc((void **)&sc.item_win, sizeof(unsigned) * (size_t)sc.max_items));
    SPL_CUDA_TRY(cudaMalloc((void **)&sc.item_seg, sizeof(unsigned) * (size_t)sc.max_items));
    sc.cap = n;
    return SPLPAK_OK;
}

void spl_assemble_scratch_free(AssembleScratch &sc) {
    free_chunk_arrays(sc);
    unsigned *u[] = {sc.wincount, sc.winstart, sc.wincursor, sc.itemstart, sc.meta};
    for (unsigned *p : u)
        if (p) cudaFree(p);
    if (sc.celltab) cudaFree(sc.celltab);
    if (sc.cellmom) cudaFree(sc.cellmom);
    if (sc.cursor1) cudaFree(sc.cursor1);
    sc.cursor1 = nullptr;
    if (sc.fxS) cudaFree(sc.fxS);
    if (sc.fxmax) cudaFree(sc.fxmax);
    if (sc.fxe) cudaFree(sc.fxe);
    sc.fxS = sc.fxg = sc.fxmax = nullptr;
    sc.fxe = nullptr;
    sc.wincount = sc.winstart = sc.wincursor = sc.itemstart = sc.meta = nullptr;
    sc.celltab = sc.cellmom = nullptr;
    spl_hist_scratch_free(sc.hist);
}

template <int NDIM, bool CELL>
static int assemble_chunk_t(const GridParams &gp, const real_t *d_x, int l1x, const real_t *d_y,
                            const real_t *d_w, int weighted, long long n, int do_hist, int rhs_only,
                            const AssembleScratch &sc, double *d_S, double *d_g, double *d_cnt,
                            double *d_totals, cudaStream_t st, int nsm, cudaEvent_t *ev) {
    using T = AccTraits<NDIM>;
    using D = AccDerived<NDIM>;
    const long long nbins = sc.nbins;
    const bool det = gp.fxS != nullptr;
    // deterministic mode, moment path: a work item is a whole cell (every moment then receives exactly one addition)
    const unsigned ch = CELL ? (det ? 0x7fffffffu : (unsigned)MOM_CH) : (unsigned)T::CH;
    GridParams gp1 = gp;                       // deterministic mode: scale-finding pass
    gp1.fxpass = 1;
    SPL_CUDA_TRY(cudaMemsetAsync(sc.wincount, 0, sizeof(unsigned) * nbins, st));
    SPL_CUDA_TRY(cudaMemsetAsync(sc.wincursor, 0, sizeof(unsigned) * nbins * sc.cursor_stride, st));
    long long nb = (n + 255) / 256;
    const long long cap = (long long)nsm * 8;
    const int grid = (int)(nb < cap ? nb : cap);

    double2 *yw = (CELL && weighted) ? reinterpret_cast<double2 *>(sc.yw) : nullptr;
    bool twolevel = false;
    if constexpr (CELL) {
        // two-level partition for large chunks of many cells (SPLPAK_B200_BINNING=atomic keeps the per-point atomics)
        const char *bm = getenv("SPLPAK_B200_BINNING");
        // (beyond ~1e5 cells a tile of 8,192 points holds less than one point per cell of its buckets: nothing to aggregate)
        twolevel = sc.pairs && sc.keys && n >= TWOLEVEL_MIN_POINTS && nbins >= 2048 && nbins <= 48 * 2048 &&
                   !(bm && strcmp(bm, "atomic") == 0);
    }
    unsigned *keys = twolevel ? sc.keys : nullptr;
    if (ev) cudaEventRecord(ev[0], st);
    {
        // two 512-thread CTAs per SM when the histogram is in shared memory (<= 2 x 96 KB), else 4
        const size_t hist_bytes = sizeof(unsigned) * (size_t)nbins;
        const bool smemh = hist_bytes <= 96 * 1024 && n >= 8 * nbins;
        long long cb = (n + 512LL * BIN_U - 1) / (512LL * BIN_U);
        const long long ccap = (long long)nsm * (smemh ? 2 : 4);
        const int cgrid = (int)(cb < ccap ? (cb < 1 ? 1 : cb) : ccap);
        // both histograms in shared memory: one 1024-thread CTA per SM
        const size_t both_bytes = sizeof(unsigned) * (size_t)((nbins + 1) & ~1LL) + sizeof(double) * (size_t)gp.ncol;
        const bool smemc = smemh && do_hist && both_bytes <= 200 * 1024 && !getenv("SPLPAK_B200_GLOBAL_HIST");
        long long cb1 = (n + 1024LL * BIN_U - 1) / (1024LL * BIN_U);
        const int cgrid1 = (int)(cb1 < nsm ? (cb1 < 1 ? 1 : cb1) : nsm);
        if (do_hist) {
            // points one shared-memory accumulator can receive (its CTA's share) -- the global limbs take 31-bit pieces
            const long long per_acc = smemc ? (n + cgrid1 - 1) / cgrid1 + 1024LL * BIN_U : 1;
            const int rh = spl_hist_prepare(sc.hist, d_w, weighted, n, per_acc, st, nsm);
            if (rh != SPLPAK_OK) return rh;
        }
        if (smemc) {
            auto kern = keys ? spl_classify_kernel<NDIM, true, CELL, true, CELL> : spl_classify_kernel<NDIM, true, CELL, true>;
            SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)both_bytes));
            kern<<<cgrid1, 1024, both_bytes, st>>>(gp, d_x, l1x, d_w, weighted, n, (int)nbins, sc.wincount, do_hist,
                                                   sc.hist.hq, sc.hist.qparams, d_totals, d_y, yw, keys);
        } else if (smemh) {
            auto kern = keys ? spl_classify_kernel<NDIM, true, CELL, false, CELL> : spl_classify_kernel<NDIM, true, CELL>;
            SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_bytes));
            kern<<<cgrid, 512, hist_bytes, st>>>(gp, d_x, l1x, d_w, weighted, n, (int)nbins, sc.wincount, do_hist,
                                                 sc.hist.hq, sc.hist.qparams, d_totals, d_y, yw, keys);
        } else {
            auto kern = keys ? spl_classify_kernel<NDIM, false, CELL, false, CELL> : spl_classify_kernel<NDIM, false, CELL>;
            kern<<<cgrid, 512, 0, st>>>(gp, d_x, l1x, d_w, weighted, n, (int)nbins,
                                                                          sc.wincount, do_hist, sc.hist.hq, sc.hist.qparams,
                                                                          d_totals, d_y, yw, keys);
        }
        if (do_hist) spl_hist_finalize(sc.hist, gp, d_cnt, d_totals, st);
    }
    if (ev) cudaEventRecord(ev[1], st);
    spl_scan_kernel<<<1, 1024, 0, st>>>(sc.wincount, nbins, ch, sc.winstart, sc.itemstart, sc.meta);
    if (twolevel) {
        int shift = 0;
        while (((nbins + (1LL << shift) - 1) >> shift) > 48) ++shift;
        const int nbuckets = (int)((nbins + (1LL << shift) - 1) >> shift);
        int span = 4 << shift;
        while (span > 2 * PART2_NT) span >>= 1;               // spl_block_exscan2: <= 2 counters per thread
        const size_t psmem = sizeof(unsigned) * 2 * (size_t)span + sizeof(uint2) * PART_TILE;
        SPL_CUDA_TRY(cudaMemsetAsync(sc.cursor1, 0, sizeof(unsigned) * 64, st));
        const long long ntiles1 = (n + PART1_TILE - 1) / PART1_TILE;
        const int pgrid1 = (int)(ntiles1 < (long long)nsm * 3 ? ntiles1 : (long long)nsm * 3);
        const long long ntiles = (n + PART_TILE - 1) / PART_TILE;
        const long long pcap = (long long)nsm * (2048 / PART2_NT);
        const int pgrid = (int)(ntiles < pcap ? ntiles : pcap);
        spl_part1_kernel<<<pgrid1, PART1_NT, 0, st>>>(sc.keys, n, sc.winstart, shift, nbuckets, sc.cursor1,
                                                      reinterpret_cast<uint2 *>(sc.pairs));
        SPL_CUDA_TRY(cudaFuncSetAttribute(spl_part2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
        spl_part2_kernel<<<pgrid, PART2_NT, psmem, st>>>(reinterpret_cast<const uint2 *>(sc.pairs), sc.meta, sc.winstart,
                                                     sc.wincursor, sc.cursor_stride, shift, span, nbins, sc.perm);
        ++g_spl_launches;
    } else {
        spl_perm_kernel<NDIM, CELL><<<grid, 256, 0, st>>>(gp, d_x, l1x, d_w, weighted, n, sc.winstart, sc.wincursor,
                                                          sc.cursor_stride, sc.perm);
    }
    spl_items_kernel<<<spl_div_up(nbins, 256), 256, 0, st>>>(sc.wincount, sc.itemstart, nbins, ch, sc.item_win,
                                                             sc.item_seg);
    if (det) {
        int passes = 1;
        while (passes < 4 && (n - 1) >> (8 * passes)) ++passes;
        long long sgrid = nbins < (long long)nsm * 2 ? nbins : (long long)nsm * 2;
        spl_segsort_kernel<<<(unsigned)sgrid, 1024, 0, st>>>(sc.perm, sc.perm2, sc.winstart, sc.wincount, nbins, passes);
        ++g_spl_launches;
        const int rf = spl_fx_begin(gp, st);
        if (rf != SPLPAK_OK) return rf;
    }
    if (ev) cudaEventRecord(ev[2], st);
    const long long max_items = nbins + n / ch + 1;
    if constexpr (CELL && NDIM == 4) {
        const size_t smem = sizeof(double) * (size_t)MOM4_PB * MOM4_RS;
        const size_t tsmem = sizeof(double) * (size_t)MOM4_TSMEM;
        auto kern = rhs_only ? spl_moments4_kernel<true> : spl_moments4_kernel<false>;
        auto tkern = rhs_only ? spl_cell_transform4_kernel<true> : spl_cell_transform4_kernel<false>;
        SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SPL_CUDA_TRY(cudaFuncSetAttribute(tkern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsmem));
        int per_sm = 1;
        SPL_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, MOM4_NT, smem));
        if (per_sm < 1) per_sm = 1;
        long long agrid = (long long)nsm * per_sm;
        if (agrid > max_items) agrid = max_items;
        kern<<<(unsigned)agrid, MOM4_NT, smem, st>>>(gp, d_x, l1x, d_y, yw, sc.perm, sc.wincount, sc.winstart,
                                                     sc.item_win, sc.item_seg, sc.meta, sc.cellmom, ch);
        if (det) {
            tkern<<<(unsigned)nbins, 256, tsmem, st>>>(gp1, sc.wincount, sc.celltab, sc.cellmom, d_S, d_g);
            const int rf = spl_fx_scale(gp, sc.fxe, st);
            if (rf != SPLPAK_OK) return rf;
            ++g_spl_launches;
        }
        tkern<<<(unsigned)nbins, 256, tsmem, st>>>(gp, sc.wincount, sc.celltab, sc.cellmom, d_S, d_g);
        g_spl_launches += 6;
    } else if constexpr (CELL) {
        static_assert(NDIM == 3, "the moment path is 3-D and 4-D");
        const size_t smem = sizeof(double) * (size_t)MOM_PB * MOM_RS;
        auto kern = rhs_only ? spl_moments_kernel<true> : spl_moments_kernel<false>;
        SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 1;
        SPL_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, MOM_NT, smem));
        if (per_sm < 1) per_sm = 1;
        long long agrid = (long long)nsm * per_sm;
        if (agrid > max_items) agrid = max_items;
        kern<<<(unsigned)agrid, MOM_NT, smem, st>>>(gp, d_x, l1x, d_y, yw, sc.perm, sc.wincount, sc.winstart,
                                                    sc.item_win, sc.item_seg, sc.meta, sc.cellmom, ch);
        auto tkern = rhs_only ? spl_cell_transform_kernel<true> : spl_cell_transform_kernel<false>;
        if (det) {
            tkern<<<(unsigned)nbins, 128, 0, st>>>(gp1, sc.wincount, sc.celltab, sc.cellmom, d_S, d_g);
            const int rf = spl_fx_scale(gp, sc.fxe, st);
            if (rf != SPLPAK_OK) return rf;
            ++g_spl_launches;
        }
        tkern<<<(unsigned)nbins, 128, 0, st>>>(gp, sc.wincount, sc.celltab, sc.cellmom, d_S, d_g);
        g_spl_launches += 6;
    } else {
        const size_t smem = sizeof(double) * (2 * (size_t)T::PB * T::RS + (size_t)D::LPGW * (T::R * 10 + D::APL));
        auto kern = rhs_only ? spl_accumulate_kernel<NDIM, true> : spl_accumulate_kernel<NDIM, false>;
        SPL_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 1;
        SPL_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, T::NT + D::NP, smem));
        if (per_sm < 1) per_sm = 1;
        long long agrid = (long long)nsm * per_sm;
        if (agrid > max_items) agrid = max_items;
        if (det) {
            kern<<<(unsigned)agrid, T::NT + D::NP, smem, st>>>(gp1, d_x, l1x, d_y, d_w, weighted, sc.perm, sc.wincount,
                                                               sc.winstart, sc.item_win, sc.item_seg, sc.meta, d_S, d_g);
            const int rf = spl_fx_scale(gp, sc.fxe, st);
            if (rf != SPLPAK_OK) return rf;
            SPL_CUDA_TRY(cudaMemsetAsync(sc.meta + 2, 0, sizeof(unsigned), st));      // work counter of the second pass
            ++g_spl_launches;
        }
        kern<<<(unsigned)agrid, T::NT + D::NP, smem, st>>>(gp, d_x, l1x, d_y, d_w, weighted, sc.perm, sc.wincount,
                                                           sc.winstart, sc.item_win, sc.item_seg, sc.meta, d_S, d_g);
        g_spl_launches += 5;
    }
    if (det) {
        const int rf = spl_fx_finish(gp, rhs_only ? nullptr : d_S, d_g, st);
        if (rf != SPLPAK_OK) return rf;
    }
    if (ev) cudaEventRecord(ev[3], st);
    SPL_CUDA_TRY(cudaGetLastError());
    return SPLPAK_OK;
}

int spl_assemble_chunk(const GridParams &gp, const real_t *d_x, int l1x, const real_t *d_y,
                       const real_t *d_w, int weighted, long long n, int do_hist, int rhs_only,
                       const AssembleScratch &sc, double *d_S, double *d_g, double *d_cnt,
                       double *d_totals, cudaStream_t st, int nsm, cudaEvent_t *ev) {
    switch (gp.ndim) {
    case 1: return assemble_chunk_t<1, false>(gp, d_x, l1x, d_y, d_w, weighted, n, do_hist, rhs_only, sc, d_S, d_g, d_cnt, d_totals, st, nsm, ev);
    case 2: return assemble_chunk_t<2, false>(gp, d_x, l1x, d_y, d_w, weighted, n, do_hist, rhs_only, sc, d_S, d_g, d_cnt, d_totals, st, nsm, ev);
    case 3:
        if (sc.moments) return assemble_chunk_t<3, true>(gp, d_x, l1x, d_y, d_w, weighted, n, do_hist, rhs_only, sc, d_S, d_g, d_cnt, d_totals, st, nsm, ev);
        return assemble_chunk_t<3, false>(gp, d_x, l1x, d_y, d_w, weighted, n, do_hist, rhs_only, sc, d_S, d_g, d_cnt, d_totals, st, nsm, ev);
    case 4:
        if (sc.moments) return assemble_chunk_t<4, true>(gp, d_x, l1x, d_y, d_w, weighted, n, do_hist, rhs_only, sc, d_S, d_g, d_cnt, d_totals, st, nsm, ev);
        return assemble_chunk_t<4, false>(gp, d_x, l1x, d_y, d_w, weighted, n, do_hist, rhs_only, sc, d_S, d_g, d_cnt, d_totals, st, nsm, ev);
    }
    return SPLPAK_ERR_NDIM;
}

#include "ortho.cuh"
