// moments.cuh -- 3-D assembly by CELL MOMENTS (included by assemble.cu).
//
// Inside one grid cell (a node interval in every dimension, or an exterior half-line) every 1-D basis
// function of bascmp (src/splpak.F90:206-389) is ONE polynomial of degree <= 3 in the local coordinate
// t = dxin*(x - x_cell), so every entry of the cell's block of
//     G = sum_p (w phi)(w phi)^T,   g = sum_p (w phi)(w y)              (:806, :837, suprls :1468-1549)
// is a fixed linear function of the cell's power sums.  Per point we therefore accumulate only
//     M[e3][e2][e1] = sum_p w^2   P_e3(t3) P_e2(t2) P_e1(t1),   e = 0..6   (343 values)
//     R[f3][f2][f1] = sum_p w^2 y P_f3(t3) P_f2(t2) P_f1(t1),   f = 0..3   ( 64 values)
// in the shifted Legendre basis P_e on [0,1] (orthogonal, so the change of basis below is well
// conditioned, unlike raw powers), i.e. 407 FMAs per point instead of the 1064 of the direct
// orthant-stencil accumulation -- and once per cell and chunk the moments are mapped to the 10^3 + 4^3
// stencil entries with the per-cell coefficient tables
//     b_i(t) b_j(t) = sum_e C_d[cell][a=(i,j)][e] P_e(t),    b_k(t) = sum_f D_d[cell][k][f] P_f(t),
// which spl_cell_tables_kernel builds by 7-point Gauss projection of the SAME device basis function the
// direct path evaluates (exact for the degree <= 12 integrands up to rounding).
//
// The result differs from the direct path only by rounding (the sums are re-associated), which the
// parity tolerance 10*eps*cond(G) covers by a wide margin; tests/test_gpu_fit.py compares both paths.
#pragma once

#include "basis.cuh"

#define MOM_NE 7                      // Legendre degrees of a pair product b_i b_j
#define MOM_NF 4                      // Legendre degrees of one basis function
#define MOM_CW (10 * MOM_NE + 4 * MOM_NF)   // doubles per (dimension, cell) of the coefficient table
#define MOM_NM 343                    // moments of G per cell
#define MOM_NR 64                     // moments of g per cell
#define MOM_MG 408                    // doubles per cell of the moment array (407 used)
#ifndef MOM_NT
#define MOM_NT 128                    // threads per CTA of the moment kernel (lane = point when staging)
#endif
#define MOM_PB 32                     // points per staged sub-batch (one warp's batch)
#ifndef MOM_MINB
#define MOM_MINB 4                    // CTAs per SM the register allocation aims at
#endif
// staged record of one point (doubles):
//   [0..7] P1[0..6], 0   [8..15] P2[0..6], 0   [16..23] A3[0..6] = w^2 P3, 0   [24..27] B3[0..3] = w^2 y P3
// RS/2 odd: the 128-bit staging stores of neighbouring points do not collide; RS = 14 mod 16: the four points
// {q, q+2, q+4, q+6} of one MMA k-group start 4 (8-byte) banks apart, so the fragment loads are conflict-free.
#define MOM_RS 30
#define MOM_OFF_P2 8
#define MOM_OFF_A3 16
#define MOM_OFF_B3 24
#define MOM_CH 4096                   // max points per work item
#define MOM_NWARP (MOM_NT / 32)

// shifted Legendre polynomials P_0..P_{N-1} at t (z = 2t-1; Bonnet recurrence with constant factors)
template <int N>
__device__ __forceinline__ void spl_legendre(double t, double *P) {
    const double z = fma(2.0, t, -1.0);
    P[0] = 1.0;
    if (N > 1) P[1] = z;
#pragma unroll
    for (int k = 1; k + 1 < N; ++k) {
        const double a = (double)(2 * k + 1) / (double)(k + 1), b = (double)k / (double)(k + 1);
        P[k + 1] = fma(a * z, P[k], -b * P[k - 1]);
    }
}

// One thread per (dimension, cell): coefficient tables C[10][7], D[4][4].
__global__ void __launch_bounds__(128)
spl_cell_tables_kernel(const __grid_constant__ GridParams gp, double *__restrict__ tab) {
    // 7-point Gauss-Legendre rule on [-1, 1]
    const double gz[7] = {0.0, -0.4058451513773972, 0.4058451513773972, -0.7415311855993945,
                          0.7415311855993945, -0.9491079123427585, 0.9491079123427585};
    const double gw[7] = {0.4179591836734694, 0.3818300505051189, 0.3818300505051189, 0.2797053914892766,
                          0.2797053914892766, 0.1294849661688697, 0.1294849661688697};
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    int d = 0;
    long long off = 0;
    for (; d < gp.ndim; ++d) {
        if (idx < gp.nodes[d] + 1) break;
        idx -= gp.nodes[d] + 1;
        off += (long long)(gp.nodes[d] + 1) * MOM_CW;
    }
    if (d >= gp.ndim) return;
    const int nod = gp.nodes[d], ic = idx, it = ic - 1;
    const int ws = min(max(it - 1, 0), nod - 4);
    const bool exterior = (ic == 0) || (ic == nod);
    double bq[7][4], Pq[7][MOM_NE];
    const double x0 = gp.xmin[d] + (double)it * gp.dx[d];
    for (int q = 0; q < 7; ++q) {
        const double tq = 0.5 * (1.0 + gz[q]);
        const double x = x0 + tq * gp.dx[d];
        // local coordinate exactly as the moment kernel forms it, so the projection sees the same t
        const double tl = spl_mul(gp.dxin[d], spl_sub(x, spl_add(gp.xmin[d], spl_mul((double)it, gp.dx[d]))));
        for (int k = 0; k < 4; ++k) bq[q][k] = spl_bas1_value(ws + k, nod, x, gp.xmin[d], gp.dx[d], gp.dxin[d]);
        spl_legendre<MOM_NE>(tl, Pq[q]);
    }
    double *C = tab + off + (long long)ic * MOM_CW;
    double *D = C + 10 * MOM_NE;
    for (int a = 0; a < 10; ++a) {
        int i, j;
        spl_pair(a, i, j);
        for (int e = 0; e < MOM_NE; ++e) {
            double s = 0.0;
            for (int q = 0; q < 7; ++q) s += 0.5 * gw[q] * bq[q][i] * bq[q][j] * Pq[q][e];
            // on an exterior half-line the basis is linear: degrees > 2 vanish identically (and their
            // moments may overflow for far-away points, so they must not be touched)
            C[a * MOM_NE + e] = (exterior && e > 2) ? 0.0 : (double)(2 * e + 1) * s;
        }
    }
    for (int k = 0; k < 4; ++k)
        for (int f = 0; f < MOM_NF; ++f) {
            double s = 0.0;
            for (int q = 0; q < 7; ++q) s += 0.5 * gw[q] * bq[q][k] * Pq[q][f];
            D[k * MOM_NF + f] = (exterior && f > 1) ? 0.0 : (double)(2 * f + 1) * s;
        }
}

__device__ __forceinline__ void spl_mom_dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// Persistent CTAs over work items (cell, segment of <= MOM_CH points).  A work item is cut into sub-batches of MOM_PB = 32
// points; warp w owns sub-batches w, w + MOM_NWARP, w + 2 MOM_NWARP, ... (a static split, so the order of every warp's
// sums, and with it the deterministic mode, does not depend on timing).  Per sub-batch the warp alone runs
//   stage   lane = point: gather through the permutation (prefetched one sub-batch ahead, the permutation two ahead),
//           Legendre values of the three local coordinates -> P1, P2, w^2 P3, w^2 y P3 into the warp's private slice of
//           shared memory (28 doubles per point);
//   accumulate   the moment sums are a GEMM over the points, M[(e3,e2)][e1] = sum_p (A3[e3] P2[e2])_p P1[e1]_p,
//           run on the FP64 tensor cores (mma.sync.m8n8k4.f64 -> DMMA.8x8x4): k = 4 points, n = e1 (7 of 8
//           columns), one m-tile of rows e2 (7 of 8) per e3, plus two tiles (rows (f3, f2)) for the
//           right-hand side.  Lane (r, k) multiplies its own A fragment A3[e3]*P2[r] of point k; the B
//           fragment P1[r] is ONE shared-memory load per 4 points, where the DFMA form needed 7 broadcast
//           loads per point -- the kernel is bound by the shared-memory pipe, not by FP64 issue.
// The two phases are separated by __syncwarp only; the CTA meets at a barrier just at the work-item claim and at the
// reduction.  Warps therefore drift apart, and the scheduler overlaps one warp's FP64 staging with another's DMMA
// stream.  (A CTA-wide batch through one buffer, with two barriers per batch, held every warp to the slowest one twice
// per batch.)  One slice per warp, not two: 2 x 32 x MOM_RS doubles per warp would not fit 16 warps per SM in shared
// memory, and holding the next sub-batch's Legendre values in registers across the DMMA stream would spill.
template <bool RHS_ONLY>
__global__ void __launch_bounds__(MOM_NT, MOM_MINB)
spl_moments_kernel(const __grid_constant__ GridParams gp, const real_t *__restrict__ x, int l1x,
                   const real_t *__restrict__ y, const double2 *__restrict__ yw,
                   const unsigned *__restrict__ perm, const unsigned *__restrict__ bincount,
                   const unsigned *__restrict__ binstart, const unsigned *__restrict__ item_bin,
                   const unsigned *__restrict__ item_seg, unsigned *__restrict__ meta,
                   double *__restrict__ MG, const unsigned ch) {
    // ch: points per work item (MOM_CH; deterministic mode: a whole cell, so that every moment receives ONE addition)
    extern __shared__ __align__(16) double s_pts[];          // MOM_NWARP x MOM_PB x MOM_RS, reused for the reduction
    __shared__ unsigned s_item;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int fr = lane >> 2, fk = lane & 3;                // MMA fragment coordinates of this lane
    const int frr = fr & 3, frh = fr >> 2;
    double *const s_warp = s_pts + warp * (MOM_PB * MOM_RS);
    const unsigned nitems = meta[0];
    const int nc1 = gp.nodes[0] + 1, nc2 = gp.nodes[1] + 1;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(meta + 2, 1u);
        __syncthreads();
        const unsigned item = s_item;
        if (item >= nitems) break;
        const unsigned cell = item_bin[item];
        const unsigned seg = item_seg[item];
        const long long first = (long long)binstart[cell] + (long long)seg * ch;
        const int npts = (int)min(ch, bincount[cell] - seg * ch);
        const int nsub = (npts + MOM_PB - 1) / MOM_PB;
        double xc[3];                                        // left end of the cell per dimension (:246 form)
        {
            const int c1 = (int)(cell % (unsigned)nc1), c2 = (int)((cell / (unsigned)nc1) % (unsigned)nc2),
                      c3 = (int)(cell / (unsigned)(nc1 * nc2));
            xc[0] = spl_add(gp.xmin[0], spl_mul((double)(c1 - 1), gp.dx[0]));
            xc[1] = spl_add(gp.xmin[1], spl_mul((double)(c2 - 1), gp.dx[1]));
            xc[2] = spl_add(gp.xmin[2], spl_mul((double)(c3 - 1), gp.dx[2]));
        }
        double acc[MOM_NE][2], racc[2][2];                   // C fragments: tile e3 (rows e2), rhs tiles
#pragma unroll
        for (int e = 0; e < MOM_NE; ++e) acc[e][0] = acc[e][1] = 0.0;
        racc[0][0] = racc[0][1] = racc[1][0] = racc[1][1] = 0.0;

        // pn: permutation entry of the sub-batch AFTER the one held in px/py/pw.  The entry a gather uses is
        // first copied to a fresh register: overwriting the register the in-flight gathers were addressed
        // from made the next permutation load wait on their scoreboard (a full memory latency per batch).
        unsigned pn;
        double px[3], py, pw;
        auto load_perm = [&](int k) {
            const int p = k * MOM_PB + lane;
            pn = (k < nsub && p < npts) ? perm[first + p] : 0xffffffffu;
        };
        auto load_data = [&](unsigned pc) {
            px[0] = px[1] = px[2] = 0.0;
            py = 0.0;
            pw = 0.0;
            if (pc != 0xffffffffu) {
                const long long i = pc;
                px[0] = (double)x[i * (long long)l1x + 0];
                px[1] = (double)x[i * (long long)l1x + 1];
                px[2] = (double)x[i * (long long)l1x + 2];
                if (yw) {                                    // weighted: interleaved (y, w) copy written by classify
                    const double2 v = __ldg(yw + i);
                    py = v.x;
                    pw = v.y;
                } else {
                    py = (double)y[i];
                    pw = 1.0;
                }
            }
        };
        load_perm(warp);
        load_data(pn);
        load_perm(warp + MOM_NWARP);
        for (int k = warp; k < nsub; k += MOM_NWARP) {
            const int nb = min(MOM_PB, npts - k * MOM_PB);
            // ---- stage ----
            if (lane < nb) {
                double P1[MOM_NE], P2[MOM_NE], P3[MOM_NE];
                spl_legendre<MOM_NE>(spl_mul(gp.dxin[0], spl_sub(px[0], xc[0])), P1);
                spl_legendre<MOM_NE>(spl_mul(gp.dxin[1], spl_sub(px[1], xc[1])), P2);
                spl_legendre<MOM_NE>(spl_mul(gp.dxin[2], spl_sub(px[2], xc[2])), P3);
                const double w2 = pw * pw;                       // row = w*phi, rhs = w*y (:806, :837)
                const double w2y = w2 * py;
                double *rec = s_warp + lane * MOM_RS;
#pragma unroll
                for (int e = 0; e < 8; e += 2) {
                    *reinterpret_cast<double2 *>(rec + e) = make_double2(P1[e], e + 1 < MOM_NE ? P1[e + 1] : 0.0);
                    *reinterpret_cast<double2 *>(rec + MOM_OFF_P2 + e) = make_double2(P2[e], e + 1 < MOM_NE ? P2[e + 1] : 0.0);
                }
                if (!RHS_ONLY) {
#pragma unroll
                    for (int e = 0; e < 8; e += 2)
                        *reinterpret_cast<double2 *>(rec + MOM_OFF_A3 + e) =
                            make_double2(w2 * P3[e], e + 1 < MOM_NE ? w2 * P3[e + 1] : 0.0);
                }
                *reinterpret_cast<double2 *>(rec + MOM_OFF_B3) = make_double2(w2y * P3[0], w2y * P3[1]);
                *reinterpret_cast<double2 *>(rec + MOM_OFF_B3 + 2) = make_double2(w2y * P3[2], w2y * P3[3]);
            } else if (lane < ((nb + 7) & ~7)) {
                // the MMA consumes whole groups of 8 points: pad the last group with zero records
                double *rec = s_warp + lane * MOM_RS;
#pragma unroll
                for (int e = 0; e < 28; e += 2) *reinterpret_cast<double2 *>(rec + e) = make_double2(0.0, 0.0);
            }
            __syncwarp();
            {
                const unsigned pc = pn;
                load_perm(k + 2 * MOM_NWARP);                    // permutation two sub-batches ahead
                if (k + MOM_NWARP < nsub) load_data(pc);         // gathers of the next sub-batch fly under the DMMAs
            }
            // ---- accumulate ----
            // unrolled over the (at most four) groups of 8 points, so the fragment loads of one group are issued under
            // the DMMAs of the previous one: 4.81 -> 4.54 ms at cfg3 (B200, 1000 W) against a loop bounded by nb
            const int ng = (nb + 7) >> 3;
#pragma unroll
            for (int g = 0; g < MOM_PB / 8; ++g) {
                if (g >= ng) break;
                const int p0 = 8 * g;
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const double *rec = s_warp + (p0 + half + 2 * fk) * MOM_RS;     // point of this lane's k
                    const double bfrag = rec[fr];                                    // B[k][n = fr] = P1[fr]
                    const double p2r = rec[MOM_OFF_P2 + frr];
                    const double b30 = rec[MOM_OFF_B3 + frh], b31 = rec[MOM_OFF_B3 + 2 + frh];
                    spl_mom_dmma(racc[0][0], racc[0][1], b30 * p2r, bfrag);        // rows (f3 = frh, f2 = frr)
                    spl_mom_dmma(racc[1][0], racc[1][1], b31 * p2r, bfrag);        // rows (f3 = 2 + frh, f2 = frr)
                    if (!RHS_ONLY) {
                        const double p2 = rec[MOM_OFF_P2 + fr];
                        double a3[8];
#pragma unroll
                        for (int e = 0; e < 8; e += 2) {
                            const double2 v = *reinterpret_cast<const double2 *>(rec + MOM_OFF_A3 + e);
                            a3[e] = v.x;
                            a3[e + 1] = v.y;
                        }
#pragma unroll
                        for (int e = 0; e < MOM_NE; ++e) spl_mom_dmma(acc[e][0], acc[e][1], a3[e] * p2, bfrag);
                    }
                }
            }
            __syncwarp();                                        // every lane has read the slice before it is restaged
        }
        // ---- reduce the warps through shared memory (over their slices: all must be done), flush once per work item ----
        __syncthreads();
        {
            // C fragment: rows fr, columns 2 fk + {0, 1}
            double *red = s_pts + warp * MOM_MG;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int col = 2 * fk + j;
                if (!RHS_ONLY && fr < MOM_NE && col < MOM_NE) {
#pragma unroll
                    for (int e = 0; e < MOM_NE; ++e) red[(e * MOM_NE + fr) * MOM_NE + col] = acc[e][j];
                }
                if (col < MOM_NF) {
                    red[MOM_NM + (frh * 4 + frr) * MOM_NF + col] = racc[0][j];
                    red[MOM_NM + ((2 + frh) * 4 + frr) * MOM_NF + col] = racc[1][j];
                }
            }
        }
        __syncthreads();
        double *dst = MG + (long long)cell * MOM_MG;
        for (int k = (RHS_ONLY ? MOM_NM : 0) + tid; k < MOM_NM + MOM_NR; k += MOM_NT) {
            double v = 0.0;
#pragma unroll
            for (int q = 0; q < MOM_NWARP; ++q) v += s_pts[q * MOM_MG + k];
            if (v != 0.0) atomicAdd(dst + k, v);
        }
    }
}

// One CTA per non-empty cell: moments -> stencil entries (three 1-D changes of basis), added into S / g.
// The cell's moments are zeroed after they are read, so the array is clean for the next chunk.
template <bool RHS_ONLY>
__global__ void __launch_bounds__(128)
spl_cell_transform_kernel(const __grid_constant__ GridParams gp, const unsigned *__restrict__ bincount,
                          const double *__restrict__ tab, double *__restrict__ MG, double *__restrict__ S,
                          double *__restrict__ g) {
    const unsigned cell = blockIdx.x;
    if (bincount[cell] == 0u) return;
    __shared__ double s_M[MOM_NM + MOM_NR];
    __shared__ double s_C[3][MOM_CW];
    __shared__ double s_T1[49 * 10], s_T2[7 * 100];
    __shared__ double s_U1[16 * 4], s_U2[4 * 16];
    const int tid = threadIdx.x;
    const int nc1 = gp.nodes[0] + 1, nc2 = gp.nodes[1] + 1;
    int c[3], ws[3];
    c[0] = (int)(cell % (unsigned)nc1);
    c[1] = (int)((cell / (unsigned)nc1) % (unsigned)nc2);
    c[2] = (int)(cell / (unsigned)(nc1 * nc2));
    long long toff = 0;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        ws[d] = min(max(c[d] - 2, 0), gp.nodes[d] - 4);
        const double *src = tab + toff + (long long)c[d] * MOM_CW;
        for (int k = tid; k < MOM_CW; k += blockDim.x) s_C[d][k] = src[k];
        toff += (long long)(gp.nodes[d] + 1) * MOM_CW;
    }
    double *mg = MG + (long long)cell * MOM_MG;
    {
        // the thread's four moments in flight together (a load / store-zero loop made one DRAM round trip per element)
        constexpr int NL = (MOM_NM + MOM_NR + 127) / 128;
        double v[NL];
#pragma unroll
        for (int q = 0; q < NL; ++q) {
            const int k = tid + 128 * q;
            v[q] = (k < MOM_NM + MOM_NR && (!RHS_ONLY || k >= MOM_NM)) ? __ldcg(mg + k) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < NL; ++q) {
            const int k = tid + 128 * q;
            if (k < MOM_NM + MOM_NR && (!RHS_ONLY || k >= MOM_NM)) {
                if (!gp.fxpass) __stcg(mg + k, 0.0);      // (the scale-finding pass of the deterministic mode reads only)
                s_M[k] = v[q];
            }
        }
    }
    __syncthreads();
    // a zero coefficient must skip its moment (it may be inf/NaN for a far exterior point)
    auto mac = [](double cf, double m, double s) { return cf != 0.0 ? fma(cf, m, s) : s; };
    if (!RHS_ONLY) {
        for (int k = tid; k < 490; k += blockDim.x) {           // T1[o][a1]
            const int o = k / 10, a1 = k - o * 10;
            double s = 0.0;
#pragma unroll
            for (int e = 0; e < MOM_NE; ++e) s = mac(s_C[0][a1 * MOM_NE + e], s_M[o * MOM_NE + e], s);
            s_T1[k] = s;
        }
    }
    if (tid < 64) {                                              // U1[ro][i1]
        const int ro = tid >> 2, i1 = tid & 3;
        double s = 0.0;
#pragma unroll
        for (int f = 0; f < MOM_NF; ++f) s = mac(s_C[0][70 + i1 * MOM_NF + f], s_M[MOM_NM + ro * MOM_NF + f], s);
        s_U1[tid] = s;
    }
    __syncthreads();
    if (!RHS_ONLY) {
        for (int k = tid; k < 700; k += blockDim.x) {           // T2[e3][a2][a1]
            const int e3 = k / 100, r = k - e3 * 100, a2 = r / 10, a1 = r - a2 * 10;
            double s = 0.0;
#pragma unroll
            for (int e = 0; e < MOM_NE; ++e) s = mac(s_C[1][a2 * MOM_NE + e], s_T1[(e3 * MOM_NE + e) * 10 + a1], s);
            s_T2[k] = s;
        }
    }
    if (tid < 64) {                                              // U2[f3][i2][i1]
        const int f3 = tid >> 4, i2 = (tid >> 2) & 3, i1 = tid & 3;
        double s = 0.0;
#pragma unroll
        for (int f = 0; f < MOM_NF; ++f) s = mac(s_C[1][70 + i2 * MOM_NF + f], s_U1[(f3 * 4 + f) * 4 + i1], s);
        s_U2[tid] = s;
    }
    __syncthreads();
    if (!RHS_ONLY) {
        for (int k = tid; k < 1000; k += blockDim.x) {          // S[a3][a2][a1]
            const int a3 = k / 100, r = k - a3 * 100;
            double s = 0.0;
#pragma unroll
            for (int e = 0; e < MOM_NE; ++e) s = mac(s_C[2][a3 * MOM_NE + e], s_T2[e * 100 + r], s);
            if (s != 0.0) {
                const int a[3] = {r % 10, r / 10, a3};
                long long node = 0, nstride = 1;
                int sten = 0, sstride = 1;
#pragma unroll
                for (int d = 0; d < 3; ++d) {
                    int i, j;
                    spl_pair(a[d], i, j);
                    node += (long long)(ws[d] + i) * nstride;
                    sten += (j - i) * sstride;
                    nstride *= gp.nodes[d];
                    sstride *= 4;
                }
                spl_add_S(gp, S, node * gp.nsten + sten, s);
            }
        }
    }
    if (tid < 64) {                                              // g[i3][i2][i1]
        const int i3 = tid >> 4, r = tid & 15;
        double s = 0.0;
#pragma unroll
        for (int f = 0; f < MOM_NF; ++f) s = mac(s_C[2][70 + i3 * MOM_NF + f], s_U2[f * 16 + r], s);
        if (s != 0.0) {
            const long long node = (long long)(ws[0] + (r & 3)) + (long long)(ws[1] + (r >> 2)) * gp.nodes[0] +
                                   (long long)(ws[2] + i3) * gp.nodes[0] * gp.nodes[1];
            spl_add_g(gp, g, node, s);
        }
    }
}

// ------------------------------------------------------------------------------------------
// 4-D: the same construction with one more factor (round 2).
//     M[e4][e3][e2][e1] = sum_p w^2   P_e4(t4) P_e3(t3) P_e2(t2) P_e1(t1),   e = 0..6   (2,401 values)
//     R[f4][f3][f2][f1] = sum_p w^2 y P_f4(t4) P_f3(t3) P_f2(t2) P_f1(t1),   f = 0..3   (  256 values)
// i.e. 2,657 FMAs per point against the 10^4 + 4^4 of the direct orthant-stencil accumulation.  As a GEMM over the
// points: rows (e4, e3, e2), columns e1, k = 4 points per DMMA.8x8x4 -- 49 m-tiles (e4, e3) with rows e2 plus 8 tiles
// (f4, f3 half) with rows (f3, f2) for the right-hand side, 57 DMMA per 4 points.  114 accumulator doubles do not fit
// one warp, so the M dimension is split over the CTA's eight warps and EVERY warp walks all the points of the batch:
// warp e4 < 7 owns the seven tiles (e4, e3 = 0..6), warp 7 the eight right-hand-side tiles (14 + 14 + 14 + 15 DMMA per
// 4 points on the four SM sub-partitions).  Nothing is reduced across warps; a work item ends with each warp adding
// its own fragment entries to the cell's moment array.
// Staged record of one point (doubles):
//   [0..7] P1, 0   [8..15] P2, 0   [16..23] P3, 0   [24..31] A4 = w^2 P4, 0   [32..35] B4 = w^2 y P4[0..3]
// MOM4_RS = 46: RS/2 odd and RS = 14 mod 16, the bank argument of MOM_RS.
// ------------------------------------------------------------------------------------------
#define MOM4_NM 2401
#define MOM4_NR 256
#define MOM4_MG 2664                  // doubles per cell (2,657 used)
#define MOM4_NT 256
#define MOM4_PB 256
#define MOM4_RS 46
#define MOM4_OFF_P2 8
#define MOM4_OFF_P3 16
#define MOM4_OFF_A4 24
#define MOM4_OFF_B4 32

template <bool RHS_ONLY>
__global__ void __launch_bounds__(MOM4_NT, 2)
spl_moments4_kernel(const __grid_constant__ GridParams gp, const real_t *__restrict__ x, int l1x,
                    const real_t *__restrict__ y, const double2 *__restrict__ yw,
                    const unsigned *__restrict__ perm, const unsigned *__restrict__ bincount,
                    const unsigned *__restrict__ binstart, const unsigned *__restrict__ item_bin,
                    const unsigned *__restrict__ item_seg, unsigned *__restrict__ meta,
                    double *__restrict__ MG, const unsigned ch) {
    extern __shared__ __align__(16) double s_pts[];          // MOM4_PB x MOM4_RS
    __shared__ unsigned s_item;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int fr = lane >> 2, fk = lane & 3;                // MMA fragment coordinates of this lane
    const int frr = fr & 3, frh = fr >> 2;
    const unsigned nitems = meta[0];
    for (;;) {
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(meta + 2, 1u);
        __syncthreads();
        const unsigned item = s_item;
        if (item >= nitems) break;
        const unsigned cell = item_bin[item];
        const unsigned seg = item_seg[item];
        const long long first = (long long)binstart[cell] + (long long)seg * ch;
        const int npts = (int)min(ch, bincount[cell] - seg * ch);
        const int nbatch = (npts + MOM4_PB - 1) / MOM4_PB;
        double xc[4];                                        // left end of the cell per dimension (:246 form)
        {
            unsigned c = cell;
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                const unsigned ncd = (unsigned)(gp.nodes[d] + 1);
                const int cd = (int)(c % ncd);
                c /= ncd;
                xc[d] = spl_add(gp.xmin[d], spl_mul((double)(cd - 1), gp.dx[d]));
            }
        }
        double acc[8][2];                                    // warps 0..6: tiles e3 = 0..6; warp 7: tiles (f4, half)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e][0] = acc[e][1] = 0.0;

        unsigned pn;
        double px[4], py, pw;
        auto load_perm = [&](int b) {
            const int p = b * MOM4_PB + tid;
            pn = (b < nbatch && p < npts) ? perm[first + p] : 0xffffffffu;
        };
        auto load_data = [&](unsigned pc) {
            px[0] = px[1] = px[2] = px[3] = 0.0;
            py = 0.0;
            pw = 0.0;
            if (pc != 0xffffffffu) {
                const long long i = pc;
#pragma unroll
                for (int d = 0; d < 4; ++d) px[d] = (double)x[i * (long long)l1x + d];
                if (yw) {                                    // weighted: interleaved (y, w) copy written by classify
                    const double2 v = __ldg(yw + i);
                    py = v.x;
                    pw = v.y;
                } else {
                    py = (double)y[i];
                    pw = 1.0;
                }
            }
        };
        load_perm(0);
        load_data(pn);
        load_perm(1);
        for (int b = 0; b < nbatch; ++b) {
            const int nb = min(MOM4_PB, npts - b * MOM4_PB);
            // ---- stage ----
            if (tid < nb) {
                double P[MOM_NE];
                double *rec = s_pts + tid * MOM4_RS;
#pragma unroll
                for (int d = 0; d < 3; ++d) {
                    spl_legendre<MOM_NE>(spl_mul(gp.dxin[d], spl_sub(px[d], xc[d])), P);
#pragma unroll
                    for (int e = 0; e < 8; e += 2)
                        *reinterpret_cast<double2 *>(rec + 8 * d + e) = make_double2(P[e], e + 1 < MOM_NE ? P[e + 1] : 0.0);
                }
                spl_legendre<MOM_NE>(spl_mul(gp.dxin[3], spl_sub(px[3], xc[3])), P);
                const double w2 = pw * pw;                       // row = w*phi, rhs = w*y (:806, :837)
                const double w2y = w2 * py;
                if (!RHS_ONLY) {
#pragma unroll
                    for (int e = 0; e < 8; e += 2)
                        *reinterpret_cast<double2 *>(rec + MOM4_OFF_A4 + e) =
                            make_double2(w2 * P[e], e + 1 < MOM_NE ? w2 * P[e + 1] : 0.0);
                }
                *reinterpret_cast<double2 *>(rec + MOM4_OFF_B4) = make_double2(w2y * P[0], w2y * P[1]);
                *reinterpret_cast<double2 *>(rec + MOM4_OFF_B4 + 2) = make_double2(w2y * P[2], w2y * P[3]);
            } else if (tid < ((nb + 7) & ~7)) {
                // the MMA consumes whole groups of 8 points: pad the last group with zero records
                double *rec = s_pts + tid * MOM4_RS;
#pragma unroll
                for (int e = 0; e < 36; e += 2) *reinterpret_cast<double2 *>(rec + e) = make_double2(0.0, 0.0);
            }
            __syncthreads();
            {
                const unsigned pc = pn;
                load_perm(b + 2);                                // permutation two batches ahead
                if (b + 1 < nbatch) load_data(pc);               // gathers of the next batch fly under the MMAs
            }
            // ---- accumulate: every warp walks all the points ----
            if (warp < 7) {
                if (!RHS_ONLY) {
                    for (int p0 = 0; p0 < nb; p0 += 8) {
#pragma unroll
                        for (int half = 0; half < 2; ++half) {
                            const double *rec = s_pts + (p0 + half + 2 * fk) * MOM4_RS;   // point of this lane's k
                            const double bfrag = rec[fr];                                  // B[k][n = fr] = P1[fr]
                            const double a4p2 = rec[MOM4_OFF_A4 + warp] * rec[MOM4_OFF_P2 + fr];
                            double p3[8];
#pragma unroll
                            for (int e = 0; e < 8; e += 2) {
                                const double2 v = *reinterpret_cast<const double2 *>(rec + MOM4_OFF_P3 + e);
                                p3[e] = v.x;
                                p3[e + 1] = v.y;
                            }
#pragma unroll
                            for (int e = 0; e < MOM_NE; ++e) spl_mom_dmma(acc[e][0], acc[e][1], a4p2 * p3[e], bfrag);
                        }
                    }
                }
            } else {
                for (int p0 = 0; p0 < nb; p0 += 8) {
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        const double *rec = s_pts + (p0 + half + 2 * fk) * MOM4_RS;
                        const double bfrag = rec[fr];
                        const double p2r = rec[MOM4_OFF_P2 + frr];
                        const double q0 = rec[MOM4_OFF_P3 + frh] * p2r;              // rows (f3 = frh, f2 = frr)
                        const double q1 = rec[MOM4_OFF_P3 + 2 + frh] * p2r;          // rows (f3 = 2 + frh, f2 = frr)
                        const double2 b01 = *reinterpret_cast<const double2 *>(rec + MOM4_OFF_B4);
                        const double2 b23 = *reinterpret_cast<const double2 *>(rec + MOM4_OFF_B4 + 2);
                        spl_mom_dmma(acc[0][0], acc[0][1], b01.x * q0, bfrag);
                        spl_mom_dmma(acc[1][0], acc[1][1], b01.x * q1, bfrag);
                        spl_mom_dmma(acc[2][0], acc[2][1], b01.y * q0, bfrag);
                        spl_mom_dmma(acc[3][0], acc[3][1], b01.y * q1, bfrag);
                        spl_mom_dmma(acc[4][0], acc[4][1], b23.x * q0, bfrag);
                        spl_mom_dmma(acc[5][0], acc[5][1], b23.x * q1, bfrag);
                        spl_mom_dmma(acc[6][0], acc[6][1], b23.y * q0, bfrag);
                        spl_mom_dmma(acc[7][0], acc[7][1], b23.y * q1, bfrag);
                    }
                }
            }
            __syncthreads();
        }
        // ---- flush: C fragment rows fr, columns 2 fk + {0, 1}; every warp owns its moments ----
        double *dst = MG + (long long)cell * MOM4_MG;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int col = 2 * fk + j;
            if (warp < 7) {
                if (!RHS_ONLY && fr < MOM_NE && col < MOM_NE) {
#pragma unroll
                    for (int e = 0; e < MOM_NE; ++e) {
                        const double v = acc[e][j];
                        if (v != 0.0) atomicAdd(dst + ((warp * MOM_NE + e) * MOM_NE + fr) * MOM_NE + col, v);
                    }
                }
            } else if (col < MOM_NF) {
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    const int f4 = t >> 1, f3 = 2 * (t & 1) + frh;
                    const double v = acc[t][j];
                    if (v != 0.0) atomicAdd(dst + MOM4_NM + ((f4 * 4 + f3) * 4 + frr) * MOM_NF + col, v);
                }
            }
        }
    }
}

// One CTA per non-empty cell: four 1-D changes of basis 2401 -> 343 x 10 -> 49 x 100 -> 7 x 1000 -> 10^4 (+ 256 -> 256
// for g), added into S / g; the cell's moments are zeroed after they are read.
// Shared memory (doubles): R1 [7000]: the moments (2,657) and T1 (3,430), later T3 (7,000) | R2 [4900]: T2 |
// coefficient tables 4 x MOM_CW | U [3 x 256].
#define MOM4_R1 7000
#define MOM4_R2 4900
#define MOM4_TSMEM (MOM4_R1 + MOM4_R2 + 4 * MOM_CW + 3 * 256)
template <bool RHS_ONLY>
__global__ void __launch_bounds__(256)
spl_cell_transform4_kernel(const __grid_constant__ GridParams gp, const unsigned *__restrict__ bincount,
                           const double *__restrict__ tab, double *__restrict__ MG, double *__restrict__ S,
                           double *__restrict__ g) {
    const unsigned cell = blockIdx.x;
    if (bincount[cell] == 0u) return;
    extern __shared__ __align__(16) double s_t4[];
    double *s_M = s_t4;                       // [2657]
    double *s_T1 = s_t4 + 2664;               // [343][10]
    double *s_T3 = s_t4;                      // [7][1000]   (over M and T1, both dead by then)
    double *s_T2 = s_t4 + MOM4_R1;            // [49][100]
    double *s_C = s_T2 + MOM4_R2;             // [4][MOM_CW]
    double *s_U1 = s_C + 4 * MOM_CW, *s_U2 = s_U1 + 256, *s_U3 = s_U2 + 256;
    const int tid = threadIdx.x;
    int ws[4], ext = 0;                       // ext: bit d set when the cell is an exterior half-line in dimension d
    {
        unsigned c = cell;
        long long toff = 0;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            const unsigned ncd = (unsigned)(gp.nodes[d] + 1);
            const int cd = (int)(c % ncd);
            c /= ncd;
            ws[d] = min(max(cd - 2, 0), gp.nodes[d] - 4);
            if (cd == 0 || cd == gp.nodes[d]) ext |= 1 << d;
            const double *src = tab + toff + (long long)cd * MOM_CW;
            for (int k = tid; k < MOM_CW; k += blockDim.x) s_C[d * MOM_CW + k] = src[k];
            toff += (long long)(gp.nodes[d] + 1) * MOM_CW;
        }
    }
    // Moments of a degree the cell's table has no coefficient for (exterior half-lines: degrees > 2 of G, > 1 of g; they may
    // be inf / NaN for a far exterior point) are dropped HERE, so the changes of basis below are plain FMAs.  The first
    // version tested every coefficient for zero inside the sums: 89k warp instructions per cell for 5.5k of FMAs, 3.5 ms at
    // cfg4 (ncu: issue-bound).
    double *mg = MG + (long long)cell * MOM4_MG;
    {
        // all of the thread's moments in flight at once: a load / store-zero loop ran one DRAM round trip per element
        // (the moments of 14,641 cells, 312 MB, do not stay in L2) -- 29 % of the kernel's stall samples
        constexpr int NL = (MOM4_NM + MOM4_NR + 255) / 256;
        double v[NL];
#pragma unroll
        for (int q = 0; q < NL; ++q) {
            const int k = tid + 256 * q;
            v[q] = (k < MOM4_NM + MOM4_NR && (!RHS_ONLY || k >= MOM4_NM)) ? __ldcg(mg + k) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < NL; ++q) {
            const int k = tid + 256 * q;
            if (k < MOM4_NM + MOM4_NR && (!RHS_ONLY || k >= MOM4_NM)) {
                if (!gp.fxpass) __stcg(mg + k, 0.0);      // (the scale-finding pass of the deterministic mode reads only)
                double val = v[q];
                if (ext) {
                    if (k < MOM4_NM) {
                        const int e1 = k % 7, e2 = (k / 7) % 7, e3 = (k / 49) % 7, e4 = k / 343;
                        if (((ext & 1) && e1 > 2) || ((ext & 2) && e2 > 2) || ((ext & 4) && e3 > 2) || ((ext & 8) && e4 > 2)) val = 0.0;
                    } else {
                        const int qq = k - MOM4_NM;
                        if (((ext & 1) && (qq & 3) > 1) || ((ext & 2) && ((qq >> 2) & 3) > 1) || ((ext & 4) && ((qq >> 4) & 3) > 1) ||
                            ((ext & 8) && (qq >> 6) > 1))
                            val = 0.0;
                    }
                }
                s_M[k] = val;
            }
        }
    }
    __syncthreads();
    // One change of basis: out[o][a][r] = sum_e C[a][e] in[o][e][r], a = 0..9 (pairs) -- a work item (o, r) loads its seven
    // inputs once and forms the ten outputs with warp-uniform coefficient loads.
    auto basis_g = [&](const double *C, const double *in, double *out, int no, int nr) {
        for (int it = tid; it < no * nr; it += blockDim.x) {
            const int o = it / nr, r = it - o * nr;
            double v[MOM_NE];
#pragma unroll
            for (int e = 0; e < MOM_NE; ++e) v[e] = in[(o * MOM_NE + e) * nr + r];
#pragma unroll
            for (int a = 0; a < 10; ++a) {
                double sum = 0.0;
#pragma unroll
                for (int e = 0; e < MOM_NE; ++e) sum = fma(C[a * MOM_NE + e], v[e], sum);
                out[(o * 10 + a) * nr + r] = sum;
            }
        }
    };
    // right-hand side: U1[(f4,f3,f2)][i1], U2[(f4,f3)][i2][i1], U3[f4][i3][i2][i1], g[i4][i3][i2][i1]
    {
        const int ro = tid >> 2, i1 = tid & 3;
        double sum = 0.0;
#pragma unroll
        for (int f = 0; f < MOM_NF; ++f) sum = fma(s_C[70 + i1 * MOM_NF + f], s_M[MOM4_NM + ro * MOM_NF + f], sum);
        s_U1[tid] = sum;
    }
    if (!RHS_ONLY) basis_g(s_C, s_M, s_T1, 343, 1);                      // T1[(e4,e3,e2)][a1]
    __syncthreads();
    {
        const int o = tid >> 4, i2 = (tid >> 2) & 3, i1 = tid & 3;   // o = (f4, f3)
        double sum = 0.0;
#pragma unroll
        for (int f = 0; f < MOM_NF; ++f) sum = fma(s_C[MOM_CW + 70 + i2 * MOM_NF + f], s_U1[(o * 4 + f) * 4 + i1], sum);
        s_U2[tid] = sum;
    }
    if (!RHS_ONLY) basis_g(s_C + MOM_CW, s_T1, s_T2, 49, 10);            // T2[(e4,e3)][a2][a1]
    __syncthreads();
    {
        const int f4 = tid >> 6, i3 = (tid >> 4) & 3, r = tid & 15;
        double sum = 0.0;
#pragma unroll
        for (int f = 0; f < MOM_NF; ++f) sum = fma(s_C[2 * MOM_CW + 70 + i3 * MOM_NF + f], s_U2[(f4 * 4 + f) * 16 + r], sum);
        s_U3[tid] = sum;
    }
    if (!RHS_ONLY) basis_g(s_C + 2 * MOM_CW, s_T2, s_T3, 7, 100);        // T3[e4][a3][a2 a1]
    __syncthreads();
    {
        const int i4 = tid >> 6, r = tid & 63;
        double sum = 0.0;
#pragma unroll
        for (int f = 0; f < MOM_NF; ++f) sum = fma(s_C[3 * MOM_CW + 70 + i4 * MOM_NF + f], s_U3[f * 64 + r], sum);
        if (sum != 0.0) {
            const long long node = (long long)(ws[0] + (r & 3)) + (long long)(ws[1] + ((r >> 2) & 3)) * gp.nodes[0] +
                                   (long long)(ws[2] + (r >> 4)) * gp.nodes[0] * gp.nodes[1] +
                                   (long long)(ws[3] + i4) * gp.nodes[0] * gp.nodes[1] * gp.nodes[2];
            spl_add_g(gp, g, node, sum);
        }
    }
    if (!RHS_ONLY) {
        // S[a4][a3][a2][a1]: a work item r = (a3, a2, a1) loads T3[0..6][r] and adds its ten entries
        const long long st3 = (long long)gp.nodes[0] * gp.nodes[1] * gp.nodes[2];
        for (int r = tid; r < 1000; r += blockDim.x) {
            double v[MOM_NE];
#pragma unroll
            for (int e = 0; e < MOM_NE; ++e) v[e] = s_T3[e * 1000 + r];
            const int a[3] = {r % 10, (r / 10) % 10, r / 100};
            long long node = 0, nstride = 1;
            int sten = 0, sstride = 1;
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                int i, j;
                spl_pair(a[d], i, j);
                node += (long long)(ws[d] + i) * nstride;
                sten += (j - i) * sstride;
                nstride *= gp.nodes[d];
                sstride *= 4;
            }
#pragma unroll
            for (int a4 = 0; a4 < 10; ++a4) {
                double sum = 0.0;
#pragma unroll
                for (int e = 0; e < MOM_NE; ++e) sum = fma(s_C[3 * MOM_CW + a4 * MOM_NE + e], v[e], sum);
                if (sum != 0.0) {
                    int i, j;
                    spl_pair(a4, i, j);
                    spl_add_S(gp, S, (node + (long long)(ws[3] + i) * st3) * gp.nsten + sten + (j - i) * 64, sum);
                }
            }
        }
    }
}
