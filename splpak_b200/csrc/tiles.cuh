// tiles.cuh -- FP64 tensor-core MMA and the cp.async staging of 64 x 64 band tiles into shared memory, shared by the
// band Cholesky solve (solve.cu) and the selected inverse (selinv.cu).
#pragma once
#include <stdint.h>

#define TILE_LD 68      // 64 + 4: (t4*68 + g) hits 16 distinct 8-byte banks per half-warp (conflict-free LDS.64)

__device__ __forceinline__ void spl_dmma_8x8x4(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}
__device__ __forceinline__ void spl_cp_async8(double *smem_dst, const double *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gsrc)
                 : "memory");
}
__device__ __forceinline__ void spl_cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void spl_cp_async16(double *smem_dst, const double *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gsrc)
                 : "memory");
}
// One 16-byte piece (two consecutive rows of one column) of an operand tile: cp.async when both rows are valid,
// otherwise an 8-byte cp.async of the valid row (if any) and zeros.  The band leading dimension is even
// (spl_band_lda) and tiles start at even rows, so every piece is 16-byte aligned on both sides.
__device__ __forceinline__ void spl_tile_piece(double *dst, const double *src, const int valid, const bool kok) {
    if (kok && valid >= 2) {
        spl_cp_async16(dst, src);
    } else if (kok && valid == 1) {
        // (asynchronous too: a blocking load here cost a full L2 round trip per column in every tile of an edge row
        // with an odd number of rows -- cfg3's half bandwidth is 1803 -- and those tiles' CTAs were the last at every
        // barrier)
        spl_cp_async8(dst, src);
        dst[1] = 0.0;
    } else {
        *reinterpret_cast<double2 *>(dst) = make_double2(0.0, 0.0);
    }
}
// 64 rows x 64 columns at src (column-major, leading dimension lda; `rows` of the rows and `nb` of the columns
// exist, the rest reads as zero) -> shared memory s[column * TILE_LD + row], with PANEL_THREADS threads: 8 pieces per
// thread, a warp covers the 64 rows of one column (512 contiguous bytes).  The caller commits the cp.async group.
__device__ __forceinline__ void spl_tile_load16(double *s, const double *src, const long long lda, const int rows,
                                                const int nb, const int t) {
    const int r = 2 * (t & 31);
    int k = t >> 5;
    const double *gp = src + r + (long long)k * lda;
    double *dp = s + k * TILE_LD + r;
    const int valid = rows - r;
    const long long gstep = 8 * lda;
#pragma unroll
    for (int q = 0; q < 8; ++q, k += 8) {
        spl_tile_piece(dp, gp, valid, k < nb);
        gp += gstep;
        dp += 8 * TILE_LD;
    }
}

