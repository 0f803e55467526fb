// Cell and gene QC on the device (filter_cells / filter_genes / calc_vmr / normalize_count,
// R/utils.R:78-95,134-218,318-327): a statistics pass over the nonzeros and a subset/scale pass
// that builds the CSC of a new handle from the arrays of an existing one.  Both are bandwidth-bound
// passes over data the GPU already holds; the matrix never crosses the bus.  Included only by
// vbnmf.cu.
#pragma once
#include "kernels_common.cuh"

namespace vb {

// Per cell: cell_sum[j] = sum_i x_ij, a warp per column with a shuffle reduction (no atomics, the
// summation order is fixed).  Per gene: gene_sum[i] = sum_j x_ij and gene_sumsq[i] = sum_j x_ij^2
// with fp64 atomics (zeroed by the caller).  For integer counts every partial sum is an integer
// below 2^53, so the result is exact and does not depend on the order the atomics land in.
// One pass: colptr, rowidx and the values are each read once.
template <typename VT>
__global__ void __launch_bounds__(kBlock)
qc_stats_kernel(int64_t m, const int64_t *__restrict__ colptr, const int32_t *__restrict__ rowidx,
                const VT *__restrict__ val, double *__restrict__ cell_sum,
                double *__restrict__ gene_sum, double *__restrict__ gene_sumsq) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * kBlock + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * kBlock) >> 5;
    for (int64_t j = warp; j < m; j += nwarps) {
        const int64_t beg = colptr[j], end = colptr[j + 1];
        double s = 0.0;
        for (int64_t t = beg + lane; t < end; t += 32) {
            const double x = (double)val[t];
            if (x == 0.0) continue;  // explicit zeros add nothing
            const int32_t i = rowidx[t];
            s += x;
            atomicAdd(gene_sum + i, x);
            atomicAdd(gene_sumsq + i, x * x);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
        if (lane == 0) cell_sum[j] = s;
    }
}

// mask (bytes) -> 0/1 in int32, the input of the exclusive scan that renumbers the kept rows
__global__ void __launch_bounds__(kBlock)
qc_mask_kernel(int64_t count, const uint8_t *__restrict__ mask, int32_t *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (t < count) out[t] = mask[t] != 0;
}

// after the scan: map[i] = new index of a kept row, -1 for a dropped one
__global__ void __launch_bounds__(kBlock)
qc_rowmap_kernel(int64_t count, const uint8_t *__restrict__ mask, int32_t *__restrict__ map) {
    const int64_t t = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (t < count && !mask[t]) map[t] = -1;
}

// a warp per kept column k (source column cols[k]): cnt[k] = entries in kept rows
__global__ void __launch_bounds__(kBlock)
qc_subset_count_kernel(int64_t mk, const int32_t *__restrict__ cols,
                       const int64_t *__restrict__ colptr, const int32_t *__restrict__ rowidx,
                       const int32_t *__restrict__ rowmap, int64_t *__restrict__ cnt) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * kBlock + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * kBlock) >> 5;
    for (int64_t k = warp; k < mk; k += nwarps) {
        const int32_t j = cols[k];
        const int64_t beg = colptr[j], end = colptr[j + 1];
        unsigned c = 0;
        for (int64_t t = beg + lane; t < end; t += 32) c += rowmap[rowidx[t]] >= 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(kFull, c, o);
        if (lane == 0) cnt[k] = c;
    }
}

// a warp per kept column k: the entries of kept rows, in their order, to out_row / out_val from
// newptr[k] on (stored zeros included).  Value = x * col_scale[j] in fp64 (no multiply without a
// scale).  With OT = float, *inexact is set when a value is not exactly representable in fp32
// (NaN included), the rule vbnmf_create applies to choose the value format.
template <typename VT, typename OT>
__global__ void __launch_bounds__(kBlock)
qc_subset_compact_kernel(int64_t mk, const int32_t *__restrict__ cols,
                         const int64_t *__restrict__ colptr, const int32_t *__restrict__ rowidx,
                         const VT *__restrict__ val, const int32_t *__restrict__ rowmap,
                         const double *__restrict__ col_scale, const int64_t *__restrict__ newptr,
                         int32_t *__restrict__ out_row, OT *__restrict__ out_val,
                         unsigned *__restrict__ inexact) {
    const int lane = threadIdx.x & 31;
    const unsigned below = (1u << lane) - 1u;
    const int64_t warp = ((int64_t)blockIdx.x * kBlock + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * kBlock) >> 5;
    bool bad = false;
    for (int64_t k = warp; k < mk; k += nwarps) {
        const int32_t j = cols[k];
        const int64_t beg = colptr[j], end = colptr[j + 1];
        const double sc = col_scale ? col_scale[j] : 1.0;
        int64_t pos = newptr[k];
        for (int64_t base = beg; base < end; base += 32) {
            const int64_t t = base + lane;
            const int32_t ni = t < end ? rowmap[rowidx[t]] : -1;
            const unsigned keep = __ballot_sync(kFull, ni >= 0);
            if (ni >= 0) {
                const int64_t o = pos + __popc(keep & below);
                double v = (double)val[t];
                if (col_scale) v *= sc;
                const OT ov = (OT)v;
                if constexpr (sizeof(OT) == 4) bad |= !((double)ov == v);
                out_row[o] = ni;
                out_val[o] = ov;
            }
            pos += __popc(keep);
        }
    }
    if (bad) atomicOr(inexact, 1u);
}

}  // namespace vb
