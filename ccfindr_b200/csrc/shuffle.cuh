// Column shuffle on the device: the null matrix of factorize(randomize = TRUE), each column of the
// counts permuted over the genes (R/factorize.R:172-173), built from the arrays of an existing
// handle.  Only the rows of the stored entries are drawn anew: colptr and every column's multiset
// of values are kept, so the matrix never has to be densified or cross the bus.  Included only by
// vbnmf.cu.
//
// The draw (restated in ccfindr_b200/synth.py:shuffle_columns_reference).  Column j with k stored
// entries (stored zeros included) out of n rows:
//   u_t = t-th next() of VbStream(seed, 3 << 62 | j), t = 0, 1, ... (tags 0, 1: init_random,
//         2: svd_init.cuh), i.e. u_t = mix(s0 + (t + 1) 0x9E3779B97F4A7C15);
//   row of draw t = umulhi(u_t, n) = (u_t n) >> 64;
//   s_0 ... s_{k-1} = the first k DISTINCT rows in draw order;
//   the t-th stored entry of the source column (ascending source row) goes to row s_t, and the
//   column is stored sorted by row.
// The first k distinct values of i.i.d. uniform draws are a uniformly random ordered k-tuple of
// distinct rows, so this is distributed as a uniform permutation of the dense column (up to the
// n / 2^64 bias of umulhi).
#pragma once
#include "kernels_common.cuh"

namespace vb {

// One warp per column holds an n-bit row bitmap and a per-32-row prefix count (8 bytes per 32
// rows) in shared memory.  One warp's tables must fit the 227 KB a CTA can address on sm_100, so
// n <= 232448 / 8 * 32 = 929,792 rows.
constexpr int kShuffleSmemMax = 232448;
constexpr int64_t kShuffleMaxRows = (int64_t)kShuffleSmemMax / 8 * 32;
constexpr int kShuffleWarps = 8;  // warps per CTA when the tables of 8 fit

VB_HD int64_t shuffle_words(int64_t n) { return (n + 31) / 32; }

// Grid-stride over columns, a warp per column, dynamic shared memory = warps * 2 * words(n) * 4.
//   select: lanes take 32 consecutive draws; duplicates inside the batch resolve to the lowest lane
//           (__match_any_sync), rows already in the bitmap are rejected, an accepted lane gets its
//           ordinal t from a ballot (ordinals >= k are dropped before any bit is set) and writes
//           s_t to out_row[beg + t];
//   rank:   pre[w] = set bits in words < w; rank(s) = pre[s / 32] + set bits below s in its word;
//           out_val[beg + rank(s_t)] = val[beg + t];
//   rows:   the set bits in ascending order over out_row (overwriting the s_t), bitmap cleared.
// *bad is set when a column holds more entries than there are rows (a CSC with repeated entries):
// k distinct rows cannot be drawn.
template <typename VT>
__global__ void __launch_bounds__(kBlock)
shuffle_columns_kernel(int64_t n, int64_t m, unsigned long long seed,
                       const int64_t *__restrict__ colptr, const VT *__restrict__ val,
                       int32_t *out_row, VT *__restrict__ out_val, unsigned *__restrict__ bad) {
    extern __shared__ unsigned shuffle_smem[];
    const int lane = threadIdx.x & 31;
    const unsigned below = (1u << lane) - 1u;
    const int64_t nw = shuffle_words(n);
    unsigned *bits = shuffle_smem + (size_t)(threadIdx.x >> 5) * 2 * nw;
    unsigned *pre = bits + nw;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = lane; w < nw; w += 32) bits[w] = 0u;
    __syncwarp();
    for (int64_t j = warp; j < m; j += nwarps) {
        const int64_t beg = colptr[j], k = colptr[j + 1] - beg;
        if (k == 0) continue;
        if (k > n) {
            if (lane == 0) atomicOr(bad, 1u);
            continue;
        }
        const unsigned long long s0 = VbStream(seed, (3ull << 62) | (unsigned long long)j).s;
        int64_t got = 0;
        for (unsigned long long t0 = 1; got < k; t0 += 32) {
            const unsigned long long u = vb_mix64(s0 + (t0 + lane) * 0x9E3779B97F4A7C15ull);
            const unsigned row = (unsigned)__umul64hi(u, (unsigned long long)n);
            const unsigned same = __match_any_sync(kFull, row);
            const bool fresh = (same & below) == 0u && !((bits[row >> 5] >> (row & 31)) & 1u);
            const unsigned acc = __ballot_sync(kFull, fresh);
            const int64_t t = got + __popc(acc & below);
            if (fresh && t < k) {
                atomicOr(bits + (row >> 5), 1u << (row & 31));
                out_row[beg + t] = (int32_t)row;
            }
            got = min(got + (int64_t)__popc(acc), k);
            __syncwarp();
        }
        unsigned carry = 0;
        for (int64_t w0 = 0; w0 < nw; w0 += 32) {
            const int64_t w = w0 + lane;
            const unsigned c = w < nw ? __popc(bits[w]) : 0u;
            unsigned x = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned y = __shfl_up_sync(kFull, x, o);
                if (lane >= o) x += y;
            }
            if (w < nw) pre[w] = carry + x - c;
            carry += __shfl_sync(kFull, x, 31);
        }
        __syncwarp();
        for (int64_t t = lane; t < k; t += 32) {
            const unsigned s = (unsigned)out_row[beg + t];
            const unsigned r = pre[s >> 5] + __popc(bits[s >> 5] & ((1u << (s & 31)) - 1u));
            out_val[beg + r] = val[beg + t];
        }
        __syncwarp();  // every s_t is read before the rows overwrite them
        for (int64_t w = lane; w < nw; w += 32) {
            unsigned b = bits[w];
            if (!b) continue;
            bits[w] = 0u;
            int32_t *o = out_row + beg + pre[w];
            for (; b; b &= b - 1u) *o++ = (int32_t)(w * 32 + __ffs(b) - 1);
        }
        __syncwarp();
    }
}

}  // namespace vb
