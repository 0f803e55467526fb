// Consensus measures of factorize() on the device (R/factorize.R:51-78,214-216,226): dispersion
// and the cophenetic correlation under average linkage, from the labels of nrun restarts, without
// the m(m-1)/2 connectivity vector.  Included only by vbnmf.cu (vbnmf_consensus documents the
// definition; oracle/oracle_consensus.py restates it).
//
//   moments:  the K x K contingency table of every run pair t <= u (pair_contingency_kernel);
//             S1 and S2 are sums of C(M, 2) over them, taken on the host in int64.
//   groups:   cells sorted stably by L[nrun-1], ..., L[0] (cub radix sort), boundary flags, a scan
//             for group ids (group_* kernels): groups in the lexicographic order of their tuples.
//   IP fill:  IP_ab = n_a n_b #{t: T_at = T_bt} for a < b, packed upper triangle (ip_fill_kernel).
//   merges:   the greedy agglomeration with a per-row cache of the best (q, b) over active b > a,
//             one persistent cooperative kernel with grid-wide barriers (merge_loop_kernel).
#pragma once
#include <cooperative_groups.h>

#include "kernels_common.cuh"

namespace vb {

// K x K uint32 counters of one run pair in shared memory: K <= 240 fits the 227 KB of a CTA.
constexpr int kConsensusMaxLabels = 240;
constexpr int kMergeBlock = 512;

VB_HD int64_t tri_index(int64_t G, int64_t a, int64_t b) {  // a < b
    return a * (2 * G - a - 1) / 2 + (b - a - 1);
}

// blockIdx.y = run pair p (t <= u, row-major over the upper triangle incl. the diagonal);
// tab[p][c][c'] += cells with L[t] = c and L[u] = c'.
__global__ void __launch_bounds__(kBlock)
pair_contingency_kernel(int64_t m, int nrun, int K, const int32_t *__restrict__ lab,
                        const int32_t *__restrict__ pair_t, const int32_t *__restrict__ pair_u,
                        unsigned long long *__restrict__ tab) {
    extern __shared__ unsigned int cons_hist[];
    const int KK = K * K;
    const int p = blockIdx.y;
    const int32_t *lt = lab + (int64_t)pair_t[p] * m, *lu = lab + (int64_t)pair_u[p] * m;
    for (int i = threadIdx.x; i < KK; i += kBlock) cons_hist[i] = 0u;
    __syncthreads();
    for (int64_t j = (int64_t)blockIdx.x * kBlock + threadIdx.x; j < m;
         j += (int64_t)gridDim.x * kBlock)
        atomicAdd(&cons_hist[lt[j] * K + lu[j]], 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < KK; i += kBlock)
        if (cons_hist[i]) atomicAdd(&tab[(int64_t)p * KK + i], (unsigned long long)cons_hist[i]);
}

__global__ void __launch_bounds__(kBlock)
group_gather_key_kernel(int64_t m, const int32_t *__restrict__ lab_t,
                        const int32_t *__restrict__ perm, uint32_t *__restrict__ key) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i < m) key[i] = (uint32_t)lab_t[perm[i]];
}

// flag[i] = 1 when sorted cell i starts a new group (its tuple differs from cell i - 1's)
__global__ void __launch_bounds__(kBlock)
group_flag_kernel(int64_t m, int nrun, const int32_t *__restrict__ lab,
                  const int32_t *__restrict__ perm, int32_t *__restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= m) return;
    int f = i == 0;
    if (!f) {
        const int64_t x = perm[i], y = perm[i - 1];
        for (int t = 0; t < nrun && !f; t++) f = lab[t * m + x] != lab[t * m + y];
    }
    flag[i] = f;
}

// gid = inclusive scan of flag (1-based group of sorted cell i): start[g] = first sorted cell of
// group g, and its tuple, 4 labels per word (byte t % 4 of word t / 4, unused bytes 0)
__global__ void __launch_bounds__(kBlock)
group_start_kernel(int64_t m, int nrun, int W, const int32_t *__restrict__ lab,
                   const int32_t *__restrict__ perm, const int32_t *__restrict__ flag,
                   const int32_t *__restrict__ gid, int64_t *__restrict__ start,
                   uint32_t *__restrict__ tup) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= m || !flag[i]) return;
    const int64_t g = gid[i] - 1, x = perm[i];
    start[g] = i;
    for (int w = 0; w < W; w++) {
        uint32_t v = 0;
        for (int k = 0; k < 4 && 4 * w + k < nrun; k++)
            v |= (uint32_t)lab[(int64_t)(4 * w + k) * m + x] << (8 * k);
        tup[g * W + w] = v;
    }
}

__global__ void __launch_bounds__(kBlock)
group_size_kernel(int64_t G, int64_t m, const int64_t *__restrict__ start, int64_t *__restrict__ size) {
    const int64_t g = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (g < G) size[g] = (g + 1 < G ? start[g + 1] : m) - start[g];
}

// IP_ab for a < b: one thread per pair, a 64-wide run of b per row a so the stores coalesce.
// Tuples are compared 4 labels at a time; the zero padding of the last word always agrees and is
// subtracted (pad = 4 W - nrun).
__global__ void __launch_bounds__(kBlock)
ip_fill_kernel(int64_t G, int W, int pad, const uint32_t *__restrict__ tup,
               const int64_t *__restrict__ size, int64_t *__restrict__ ip) {
    const int64_t a0 = (int64_t)blockIdx.y * 4, b = (int64_t)blockIdx.x * 64 + (threadIdx.x & 63);
    const int64_t a = a0 + (threadIdx.x >> 6);
    if (a >= G || b >= G || b <= a) return;
    int agree = -pad;
    for (int w = 0; w < W; w++)
        agree += __popc(__vcmpeq4(__ldg(tup + a * W + w), __ldg(tup + b * W + w))) >> 3;
    ip[tri_index(G, a, b)] = size[a] * size[b] * (int64_t)agree;
}

// (q, j) beats (q2, j2): larger q, then smaller j
__device__ __forceinline__ bool cons_better(double q, int64_t j, double q2, int64_t j2) {
    return q > q2 || (q == q2 && j < j2);
}

// block-wide argmax of (q, j) over the threads' candidates; every thread gets the result
template <int NT>
__device__ void block_argmax(double &q, int64_t &j, double *sq, int64_t *sj) {
    for (int o = 16; o > 0; o >>= 1) {
        const double q2 = __shfl_xor_sync(kFull, q, o);
        const int64_t j2 = __shfl_xor_sync(kFull, j, o);
        if (cons_better(q2, j2, q, j)) { q = q2; j = j2; }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();  // sq / sj may still be read by a previous call
    if (lane == 0) { sq[warp] = q; sj[warp] = j; }
    __syncthreads();
    q = sq[0]; j = sj[0];
    for (int w = 1; w < NT / 32; w++)
        if (cons_better(sq[w], sj[w], q, j)) { q = sq[w]; j = sj[w]; }
}

// Scan of row k by one block: the best active j > k.  Retired groups have size 0; during a merge
// step (a, b) group a already counts na + nb members and b is retired (ov_a >= 0), because the
// sizes are only written after the rescans.  (No __restrict__ on ip and size: inside the merge loop
// other blocks write them, and the non-coherent read-only path would miss that.)
template <int NT>
__device__ void scan_row(int64_t G, int nrun, int64_t k, const int64_t *ip,
                         const int64_t *size, int64_t ov_a, int64_t ov_na, int64_t ov_b,
                         double *bq, int32_t *bb, double *sq, int64_t *sj) {
    const int64_t nk = k == ov_a ? ov_na : size[k];
    const int64_t base = tri_index(G, k, k + 1) - (k + 1);
    double q = -1.0;
    int64_t j = INT64_MAX;
    for (int64_t c = k + 1 + threadIdx.x; c < G; c += NT) {
        const int64_t nc = c == ov_a ? ov_na : (c == ov_b ? 0 : size[c]);
        if (nc == 0) continue;
        const double v = (double)ip[base + c] / (double)((int64_t)nrun * nk * nc);
        if (cons_better(v, c, q, j)) { q = v; j = c; }
    }
    block_argmax<NT>(q, j, sq, sj);
    if (threadIdx.x == 0) { bq[k] = q; bb[k] = j == INT64_MAX ? -1 : (int32_t)j; }
}

// initial row cache: one block per row
__global__ void __launch_bounds__(kMergeBlock)
row_best_kernel(int64_t G, int nrun, const int64_t *__restrict__ ip, const int64_t *__restrict__ size,
                double *__restrict__ bq, int32_t *__restrict__ bb) {
    __shared__ double sq[kMergeBlock / 32];
    __shared__ int64_t sj[kMergeBlock / 32];
    for (int64_t k = blockIdx.x; k < G; k += gridDim.x)
        scan_row<kMergeBlock>(G, nrun, k, ip, size, -1, 0, -1, bq, bb, sq, sj);
}

struct MergeArgs {
    int64_t G;
    int nrun;
    int64_t *ip;        // packed upper triangle, updated in place
    int64_t *size;      // members per group, 0 once retired
    double *bq;         // row cache: best q over active b > a (-1: none)
    int32_t *bb;        //            and its b (-1: none)
    int64_t *merges;    // (G - 1) x 5: a, b, IP_ab, N_a, N_b
    int32_t *resc;      // rows to rescan in the current step (G)
    unsigned *nresc;    // [0] rows in resc
    double *part_q;     // per-block argmax partials (gridDim.x)
    int64_t *part_a;
    unsigned long long *rescans;  // total rows rescanned
};

// The G - 1 merge steps.  Each step, between grid-wide barriers:
//   A  argmax of the cached (q, a) over active rows, per block -> partials;
//   B  every block reduces the partials to the same (a, b); IP_ak += IP_bk for every active k,
//      and the caches of rows k < a are updated (adopt a, or rescan when their best was a or b and
//      q(k, a) fell below it); rows a < k < b whose best was b, and row a, are queued for a rescan;
//   C  the queued rows are rescanned (a block per row); the sizes of a and b are written.
__global__ void __launch_bounds__(kMergeBlock)
merge_loop_kernel(MergeArgs A) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double sq[kMergeBlock / 32];
    __shared__ int64_t sj[kMergeBlock / 32];
    const int64_t G = A.G;
    const int64_t tid = (int64_t)blockIdx.x * kMergeBlock + threadIdx.x;
    const int64_t nthreads = (int64_t)gridDim.x * kMergeBlock;
    for (int64_t s = 0; s + 1 < G; s++) {
        // ---- A
        {
            double q = -1.0;
            int64_t a = INT64_MAX;
            for (int64_t k = tid; k < G; k += nthreads)
                if (A.bb[k] >= 0 && cons_better(A.bq[k], k, q, a)) { q = A.bq[k]; a = k; }
            block_argmax<kMergeBlock>(q, a, sq, sj);
            if (threadIdx.x == 0) { A.part_q[blockIdx.x] = q; A.part_a[blockIdx.x] = a; }
            if (tid == 0) A.nresc[0] = 0u;
        }
        grid.sync();
        // ---- B
        double q = -1.0;
        int64_t a = INT64_MAX;
        for (int64_t i = threadIdx.x; i < gridDim.x; i += kMergeBlock)
            if (cons_better(A.part_q[i], A.part_a[i], q, a)) { q = A.part_q[i]; a = A.part_a[i]; }
        block_argmax<kMergeBlock>(q, a, sq, sj);
        const int64_t b = A.bb[a];
        const int64_t na = A.size[a], nb = A.size[b], nab = na + nb;
        if (tid == 0) {
            int64_t *rec = A.merges + s * 5;
            rec[0] = a; rec[1] = b; rec[2] = A.ip[tri_index(G, a, b)]; rec[3] = na; rec[4] = nb;
            A.resc[atomicAdd(A.nresc, 1u)] = (int32_t)a;
        }
        for (int64_t k = tid; k < G; k += nthreads) {
            if (k == a || k == b) continue;
            const int64_t nk = A.size[k];
            if (nk == 0) continue;
            const int64_t ia = k < a ? tri_index(G, k, a) : tri_index(G, a, k);
            const int64_t ib = k < b ? tri_index(G, k, b) : tri_index(G, b, k);
            const int64_t v = A.ip[ia] + A.ip[ib];
            A.ip[ia] = v;
            if (k < a) {
                const double qn = (double)v / (double)((int64_t)A.nrun * nk * nab);
                const int32_t c = A.bb[k];
                const double qc = A.bq[k];
                if (c == a || c == b) {
                    if (qn >= qc) { A.bq[k] = qn; A.bb[k] = (int32_t)a; }
                    else A.resc[atomicAdd(A.nresc, 1u)] = (int32_t)k;
                } else if (cons_better(qn, a, qc, c)) {
                    A.bq[k] = qn; A.bb[k] = (int32_t)a;
                }
            } else if (k < b && A.bb[k] == b) {
                A.resc[atomicAdd(A.nresc, 1u)] = (int32_t)k;
            }
        }
        grid.sync();
        // ---- C
        const unsigned nr = A.nresc[0];
        for (unsigned i = blockIdx.x; i < nr; i += gridDim.x)
            scan_row<kMergeBlock>(G, A.nrun, A.resc[i], A.ip, A.size, a, nab, b, A.bq, A.bb, sq, sj);
        if (tid == 0) {
            A.size[a] = nab; A.size[b] = 0; A.bb[b] = -1;
            *A.rescans += nr;
        }
        grid.sync();
    }
}

}  // namespace vb
