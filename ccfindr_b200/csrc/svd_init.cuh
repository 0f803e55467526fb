// vb_init(initializer = 'svd2') on the device (R/bayesian.R:150-159):
//   s <- irlba(mat, rank);  w <- abs(s$u);  h <- abs(diag(s$d) %*% t(s$v));
//   scale <- bh / mean(h);  h <- h * scale;  w <- w / scale
// and vb_init(initializer = 'svd') (R/bayesian.R:116-149), the NNDSVD of Boutsidis & Gallopoulos
// (2008) on the same truncated SVD, every pair (u_k, v_k), k >= 1, oriented first (vbnmf.h).
// The truncated SVD is a randomized range finder on the CSC matrix already resident on the GPU
// (Halko, Martinsson & Tropp 2011, alg. 4.4 + 5.1): Y = X Omega with k = rank + oversampling
// Gaussian columns, a few power iterations Y <- X (X^T Q) with Cholesky-QR re-orthonormalisation
// in between, B^T = X^T Q, and the k x k eigenproblem of B B^T on the host (Jacobi).  Only k x k
// matrices ever cross the bus.  With the cells sharded over GPUs the sums over cells (Y, the
// Gram matrices, mean(h)) are all-reduced.
// The accumulation Y += x_ij z_j uses fp64 atomics: the result is reproducible to rounding (the
// order of the additions is not fixed), unlike the bitwise-reproducible update kernels.
// Included only by vbnmf.cu.
#pragma once
#include "kernels_common.cuh"

namespace vb {

constexpr int kSvdMaxK = 96;  // rank + oversampling

// out[row * k + c] ~ N(0, 1), keyed by (seed, global row, c)
__global__ void __launch_bounds__(kBlock)
gauss_fill_kernel(int64_t rows, int k, unsigned long long seed, int64_t row_offset,
                  double *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (t >= rows * k) return;
    const int64_t row = t / k;
    const int c = (int)(t - row * k);
    VbStream st(seed, (2ull << 62) | ((unsigned long long)(row + row_offset) << 7) |
                          (unsigned long long)c);
    out[t] = st.normal();
}

// out (m x k) = X^T Q, Q n x k row-major: one warp per column of X, lanes over the k columns
template <typename VT>
__global__ void __launch_bounds__(kBlock)
spmm_xt_kernel(int64_t m, int k, const int64_t *__restrict__ colptr,
               const int32_t *__restrict__ rowidx, const VT *__restrict__ val,
               const double *__restrict__ Q, double *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * kBlock + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * kBlock) >> 5;
    for (int64_t j = warp; j < m; j += nwarps) {
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;
        const int64_t beg = colptr[j], end = colptr[j + 1];
        for (int64_t t = beg; t < end; t++) {
            const double x = (double)val[t];
            const double *q = Q + (int64_t)rowidx[t] * k;
            if (lane < k) a0 = fma(x, q[lane], a0);
            if (lane + 32 < k) a1 = fma(x, q[lane + 32], a1);
            if (lane + 64 < k) a2 = fma(x, q[lane + 64], a2);
        }
        double *o = out + j * k;
        if (lane < k) o[lane] = a0;
        if (lane + 32 < k) o[lane + 32] = a1;
        if (lane + 64 < k) o[lane + 64] = a2;
    }
}

// Y (n x k, zeroed before) += X Z, Z m x k row-major: one warp per column, fp64 atomics on Y
template <typename VT>
__global__ void __launch_bounds__(kBlock)
spmm_x_kernel(int64_t m, int k, const int64_t *__restrict__ colptr,
              const int32_t *__restrict__ rowidx, const VT *__restrict__ val,
              const double *__restrict__ Z, double *__restrict__ Y) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * kBlock + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * kBlock) >> 5;
    for (int64_t j = warp; j < m; j += nwarps) {
        const double *z = Z + j * k;
        const double z0 = lane < k ? z[lane] : 0.0, z1 = lane + 32 < k ? z[lane + 32] : 0.0,
                     z2 = lane + 64 < k ? z[lane + 64] : 0.0;
        const int64_t beg = colptr[j], end = colptr[j + 1];
        for (int64_t t = beg; t < end; t++) {
            const double x = (double)val[t];
            double *y = Y + (int64_t)rowidx[t] * k;
            if (lane < k) atomicAdd(y + lane, x * z0);
            if (lane + 32 < k) atomicAdd(y + lane + 32, x * z1);
            if (lane + 64 < k) atomicAdd(y + lane + 64, x * z2);
        }
    }
}

// part[b][a * k + c] = sum over the rows of CTA b of A[row][a] A[row][c]  (A rows x k)
constexpr int kGramRows = 32;
__global__ void __launch_bounds__(kBlock)
gram_part_kernel(int64_t rows, int k, const double *__restrict__ A, double *__restrict__ part) {
    extern __shared__ double gtile[];  // kGramRows x k
    const int kk = k * k;
    double acc[(kSvdMaxK * kSvdMaxK + kBlock - 1) / kBlock];
#pragma unroll
    for (int q = 0; q < (kSvdMaxK * kSvdMaxK + kBlock - 1) / kBlock; q++) acc[q] = 0.0;
    for (int64_t r0 = (int64_t)blockIdx.x * kGramRows; r0 < rows; r0 += (int64_t)gridDim.x * kGramRows) {
        const int nr = (int)min((int64_t)kGramRows, rows - r0);
        __syncthreads();
        for (int t = threadIdx.x; t < nr * k; t += kBlock) gtile[t] = A[r0 * k + t];
        __syncthreads();
        int q = 0;
        for (int p = threadIdx.x; p < kk; p += kBlock, q++) {
            const int a = p / k, c = p - a * k;
            double s = acc[q];
            for (int r = 0; r < nr; r++) s = fma(gtile[r * k + a], gtile[r * k + c], s);
            acc[q] = s;
        }
    }
    int q = 0;
    for (int p = threadIdx.x; p < kk; p += kBlock, q++) part[(size_t)blockIdx.x * kk + p] = acc[q];
}
// G[p] = sum_b part[b][p] in CTA order
__global__ void __launch_bounds__(kBlock)
gram_sum_kernel(int nblocks, int kk, const double *__restrict__ part, double *__restrict__ G) {
    const int p = blockIdx.x * kBlock + threadIdx.x;
    if (p >= kk) return;
    double s = 0.0;
    for (int b = 0; b < nblocks; b++) s += part[(size_t)b * kk + p];
    G[p] = s;
}

// out (rows x kout) = A (rows x k) M (k x kout, row-major, in global memory)
__global__ void __launch_bounds__(kBlock)
right_mult_kernel(int64_t rows, int k, int kout, const double *__restrict__ A,
                  const double *__restrict__ M, double *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (t >= rows * kout) return;
    const int64_t row = t / kout;
    const int c = (int)(t - row * kout);
    double s = 0.0;
    for (int a = 0; a < k; a++) s = fma(A[row * k + a], M[a * kout + c], s);
    out[t] = s;
}

// sum of |A| over all entries (rows x r), per-CTA partials then last-block reduction
__global__ void __launch_bounds__(kBlock)
abs_sum_kernel(int64_t count, const double *__restrict__ A, double *__restrict__ part,
               double *__restrict__ out, unsigned *counter) {
    __shared__ double sm[kWarpsPerBlock];
    double s = 0.0;
    for (int64_t t = (int64_t)blockIdx.x * kBlock + threadIdx.x; t < count;
         t += (int64_t)gridDim.x * kBlock)
        s += fabs(A[t]);
    s = block_sum(s, sm);
    if (threadIdx.x == 0) part[blockIdx.x] = s;
    last_block_reduce(part, 1, out, counter, sm);
}

// panel[dev[row]][c] = |A[row][c]| * f for c < r, into the l panel (layout tsplit) and its
// row-major mirror (alw / alh hold ew / eh = w / h before the first update, R/bayesian.R:170)
__global__ void __launch_bounds__(kBlock)
svd_store_kernel(int64_t rows, int r, int rs, const int32_t *__restrict__ dev,
                 const double *__restrict__ A, double f, double *__restrict__ panel,
                 double *__restrict__ mirror, int tsplit) {
    const int64_t t = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (t >= rows * r) return;
    const int64_t row = t / r;
    const int c = (int)(t - row * r);
    const double v = fabs(A[t]) * f;
    const int64_t d = dev[row];
    panel[panel_ofs(d, c, rs, tsplit)] = v;
    mirror[d * rs + c] = v;
}

// part[b][2c] / part[b][2c + 1] = sum over the rows of CTA b of A[row][c]^2 where A[row][c] > 0 /
// where A[row][c] < 0 (A rows x r, r <= kBlock); CTA b takes rows b*per .. b*per + per - 1, then
// steps by gridDim.x*per; the per rows are added in order: the sums do not depend on timing
__global__ void __launch_bounds__(kBlock)
signed_sq_part_kernel(int64_t rows, int r, const double *__restrict__ A, double *__restrict__ part) {
    __shared__ double sp[kBlock], sn[kBlock];
    const int per = kBlock / r, lr = threadIdx.x / r, c = threadIdx.x - lr * r;
    double p = 0.0, q = 0.0;
    if (lr < per)
        for (int64_t row = (int64_t)blockIdx.x * per + lr; row < rows; row += (int64_t)gridDim.x * per) {
            const double a = A[row * r + c];
            if (a > 0.0) p = fma(a, a, p);
            else q = fma(a, a, q);
        }
    sp[threadIdx.x] = p;
    sn[threadIdx.x] = q;
    __syncthreads();
    if (threadIdx.x < r) {
        for (int t = 1; t < per; t++) {
            p += sp[t * r + threadIdx.x];
            q += sn[t * r + threadIdx.x];
        }
        part[(size_t)blockIdx.x * 2 * r + 2 * threadIdx.x] = p;
        part[(size_t)blockIdx.x * 2 * r + 2 * threadIdx.x + 1] = q;
    }
}

// panel[dev[row]][c] = f[c] * max(s[c] * A[row][c], 0) for 1 <= c < r and f[0] * s[0] * A[row][0],
// into the l panel and its mirror as svd_store_kernel: the 'svd' factors (f, s: r values each)
__global__ void __launch_bounds__(kBlock)
svd_pos_store_kernel(int64_t rows, int r, int rs, const int32_t *__restrict__ dev,
                     const double *__restrict__ A, const double *__restrict__ f,
                     const double *__restrict__ s, double *__restrict__ panel,
                     double *__restrict__ mirror, int tsplit) {
    const int64_t t = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (t >= rows * r) return;
    const int64_t row = t / r;
    const int c = (int)(t - row * r);
    const double a = s[c] * A[t];
    const double v = f[c] * (c == 0 ? a : fmax(a, 0.0));
    const int64_t d = dev[row];
    panel[panel_ofs(d, c, rs, tsplit)] = v;
    mirror[d * rs + c] = v;
}

}  // namespace vb

// ---- k x k host linear algebra (k <= 96) ---------------------------------------------------------
namespace svdhost {

// upper-triangular R with G = R^T R (row-major k x k); false when G is not positive definite
inline bool cholesky_upper(int k, const std::vector<double> &G, std::vector<double> &R) {
    R.assign((size_t)k * k, 0.0);
    for (int j = 0; j < k; j++) {
        double d = G[(size_t)j * k + j];
        for (int p = 0; p < j; p++) d -= R[(size_t)p * k + j] * R[(size_t)p * k + j];
        if (!(d > 0.0)) return false;
        const double rjj = std::sqrt(d);
        R[(size_t)j * k + j] = rjj;
        for (int c = j + 1; c < k; c++) {
            double s = G[(size_t)j * k + c];
            for (int p = 0; p < j; p++) s -= R[(size_t)p * k + j] * R[(size_t)p * k + c];
            R[(size_t)j * k + c] = s / rjj;
        }
    }
    return true;
}

// inverse of an upper-triangular matrix
inline void invert_upper(int k, const std::vector<double> &R, std::vector<double> &Ri) {
    Ri.assign((size_t)k * k, 0.0);
    for (int j = 0; j < k; j++) {
        Ri[(size_t)j * k + j] = 1.0 / R[(size_t)j * k + j];
        for (int i = j - 1; i >= 0; i--) {
            double s = 0.0;
            for (int p = i + 1; p <= j; p++) s += R[(size_t)i * k + p] * Ri[(size_t)p * k + j];
            Ri[(size_t)i * k + j] = -s / R[(size_t)i * k + i];
        }
    }
}

// eigen-decomposition of a symmetric k x k matrix by cyclic Jacobi rotations: A = V diag(ev) V^T,
// eigenvalues in decreasing order, eigenvectors in the columns of V (row-major)
inline void jacobi_eigen(int k, std::vector<double> A, std::vector<double> &ev, std::vector<double> &V) {
    V.assign((size_t)k * k, 0.0);
    for (int i = 0; i < k; i++) V[(size_t)i * k + i] = 1.0;
    for (int sweep = 0; sweep < 100; sweep++) {
        double off = 0.0, diag = 0.0;
        for (int i = 0; i < k; i++)
            for (int j = 0; j < k; j++) (i == j ? diag : off) += A[(size_t)i * k + j] * A[(size_t)i * k + j];
        if (off <= 1e-30 * diag) break;
        for (int p = 0; p < k - 1; p++)
            for (int q = p + 1; q < k; q++) {
                const double apq = A[(size_t)p * k + q];
                if (apq == 0.0) continue;
                const double theta = (A[(size_t)q * k + q] - A[(size_t)p * k + p]) / (2.0 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
                for (int i = 0; i < k; i++) {  // columns p, q
                    const double aip = A[(size_t)i * k + p], aiq = A[(size_t)i * k + q];
                    A[(size_t)i * k + p] = c * aip - s * aiq;
                    A[(size_t)i * k + q] = s * aip + c * aiq;
                }
                for (int i = 0; i < k; i++) {  // rows p, q
                    const double api = A[(size_t)p * k + i], aqi = A[(size_t)q * k + i];
                    A[(size_t)p * k + i] = c * api - s * aqi;
                    A[(size_t)q * k + i] = s * api + c * aqi;
                }
                for (int i = 0; i < k; i++) {
                    const double vip = V[(size_t)i * k + p], viq = V[(size_t)i * k + q];
                    V[(size_t)i * k + p] = c * vip - s * viq;
                    V[(size_t)i * k + q] = s * vip + c * viq;
                }
            }
    }
    std::vector<int> order((size_t)k);
    for (int i = 0; i < k; i++) order[(size_t)i] = i;
    std::sort(order.begin(), order.end(),
              [&](int a, int b) { return A[(size_t)a * k + a] > A[(size_t)b * k + b]; });
    std::vector<double> Vs((size_t)k * k);
    ev.resize((size_t)k);
    for (int c = 0; c < k; c++) {
        ev[(size_t)c] = A[(size_t)order[(size_t)c] * k + order[(size_t)c]];
        for (int i = 0; i < k; i++) Vs[(size_t)i * k + c] = V[(size_t)i * k + order[(size_t)c]];
    }
    V.swap(Vs);
}

}  // namespace svdhost
