// CUDA kernels of the VB-NMF engine that depend on the padded rank (sm_100a).  See DESIGN.md for
// the data layout and the roofline of each kernel.  Reference maths: src/vbnmf_update.cpp:33-90
// (file:line cited per kernel).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "special.cuh"

#ifndef VB_SPLIT_PRED
#define VB_SPLIT_PRED 0   // split kernels: entries with count 0 (holes) skip their gathers.  Measured
                          // SLOWER (C3-shaped, r = 20: cell-owner pass 3.09 -> 3.49 ms): the branch
                          // around the gathers costs more than the wavefronts it saves
#endif
#ifndef VB_SKIP_DEAD
#define VB_SKIP_DEAD 1    // split kernels: skip the all-hole steps at the end of a segment (their
                          // number rides in the low 2 bits of the segment's quad pointer)
#endif
#ifndef VB_DOT_CHAINS
#define VB_DOT_CHAINS 2   // independent FMA chains of the rank-r dot product (fp64)
#endif
#ifndef VB_LPN_BYTES
#define VB_LPN_BYTES 160    // widest row a single lane gathers; wider rows are split over 2 lanes
#endif

namespace vb {

constexpr int kBlock = 256;  // threads per CTA of the elementwise / reduction kernels
constexpr int kWarpsPerBlock = kBlock / 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kGroup = 8;    // lanes that share one sweep segment (= one LDS.128 bank phase)

// Panel row stride (doubles) for compute width RP (even): RP when RP/2 is odd, else RP + 2, so that
// a row is an ODD number of 16-byte units.  Rows whose indices differ mod 8 then start in
// different 16-byte bank groups of shared memory, which is what the build-time ordering of the
// nonzeros relies on to make the 8 gathers of a quarter-warp conflict-free.
__host__ __device__ constexpr int row_stride(int rp) { return ((rp / 2) & 1) ? rp : rp + 2; }

// fp32 mirror panels (VBNMF_FP32_STORAGE): stride in floats, a multiple of 4 (16 bytes) whose
// number of 16-byte units is odd, for the same bank argument
__host__ __device__ constexpr int row_stride_f32(int rp) {
    return ((((rp + 3) / 4) & 1) ? ((rp + 3) / 4) : ((rp + 3) / 4) + 1) * 4;
}
template <typename PT>
__host__ __device__ constexpr int panel_stride(int rp) {
    return sizeof(PT) == 8 ? row_stride(rp) : row_stride_f32(rp);
}

// ---- split layout of the gathered fp64 panels (lw, lh) -----------------------------------------
// Rows gathered by one lane per nonzero are stored per slab of T rows as two blocks: A = the first
// SA sixteen-byte units of every row with row stride exactly SA units (SA = 8 for ranks 16..20,
// 4 for ranks 8..14), then B = T x split_bs(rp) doubles (the remaining units).
//   SA = 8: block B is dense, RP - 16 doubles per row (0, 1 or 2 units), so a slab is T x RP
//     doubles.  With 2 units (ranks 19, 20) a row of block B covers bank groups 2 (i mod 4) and
//     2 (i mod 4) + 1: four residue classes of TWO lanes each -- lanes l and l + 4 hold rows of
//     class l mod 4, lane l reads unit 8 first and unit 9 second, lane l + 4 the other way round
//     (the registers of block B are rotated by bit 2 of the lane like those of block A by the
//     whole lane index), so a step with at most two rows per class is conflict free.
//   SA = 4: RS - 8 doubles per row (stride an odd number of units or a single unit).
//   SA = 8: a row of block A presents the 8 bank groups of shared memory identically, so the 8
//     lanes of a group, reading unit (c XOR lane) of THEIR row in step c, hit 8 different bank
//     groups whatever the rows are: conflict free with no scheduling at all.
//   SA = 4: a row of block A covers bank groups 0..3 (even row) or 4..7 (odd row); lanes l and
//     l + 4 read the same unit (c XOR (l & 3)), so a step is conflict free when lanes 0..3 hold
//     even rows and lanes 4..7 odd rows -- two parity classes instead of eight residue classes.
// Only block B still depends on the residue schedule of the segment.  tsplit = T selects this
// layout (0: plain row-major rows of RS doubles).
__host__ __device__ constexpr int split_units(int rp) {
    return rp * 8 > VB_LPN_BYTES ? 0 : (rp >= 16 ? 8 : (rp >= 8 ? 4 : 0));
}
__host__ __device__ constexpr bool split_rank(int rp) { return split_units(rp) != 0; }
// doubles per row of block B, and of a whole row of the split layout
__host__ __device__ constexpr int split_bs(int rp) {
    return split_units(rp) == 8 ? rp - 16 : (split_units(rp) == 4 ? row_stride(rp) - 8 : 0);
}
__host__ __device__ constexpr int split_ps(int rp) {
    return split_units(rp) ? 2 * split_units(rp) + split_bs(rp) : row_stride(rp);
}
// tsplit = 0: plain rows of rs doubles; else T | (doubles per row of block B) << 16
__host__ __device__ constexpr int make_tsplit(int T, int rp) { return T | (split_bs(rp) << 16); }
__host__ __device__ __forceinline__ int64_t panel_ofs(int64_t row, int k, int rs, int tsplit) {
    if (tsplit == 0) return row * rs + k;
    const int aw = rs >= 18 ? 16 : 8;  // doubles of block A (rs 10, 14: ranks 8..14; 18, 22: 16..20)
    const int T = tsplit & 0xffff, bs = tsplit >> 16;
    const int64_t slab = row / T, local = row - slab * T;
    return slab * T * (aw + bs) +
           (k < aw ? local * aw + k : (int64_t)T * aw + local * bs + (k - aw));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// deterministic block sum for any blockDim that is a multiple of 32 (<= 1024); valid in thread 0
__device__ __forceinline__ double block_sum(double v, double *sm /* >= blockDim/32 */) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if (lane == 0) sm[w] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < nw; i++) t += sm[i];
    return t;
}

// "last CTA finishes" reduction of per-CTA partial rows: part[b*W + c], b < gridDim.x.
// The last CTA to arrive sums every column c in fixed CTA order into out[c].  counter wraps
// back to 0 by itself (atomicInc), so the same counter serves every launch.
__device__ __forceinline__ void last_block_reduce(const double *part, int W, double *out,
                                                  unsigned *counter, double *sm) {
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t = atomicInc(counter, gridDim.x - 1);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    const int nb = gridDim.x;
    for (int c = 0; c < W; c++) {
        double a = 0.0;
        for (int b = threadIdx.x; b < nb; b += blockDim.x) a += __ldcg(part + (size_t)b * W + c);
        const double s = block_sum(a, sm);
        if (threadIdx.x == 0) out[c] = s;
    }
}

// load one panel row (RP of RS entries, 16-byte aligned) into registers through the read-only path
template <int RP>
__device__ __forceinline__ void load_row_d(const double *__restrict__ base, int64_t row,
                                           double (&out)[RP]) {
    const double2 *p = reinterpret_cast<const double2 *>(base + row * row_stride(RP));
#pragma unroll
    for (int k = 0; k < RP / 2; k++) {
        const double2 v = __ldg(p + k);
        out[2 * k] = v.x;
        out[2 * k + 1] = v.y;
    }
}

// 1/p to ~1 ulp: hardware seed (>= 20 bits) + two Newton steps.  p is a positive normal double
// here (p >= r * fudge^2 > 0), so no special-case handling is needed.
__device__ __forceinline__ double fast_rcp(double p) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(p));
    r = fma(fma(-p, r, 1.0), r, r);
    r = fma(fma(-p, r, 1.0), r, r);
    return r;
}

// ---- mbarrier / bulk-copy (TMA) primitives ---------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
    // bounded spin: a bulk copy that never lands (bad address) traps instead of hanging the GPU
    for (unsigned spin = 0; !mbar_try_wait(bar, parity); spin++)
        if (spin > (1u << 26)) __trap();
}
// one bulk asynchronous copy global -> shared (the TMA engine, SASS UBLKCP); bytes % 16 == 0
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, unsigned bytes,
                                         uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ------------------------------------------------------------------------------------------
// Tiled nonzero sweep.  Both passes of the sweep are this kernel:
//   COLS = true  (cell-owner pass, src/vbnmf_update.cpp:33-34,36 and the data term of :73-77)
//       owner = cell j (lh_j in registers), tile = a slab of T gene rows of lw in shared memory,
//       Part[slab][j][k] = sum_{i in slab} lw_ik q_ij ; plus sum x_ij log p_ij
//   COLS = false (gene-owner pass, src/vbnmf_update.cpp:33-35)
//       owner = gene i (lw_i in registers), tile = a slab of T cell rows of lh in shared memory,
//       Part[slab][i][k] = sum_{j in slab} q_ij lh_kj
// with p_ij = sum_k lw_ik lh_kj and q_ij = x_ij / p_ij recomputed in each pass.
//
// Work decomposition: the nonzeros are stored slab-major in "segments" e = slab * NO + owner
// (ptr[e] .. ptr[e+1]).  CTA b owns the contiguous segment range split[b] .. split[b+1], chosen at
// build time so that every CTA gets the same number of nonzeros; it stages each slab it touches
// with ONE bulk asynchronous copy (TMA) into shared memory, then its 8-lane groups walk their
// segments gathering tile rows with 128-bit shared loads.  Outputs are plain stores: no atomics.
//
// The build step orders the nonzeros of a segment so that 8 consecutive ones hit tile rows that
// differ mod 8 -> with an odd row stride the 8 gathers of a group are bank-conflict free.
// This kernel serves the 8-byte {row, float} and the {row} + {double} entry formats; integer
// counts below 2^16 take sweep_p16_kernel further down (same passes, same outputs).
// VB_UNROLL: nonzeros per lane whose index/count loads are in flight together and whose arithmetic
// chains are interleaved: 6 for the fp64 single-lane configuration, 4 otherwise (measured on C2:
// fp64 1.81 -> 1.76 ms with 6; the fp32 mode and the two-lane variant are faster with 4, 2 is
// slower everywhere)
#ifndef VB_UNROLL
#define VB_UNROLL 0
#endif
#ifndef VB_SWEEP_THREADS
#define VB_SWEEP_THREADS 512  // threads per sweep CTA for the narrow-rank configuration
#endif
#ifndef VB_SWEEP_THREADS_F32
#define VB_SWEEP_THREADS_F32 640  // ... of the fp32-storage kernels with rows of up to 48 bytes
                                  // (C2: 0.98 -> 0.94 ms per iteration against 512; 768: 0.95)
#endif
#ifndef VB_MID_THREADS
#define VB_MID_THREADS 384   // threads per sweep CTA when a lane holds 97..160 bytes of a row
#endif
#ifndef VB_MID_THREADS_COLS
#define VB_MID_THREADS_COLS VB_MID_THREADS
#endif
#ifndef VB_WIDE_THREADS
#define VB_WIDE_THREADS 256  // ... more than 160 bytes
#endif
#ifndef VB_G4_NU9
#define VB_G4_NU9 1       // 4-lane groups also for rows of 9 units (ranks 17, 18).  The single unit of
                          // block B (bank group = row mod 8) makes lanes l and l + 4 of a bank phase
                          // collide when their rows agree in bit 2; the builder orders the classes of
                          // even / odd positions in opposite directions to avoid most of it.  Measured
                          // (C2 matrix, r = 18): 2.35 -> 2.20 ms per iteration against 8-lane groups
#endif
#ifndef VB_OWN_AHEAD
#define VB_OWN_AHEAD(dflt) (dflt)
#endif
#ifndef VB_OWN_EARLY
#define VB_OWN_EARLY 1    // owner rows that cannot be requested a whole segment ahead (register budget)
                          // are requested before the cross-lane sum of the previous segment, when
                          // the registers of the old owner row are free, instead of at segment start
                          // (measured at C2: cell-owner pass 0.744 -> 0.708 ms)
#endif
#ifndef VB_OWN_STAGE
#define VB_OWN_STAGE 0    // 1: owner rows that cannot be requested a whole segment ahead in registers are
                          // staged through shared memory instead: cp.async into an 8-lane group's own
                          // slot behind the tile during the previous segment, read back with LDS at
                          // segment start.  Built and measured: -0.7 % at r = 20 before the segments
                          // were length-sorted, but with the final layouts the slots' share of the
                          // tile costs more than the latency they hide (C2 matrix: r = 10 1.379 vs
                          // 1.360 ms per iteration without, r = 12 1.70 vs 1.62, r = 30 4.96 vs
                          // 4.73), so it is off: the row is requested before the cross-lane sum of
                          // the previous segment (VB_OWN_EARLY)
#endif

template <int RP, typename PT>
struct SweepCfg {
    // Register budget per lane: own + acc + tile row = 3 * KL values of PT plus the prefetched
    // entries.  A lane gathers rows of up to 160 bytes by itself (r <= 20 in fp64), with 512 threads
    // per SM up to 96 bytes and 384 beyond; measured at C2 size, one lane per nonzero at 384
    // threads beats two lanes at 512 by 25 % (r = 14) to 7 % (r = 20).  Wider rows are split over
    // LPN = 2 lanes per nonzero (each lane takes every other 16-byte unit of the row).
    static constexpr int kUE = 16 / (int)sizeof(PT);             // elements per 16-byte unit
    static constexpr int kNU = (RP + kUE - 1) / kUE;             // units per row
    static constexpr int kLPN = (RP * (int)sizeof(PT) > VB_LPN_BYTES) ? 2 : 1;  // lanes per nonzero
    static constexpr int kNUL = (kNU + kLPN - 1) / kLPN;         // units per lane
    static constexpr int kKL = kNUL * kUE;                       // rank entries per lane
    static constexpr int kNPG = kGroup / kLPN;                   // nonzeros per group step
    static constexpr int kRowShare = kKL * (int)sizeof(PT);      // bytes of a row per lane
    static constexpr int kThreads = kRowShare <= 96 ? (sizeof(PT) == 4 && kRowShare <= 48
                                                           ? VB_SWEEP_THREADS_F32 : VB_SWEEP_THREADS)
                                    : (kRowShare <= 160 ? VB_MID_THREADS : VB_WIDE_THREADS);
    // unroll of the chunk loop; the fp32 cell-owner pass (with its log) is the one that prefers 4
    __host__ __device__ static constexpr int unroll(bool cols) {
        return VB_UNROLL ? VB_UNROLL : ((kLPN == 1 && (sizeof(PT) == 8 || !cols)) ? 6 : 4);
    }
    static constexpr int kGroups = kThreads / kGroup;
    // threads of the packed-16 kernel per pass: the fp64 cell-owner pass of the 97..160-byte rows
    // also carries the log-product state and spills at kThreads
    __host__ __device__ static constexpr int p16_threads(bool cols) {
        return (cols && sizeof(PT) == 8 && kRowShare > 96 && kRowShare <= 160) ? VB_MID_THREADS_COLS
                                                                               : kThreads;
    }
    // packed-16 kernels: the next owner row is requested a whole segment ahead, into registers,
    // where the register budget allows it (checked with -Xptxas -v: wider row shares, and the fp64
    // cell-owner pass with its log, spill) ...
    __host__ __device__ static constexpr bool own_ahead(bool cols) {
        return VB_OWN_AHEAD(kRowShare <= 48 ||
                            (kRowShare <= 80 && sizeof(PT) == 8 && !cols && kLPN == 1));
    }
    // ... and staged through shared memory otherwise: bytes of one group's slot (all kNU units of
    // a row), and of the slots of the larger of the two passes' CTAs (what the host leaves free
    // behind the tile)
    __host__ __device__ static constexpr int stage_bytes(bool, bool) { return kNU * 16; }
    __host__ __device__ static constexpr int stage_pass(bool cols, int g) {
        return (VB_OWN_STAGE && g == 8 && !own_ahead(cols)) ? p16_threads(cols) / g * kNU * 16 : 0;
    }
    __host__ __device__ static constexpr int stage_total(int g = 8) {
        return stage_pass(true, g) > stage_pass(false, g) ? stage_pass(true, g) : stage_pass(false, g);
    }
    // 4-lane groups (sweep_p16_kernel, G = 4): split layout with an 8-unit block A and no
    // single-unit block B
    __host__ __device__ static constexpr bool g4() {
        return sizeof(PT) == 8 && kLPN == 1 && split_units(RP) == 8 && (VB_G4_NU9 || kNU != 9);
    }
};


// log(p) for a positive normal double, ~1 ulp: p = 2^e m with m in [sqrt(1/2), sqrt(2)),
// log m = 2 atanh(t), t = (m-1)/(m+1), |t| <= 0.1716, odd series through t^17 (next term < 3e-16).
// No special cases (p > 0 finite is guaranteed by the fudge floor), ~20 FP64 + ~8 integer ops
// against ~90 for the general log().
static __constant__ double kLogC[10] = {2.0 / 17.0, 2.0 / 15.0, 2.0 / 13.0, 2.0 / 11.0, 2.0 / 9.0,
                                 2.0 / 7.0,  2.0 / 5.0,  2.0 / 3.0,
                                 6.93147180369123816490e-01,   // ln2 hi (exact product with e)
                                 1.90821492927058770002e-10};  // ln2 lo
__device__ __forceinline__ double fast_log_pos(double p) {
    int hi = __double2hiint(p);
    const int lo = __double2loint(p);
    int e = (hi >> 20) - 1023;
    hi = (hi & 0x000fffff) | 0x3ff00000;
    if (hi >= 0x3ff6a09f) { hi -= 0x00100000; e += 1; }
    const double m = __hiloint2double(hi, lo);
    const double t = (m - 1.0) * fast_rcp(m + 1.0);
    const double t2 = t * t;
    double s = kLogC[0];
#pragma unroll
    for (int i = 1; i < 8; i++) s = fma(s, t2, kLogC[i]);
    const double lm = fma(t * t2, s, t + t);
    const double de = (double)e;
    return fma(de, kLogC[8], fma(de, kLogC[9], lm));
}

// 128-bit shared load from a 32-bit shared-window address (keeps the tile base in one register
// instead of re-deriving it from the generic pointer at every gather)
__device__ __forceinline__ double2 lds128(uint32_t addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}

__device__ __forceinline__ float4 lds128f(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "r"(addr));
    return v;
}
__device__ __forceinline__ double rcp_t(double p) { return fast_rcp(p); }
__device__ __forceinline__ float rcp_t(float p) { return __frcp_rn(p); }
__device__ __forceinline__ double log_t(double p) { return fast_log_pos(p); }
__device__ __forceinline__ float log_t(float p) { return __logf(p); }

__device__ __forceinline__ void prefetch_l2(const void *p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// storage formats of the nonzeros in the tiled layouts
enum { kEntF32 = 0,   // 8 bytes {int32 tile row, float count}
       kEntF64 = 1,   // int32 tile row + double count in two arrays (counts not exact in fp32)
       kEntP16 = 2 }; // 4 bytes {count << 16 | tile row}: integer counts < 2^16 (sweep_p16_kernel)

struct SweepTiledArgs {
    int64_t NO;              // owners per slab (device-ordered rows of the owner panel)
    int T;                   // tile rows
    const int64_t *split;    // gridDim.x + 1 segment indices
    const int64_t *ptr;      // segment pointers, nslabs*NO + 1
    const void *ent;         // float counts: packed {int32 tile row, float count} per nonzero
    const int32_t *idx;      // double counts: tile row of each nonzero ...
    const double *val;       // ... and its count
    const void *owner;       // owner panel, NO x stride (double, or float in fp32-storage mode)
    const void *tiles;       // tile panel, nslabs*T x stride
    double *Part;            // nslabs x NO x RS
    double *xl_part;         // COLS: gridDim.x partial sums of x log p
    const double *ctl;       // device loop control block (see control_kernel) or nullptr
    const uint32_t *ptr4;    // packed-16 layout: segment pointers in units of 4 entries (16 bytes)
    const uint32_t *seg;     // packed-16 layout: owner row of each segment position (inside windows
                             // of consecutive owners the segments are stored by decreasing length)
};

// Device loop control block (doubles).  When a kernel is given it and ctl[kCtlDone] != 0 the run
// has ended (converged / NaN / Itmax) and the kernel returns at once, so iterations launched ahead
// of the host's knowledge are no-ops.
enum { kCtlDone = 0, kCtlIt = 1, kCtlLk0 = 2, kCtlReason = 3, kCtlHyper = 4 /*aw,bw,ah,bh*/,
       kCtlHyperErr = 8, kCtlLkh = 9, kCtlAcc = 10 /*wacc[3], hacc[3]*/, kCtlBew = 16,
       kCtlBeh = 16 + 64, kCtlEhsum = 16 + 128, kCtlLen = 16 + 192 };

template <typename VT>
__device__ __forceinline__ void load_entry(const SweepTiledArgs &a, int64_t t, int32_t &ti, double &x);
template <>
__device__ __forceinline__ void load_entry<float>(const SweepTiledArgs &a, int64_t t, int32_t &ti,
                                                  double &x) {
    const int2 v = __ldcs(reinterpret_cast<const int2 *>(a.ent) + t);
    ti = v.x;
    x = (double)__int_as_float(v.y);
}
template <>
__device__ __forceinline__ void load_entry<double>(const SweepTiledArgs &a, int64_t t, int32_t &ti,
                                                   double &x) {
    ti = __ldcs(a.idx + t);
    x = __ldcs(a.val + t);
}

// one 16-byte unit of a panel row from global memory (read-only path) / shared memory
__device__ __forceinline__ void ldg_unit(const double *row, int u, double *out) {
    const double2 v = __ldg(reinterpret_cast<const double2 *>(row) + u);
    out[0] = v.x; out[1] = v.y;
}
__device__ __forceinline__ void ldg_unit(const float *row, int u, float *out) {
    const float4 v = __ldg(reinterpret_cast<const float4 *>(row) + u);
    out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
}
__device__ __forceinline__ void lds_unit(uint32_t addr, double *out) {
    const double2 v = lds128(addr);
    out[0] = v.x; out[1] = v.y;
}
__device__ __forceinline__ void lds_unit(uint32_t addr, float *out) {
    const float4 v = lds128f(addr);
    out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
}

template <int RP, typename VT, bool COLS, typename PT>
__global__ void __launch_bounds__(SweepCfg<RP, PT>::kThreads, 1)
sweep_tiled_kernel(const SweepTiledArgs a) {
    using Cfg = SweepCfg<RP, PT>;
    constexpr int RS = row_stride(RP);          // stride of the fp64 Part rows
    constexpr int PS = panel_stride<PT>(RP);    // stride of the gathered / owner panels
    constexpr int NT = Cfg::kThreads, U = Cfg::unroll(COLS);
    constexpr int UE = Cfg::kUE, NU = Cfg::kNU, LPN = Cfg::kLPN, NUL = Cfg::kNUL, KL = Cfg::kKL;
    constexpr int NPG = Cfg::kNPG;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    PT *tile = reinterpret_cast<PT *>(smem_raw);
    const uint32_t tile_s = smem_u32(tile);
    __shared__ __align__(8) uint64_t mbar;
    __shared__ double red[NT / 32];
    const int gid = threadIdx.x / kGroup, gl = threadIdx.x % kGroup;
    const int slot = gl / LPN, hf = gl % LPN;   // nonzero slot within the group step, rank half
    // the 4 groups of a warp run different trip counts: shuffles name only their own 8 lanes
    const unsigned gmask = 0xffu << ((threadIdx.x & 31) & ~(kGroup - 1));
    const int64_t e0 = a.split[blockIdx.x], e1 = a.split[blockIdx.x + 1];
    const unsigned tile_bytes = (unsigned)a.T * PS * (unsigned)sizeof(PT);
    if (a.ctl && a.ctl[kCtlDone] != 0.0) return;  // uniform over the grid: the run has ended
    if (threadIdx.x == 0) mbar_init(&mbar, 1);
    __syncthreads();
    unsigned parity = 0;
    double xl = 0.0;  // sum x log p of this thread's nonzeros (COLS)

    for (int64_t ebase = e0; ebase < e1;) {
        const int64_t slab = ebase / a.NO;
        const int64_t eend = min(e1, (slab + 1) * a.NO);
        __syncthreads();  // every group is done with the previous tile
        if (threadIdx.x == 0) {
            mbar_expect_tx(&mbar, tile_bytes);
            bulk_g2s(tile, reinterpret_cast<const PT *>(a.tiles) + slab * (int64_t)a.T * PS,
                     tile_bytes, &mbar);
        }
        mbar_wait(&mbar, parity);
        parity ^= 1;
        for (int64_t e = ebase + gid; e < eend; e += Cfg::kGroups) {
            const int64_t o = e - slab * a.NO;
            const int64_t beg = __ldg(a.ptr + e), end = __ldg(a.ptr + e + 1);
            // pull the entries of this group's NEXT segment from HBM into L2 while this one runs
            if (sizeof(VT) == 4 && e + Cfg::kGroups < eend) {
                const int64_t nb = __ldg(a.ptr + e + Cfg::kGroups);
                const int64_t ne = __ldg(a.ptr + e + Cfg::kGroups + 1);
                for (int64_t t = nb + gl * 16; t < ne; t += kGroup * 16)
                    prefetch_l2(reinterpret_cast<const int2 *>(a.ent) + t);
            }
            PT acc[KL];
            PT xls = 0;  // x log p of this segment in the arithmetic type
#pragma unroll
            for (int k = 0; k < KL; k++) acc[k] = 0;
            if (beg < end) {
                // this lane's share of the owner row: units hf, hf + LPN, ...
                PT own[KL];
                const PT *orow = reinterpret_cast<const PT *>(a.owner) + o * PS;
#pragma unroll
                for (int c = 0; c < NUL; c++) {
                    const int u = LPN * c + hf;
#pragma unroll
                    for (int j = 0; j < UE; j++) own[c * UE + j] = 0;
                    if (u < NU) ldg_unit(orow, u, own + c * UE);
                }
                // software pipeline: the U index/count loads of the next chunk are issued before
                // the current chunk is processed.  Slots past the end of the segment carry a zero
                // count and tile row 0: they run through the same arithmetic and add nothing, so
                // the U chains of a chunk are branch-free and can be interleaved by the scheduler.
                const int len = (int)(end - beg);
                int32_t ti[U], tn[U];
                double xv[U], xn[U];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int t = slot + u * NPG;
                    ti[u] = 0; xv[u] = 0.0;
                    if (t < len) load_entry<VT>(a, beg + t, ti[u], xv[u]);
                }
                for (int c0 = 0; c0 < len; c0 += U * NPG) {
                    PT pu[U], xu[U];  // LPN == 2: p and count of the chunk for the paired log
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        const int t = c0 + U * NPG + slot + u * NPG;
                        tn[u] = 0; xn[u] = 0.0;
                        if (t < len) load_entry<VT>(a, beg + t, tn[u], xn[u]);
                    }
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        const PT x = (PT)xv[u];
                        const uint32_t raddr = tile_s + (uint32_t)ti[u] * (PS * (int)sizeof(PT));
                        PT tr[KL];
#pragma unroll
                        for (int c = 0; c < NUL; c++) {
                            const int uu = LPN * c + hf;
                            if (LPN == 1 || uu < NU) {
                                lds_unit(raddr + uu * 16, tr + c * UE);
                            } else {
#pragma unroll
                                for (int j = 0; j < UE; j++) tr[c * UE + j] = 0;
                            }
                        }
                        PT p0 = 0, p1 = 0;
#pragma unroll
                        for (int k = 0; k < KL; k += 2) {
                            p0 = fma(own[k], tr[k], p0);
                            p1 = fma(own[k + 1], tr[k + 1], p1);
                        }
                        PT p = p0 + p1;
                        if (LPN == 2) p += __shfl_xor_sync(gmask, p, 1);
                        const PT q = x * rcp_t(p);
#pragma unroll
                        for (int k = 0; k < KL; k++) acc[k] = fma(tr[k], q, acc[k]);
                        if (COLS) {
                            if (LPN == 1) xls = fma(x, log_t(p), xls);
                            else { pu[u] = p; xu[u] = x; }
                        }
                    }
                    if (COLS && LPN == 2) {
                        // both lanes of a pair hold p: each takes the log of every other nonzero
#pragma unroll
                        for (int v = 0; v < U / 2; v++) {
                            const PT pm = hf ? pu[2 * v + 1] : pu[2 * v];
                            const PT xm = hf ? xu[2 * v + 1] : xu[2 * v];
                            xls = fma(xm, log_t(pm), xls);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < U; u++) { ti[u] = tn[u]; xv[u] = xn[u]; }
                }
                if (COLS) xl += (double)xls;
            }
            // sum over the lanes of the group that hold the same rank entries, in fp64
            double *out = a.Part + e * RS;
#pragma unroll
            for (int k = 0; k < KL; k++) {
                double s = (double)acc[k];  // fp64 from here on (sums over lanes, slabs, ranks)
                s += __shfl_xor_sync(gmask, s, 4);
                s += __shfl_xor_sync(gmask, s, 2);
                if (LPN == 1) s += __shfl_xor_sync(gmask, s, 1);
                const int kk = (LPN * (k / UE) + hf) * UE + (k % UE);  // rank index of entry k
                if (LPN == 1) {
                    if ((k % kGroup) == gl && kk < RP) out[kk] = s;
                } else {
                    if (slot == (k % NPG) && kk < RP) out[kk] = s;
                }
            }
        }
        ebase = eend;
    }
    if (COLS) {
        xl = block_sum(xl, red);
        if (threadIdx.x == 0) a.xl_part[blockIdx.x] = xl;
    }
}

// ------------------------------------------------------------------------------------------
// Packed-16 variant of the tiled sweep (same maths, same outputs as sweep_tiled_kernel).
//
// When every count is an integer below 2^16 (true for raw UMI counts) a nonzero is ONE 32-bit word
// {count << 16 | tile row}: half the bytes of the {int32, float} entries, and a lane fetches FOUR
// nonzeros with one 128-bit load.  Segments are padded to a multiple of 4 entries with zero words
// (row 0, count 0: they run through the arithmetic and add nothing), so every segment starts on a
// 16-byte boundary and the pointers are 32-bit quad indices (ptr4).
//
// Placement inside a segment (build_segments_p16_kernel): the round-robin residue order of the
// 8-byte layout is kept, but in blocks of 4*NPG entries item p goes to quad (p mod q), word
// (p div q), q = quads of the block: the nonzeros the lanes of a group process in the same step
// are consecutive items of that order -> the same conflict-free gathers.
//
// Latency: everything a segment needs first is already in registers when it starts -- its first
// quad and its owner row were requested while the previous segment ran, its pointers one segment
// before that -- and the rest of its entries were pulled into L2 by ONE bulk prefetch (TMA unit,
// no LSU wavefronts).  Inside a segment the quads are loaded two chunks ahead.
// The cross-lane sum of the per-lane accumulators is a recursive halving (each step a lane keeps
// half of its values and sends the other half): KL/2 + KL/4 + .. shuffles instead of 3*KL.
__device__ __forceinline__ void bulk_prefetch_l2(const void *p, unsigned bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint4 ldcs_quad(const uint4 *p) { return __ldcs(p); }

// Packed fp32 arithmetic (Blackwell FFMA2: two fp32 FMAs per instruction on a 64-bit register
// pair): 2*KL of the ~60 instructions per nonzero of the fp32-storage sweep are FMAs on pairs of
// adjacent rank entries.  Measured at C2 it changes nothing (0.979 -> 0.988 ms per iteration at
// 512 threads, 0.941 -> 0.939 at 640): the pass is not issue-limited.  Off by default (VB_FFMA2).
__device__ __forceinline__ unsigned long long pack_f2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack_f2(unsigned long long v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b,
                                                    unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
// p = sum_k own[k] tr[k];  acc[k] += tr[k] * x / p   (one nonzero; returns p)
template <int KL>
__device__ __forceinline__ double dot_rows(const double (&own)[KL], const double (&tr)[KL]) {
    if (VB_DOT_CHAINS == 4 && KL % 4 == 0) {
        double p0 = 0, p1 = 0, p2 = 0, p3 = 0;
#pragma unroll
        for (int k = 0; k < KL; k += 4) {
            p0 = fma(own[k], tr[k], p0);
            p1 = fma(own[k + 1], tr[k + 1], p1);
            p2 = fma(own[k + 2], tr[k + 2], p2);
            p3 = fma(own[k + 3], tr[k + 3], p3);
        }
        return (p0 + p1) + (p2 + p3);
    }
    double p0 = 0, p1 = 0;
#pragma unroll
    for (int k = 0; k < KL; k += 2) {
        p0 = fma(own[k], tr[k], p0);
        p1 = fma(own[k + 1], tr[k + 1], p1);
    }
    return p0 + p1;
}
template <int KL>
__device__ __forceinline__ void axpy_row(double (&acc)[KL], const double (&tr)[KL], double q) {
#pragma unroll
    for (int k = 0; k < KL; k++) acc[k] = fma(tr[k], q, acc[k]);
}
#ifndef VB_FFMA2
#define VB_FFMA2 0
#endif
template <int KL>
__device__ __forceinline__ float dot_rows(const float (&own)[KL], const float (&tr)[KL]) {
    if (VB_FFMA2 && KL % 4 == 0) {
        unsigned long long pa = 0ull, pb = 0ull;  // two chains of pairs
#pragma unroll
        for (int k = 0; k < KL; k += 4) {
            pa = ffma2(pack_f2(own[k], own[k + 1]), pack_f2(tr[k], tr[k + 1]), pa);
            pb = ffma2(pack_f2(own[k + 2], own[k + 3]), pack_f2(tr[k + 2], tr[k + 3]), pb);
        }
        float a0, a1, b0, b1;
        unpack_f2(pa, a0, a1);
        unpack_f2(pb, b0, b1);
        return (a0 + a1) + (b0 + b1);
    }
    float p0 = 0, p1 = 0;
#pragma unroll
    for (int k = 0; k < KL; k += 2) {
        p0 = fmaf(own[k], tr[k], p0);
        p1 = fmaf(own[k + 1], tr[k + 1], p1);
    }
    return p0 + p1;
}
template <int KL>
__device__ __forceinline__ void axpy_row(float (&acc)[KL], const float (&tr)[KL], float q) {
    if (VB_FFMA2 && KL % 2 == 0) {
        const unsigned long long qq = pack_f2(q, q);
#pragma unroll
        for (int k = 0; k < KL; k += 2) {
            const unsigned long long r = ffma2(pack_f2(tr[k], tr[k + 1]), qq, pack_f2(acc[k], acc[k + 1]));
            unpack_f2(r, acc[k], acc[k + 1]);
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < KL; k++) acc[k] = fmaf(tr[k], q, acc[k]);
}

// one halving step over the lanes that differ in bit BIT of the group lane: N values -> ceil(N/2)
template <int N, int BIT>
__device__ __forceinline__ void halve_step(const double (&in)[N], double (&out)[(N + 1) / 2],
                                           int gl, unsigned gmask) {
    constexpr int Hh = (N + 1) / 2;
    const bool hi = (gl & BIT) != 0;
#pragma unroll
    for (int k = 0; k < Hh; k++) {
        const double lo_v = in[k];
        const double hi_v = (Hh + k < N) ? in[Hh + k] : 0.0;
        const double send = hi ? lo_v : hi_v;
        const double keep = hi ? hi_v : lo_v;
        out[k] = keep + __shfl_xor_sync(gmask, send, BIT);
    }
}

// sum of N per-lane values over the 8 lanes of a group by recursive halving, then out[i] = sum_i
// for i < limit: every lane ends up with at most ceil(N/8) of the sums and stores those
template <int N>
__device__ __forceinline__ void halve_reduce_store(const double (&v0)[N], int gl, unsigned gmask,
                                                   double *out, int limit) {
    constexpr int H1 = (N + 1) / 2, H2 = (H1 + 1) / 2, H3 = (H2 + 1) / 2;
    double v1[H1], v2[H2], v3[H3];
    halve_step<N, 4>(v0, v1, gl, gmask);
    halve_step<H1, 2>(v1, v2, gl, gmask);
    halve_step<H2, 1>(v2, v3, gl, gmask);
    const int o1 = (gl & 4) ? H1 : 0, o2 = (gl & 2) ? H2 : 0, o3 = (gl & 1) ? H3 : 0;
#pragma unroll
    for (int k = 0; k < H3; k++) {
        const int i2 = k + o3, i1 = i2 + o2, i0 = i1 + o1;  // index in v0[]
        if (i2 < H2 && i1 < H1 && i0 < N && i0 < limit) out[i0] = v3[k];
    }
}

// x log p of the fp64 cell-owner pass through products (integer counts): with p = 2^e m and
// x' = x mod 2^kLpBits,
//   sum x' log p = ln2 * sum x' e + log prod m^x',   m^x' = prod_{bit b of x' set} m^(2^b),
// so a nonzero costs kLpBits - 1 squarings, kLpBits selected multiplies and a few integer
// operations instead of a log (~35 instructions), and the state is one product, one exponent sum
// and one accumulator.  The product grows by less than 2^(4 (2^kLpBits - 1)) per chunk of four
// nonzeros and is renormalised after each.  The rest of a count >= 2^kLpBits, (x - x') log p,
// takes the log in an out-of-line slow path.
#ifndef VB_LP_BITS
#define VB_LP_BITS 3   // 4 keeps counts up to 15 in the fast path (data with heavier tails)
#endif
constexpr int kLpBits = VB_LP_BITS;
struct LogProd {
    double P;       // prod m^(x mod 2^kLpBits), renormalised to [1, 2) after every chunk
    int E;          // sum x e and the exponents taken out of P, of the current segment
    double sum;     // ln2 E of the finished segments and the slow-path terms
    __device__ __forceinline__ void init() { P = 1.0; E = 0; sum = 0.0; }
    // v: packed entry, count in the high 16 bits
    __device__ __forceinline__ void add(uint32_t v, double p) {
        const int hi = __double2hiint(p);
        const int e = (hi >> 20) - 1023;  // p > 0: the sign bit is clear
        double m = __hiloint2double(hi - (e << 20), __double2loint(p));
        E += (int)((v >> 16) & ((1u << kLpBits) - 1u)) * e;
#pragma unroll
        for (int b = 0; b < kLpBits; b++) {
            if (b) m *= m;
            if ((v >> (16 + b)) & 1u) P *= m;
        }
    }
    __device__ __forceinline__ void renorm() {
        const int hi = __double2hiint(P);
        const int e = (hi >> 20) - 1023;
        E += e;
        P = __hiloint2double(hi - (e << 20), __double2loint(P));
    }
    // counts >= 2^kLpBits (rare): the bits above the low kLpBits
    __device__ __forceinline__ void add_slow(uint32_t v, double p) {
        sum = fma((double)(int)((v >> (16 + kLpBits)) << kLpBits), fast_log_pos(p), sum);
    }
    __device__ __forceinline__ void end_segment() {
        sum = fma((double)E, 0.6931471805599453094, sum);
        E = 0;
    }
    __device__ __forceinline__ double total() const { return sum + log(P); }
};

// SPLIT (fp64 panels, one lane per nonzero, rows of >= 8 units; see split_rank / panel_ofs): the
// tile is stored as block A (T x 128 bytes) + block B; lane gl gathers unit c ^ gl of block A in
// step c -- conflict free for ANY 8 rows -- and holds its owner row and accumulators in the same
// rotated order; the cross-lane sum un-rotates for free (partner gl ^ b holds my unit of register
// c in its register c ^ b).  Schedule holes (count 0) gather a real row and add nothing; with
// VB_SPLIT_PRED they would skip their gathers (measured slower).
// G = lanes per segment: 8, or 4 for the split layout with an 8-unit block A.  The rotation of
// block A only needs the 8 lanes of a quarter-warp to read 8 different units, whatever segments
// their rows belong to, so two 4-lane groups can share a bank phase; each lane then walks twice as
// many steps per segment and the per-segment work (owner row, pointers, cross-lane sum, pipeline
// drain and fill) is paid half as often per nonzero.  Block B (two dense units): the groups of a
// quarter-warp read its units in opposite order (even / odd bank groups), and inside a group the
// four rows of a step must differ mod 4 (kSchedOne4).
template <int RP, bool COLS, typename PT, bool SPLIT = false, int G = 8>
__global__ void __launch_bounds__(SweepCfg<RP, PT>::p16_threads(COLS), 1)
sweep_p16_kernel(const SweepTiledArgs a) {
    using Cfg = SweepCfg<RP, PT>;
    constexpr int RS = row_stride(RP);
    constexpr int PS = panel_stride<PT>(RP);
    static_assert(!SPLIT || (sizeof(PT) == 8 && Cfg::kLPN == 1 && split_units(RP) != 0),
                  "split layout: fp64 panels, one lane per nonzero, 4..10 units per row");
    constexpr int SA = SPLIT ? split_units(RP) : 8;          // units of block A (8 or 4)
    constexpr int NUB = SPLIT ? Cfg::kNU - SA : 0;           // units of block B
    constexpr int BSD = SPLIT ? split_bs(RP) : 0;            // doubles per row of block B
    constexpr int BSB = BSD * 8;                             // ... bytes
    constexpr int PSS = SPLIT ? split_ps(RP) : PS;           // doubles per row of a slab
    // block B of two dense units: registers rotated by bit 2 of the lane (see split layout above)
    constexpr bool kRotB = SPLIT && SA == 8 && NUB == 2 && BSD == 4;
    constexpr int NT = Cfg::p16_threads(COLS);
    constexpr int UE = Cfg::kUE, NU = Cfg::kNU, LPN = Cfg::kLPN, NUL = Cfg::kNUL, KL = Cfg::kKL;
    static_assert(G == 8 || (G == 4 && SPLIT && split_units(RP) == 8 && (VB_G4_NU9 || Cfg::kNU != 9)),
                  "4-lane groups: split layout, 8-unit block A, block B empty or two dense units");
    constexpr int NPG = G / LPN;
    constexpr int kGroups = NT / G;
    // the next owner row is requested one segment ahead where the register budget allows it
    // (checked with -Xptxas -v: wider row shares, and the fp64 cell-owner pass with its log, spill)
    constexpr int kRowShare = KL * (int)sizeof(PT);  // bytes of a row held per lane
    constexpr bool kOwnAhead = Cfg::own_ahead(COLS);
    // 1: a whole segment ahead; 2: before the cross-lane sum of the previous segment (the old owner
    // row's registers are free by then); 0: at the start of its segment
    // 3: staged through shared memory a segment ahead (sweep_stage_bytes() behind the tile)
    // (4-lane groups: twice the slots would cost 5 % of the tile height; measured 0.8 % slower)
    constexpr int kOwnMode = kOwnAhead ? 1 : ((VB_OWN_STAGE && G == 8) ? 3 : (VB_OWN_EARLY ? 2 : 0));
    static_assert(kOwnMode != 3 || Cfg::stage_bytes(COLS, SPLIT) > 0, "staging slot size");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    PT *tile = reinterpret_cast<PT *>(smem_raw);
    const uint32_t tile_s = smem_u32(tile);
    __shared__ __align__(8) uint64_t mbar;
    __shared__ double red[NT / 32];
    __shared__ uint32_t range_end;  // e1 below, read once per slab instead of held in a register
    const int gid = threadIdx.x / G, gl = threadIdx.x % G;
    const int l8 = threadIdx.x & 7;  // lane in the quarter-warp (bank phase): rotation of the gathers
    const int slot = gl / LPN, hf = gl % LPN;
    const unsigned gmask = ((1u << G) - 1u) << ((threadIdx.x & 31) & ~(G - 1));
    const unsigned pmask = 3u << ((threadIdx.x & 31) & ~1);  // the two lanes of a nonzero (LPN == 2)
    // segment positions fit in 32 bits with a group stride to spare (build_pass checks it)
    const uint32_t e0 = (uint32_t)a.split[blockIdx.x], e1 = (uint32_t)a.split[blockIdx.x + 1];
    const uint32_t NO = (uint32_t)a.NO;
    const unsigned tile_bytes = (unsigned)a.T * PSS * (unsigned)sizeof(PT);
    const uint4 *ent4 = reinterpret_cast<const uint4 *>(a.ent);
    if (a.ctl && a.ctl[kCtlDone] != 0.0) return;
    // the tile barrier completes one phase per slab; its phase parity is kept equal to the parity
    // of the slab index (one empty phase first when the CTA starts at an odd slab), so that no
    // register has to count the phases
    if (threadIdx.x == 0) {
        range_end = e1;
        mbar_init(&mbar, 1);
        if ((e0 / NO) & 1u) mbar_arrive(&mbar);
    }
    __syncthreads();
    double xl = 0.0;
    constexpr bool kLogProd = COLS && sizeof(PT) == 8;  // fp64 cell-owner pass: log-product
    LogProd lp;
    if (kLogProd) lp.init();

    // tile bases of the split layout plus this lane's rotation: a row of block A starts at a
    // multiple of SA * 16 bytes, one of block B with kRotB at a multiple of 32, so that adding the
    // rotation to the base is XORing it into the row address
    const uint32_t tileA_r = tile_s + ((uint32_t)(l8 & (SA - 1)) << 4);
    const uint32_t tileB_r = tile_s + (uint32_t)a.T * (uint32_t)(SA * 16) +
                             (kRotB ? (uint32_t)((l8 >> 2) & 1) << 4 : 0u);
    if (SPLIT && (tile_s & 127u)) __trap();  // block A rows must start on SA * 16-byte boundaries

    // Owner rows.  A lane holds units hf, hf + LPN, ... of the row (SPLIT: in the rotated order of
    // its tile gathers).  SPLIT: the owner panel is stored in slabs of T rows (block A, block B);
    // (oso, olo) = slab and row in the slab of the owner being requested.
    uint32_t oso = 0, olo = 0;
    auto own_seek = [&](uint32_t o) {
        if constexpr (SPLIT) {
            oso = o / (uint32_t)a.T; olo = o - oso * (uint32_t)a.T;
        }
    };
    // storage unit (16 bytes) held by register unit c of this lane
    auto own_unit = [&](int c) -> int {
        if constexpr (SPLIT) {
            return c < SA ? (c ^ (l8 & (SA - 1))) : SA + (kRotB ? ((c - SA) ^ ((l8 >> 2) & 1)) : (c - SA));
        } else {
            return LPN * c + hf;
        }
    };
    // global address of storage unit u of owner o (SPLIT: of owner (oso, olo))
    auto own_src = [&](int64_t o, int u) -> const PT * {
        if constexpr (SPLIT) {
            const PT *blk = reinterpret_cast<const PT *>(a.owner) + (int64_t)oso * a.T * PSS;
            return u < SA ? blk + (int64_t)olo * (2 * SA) + u * UE
                          : blk + (int64_t)a.T * (2 * SA) + (int64_t)olo * BSD + (u - SA) * UE;
        } else {
            return reinterpret_cast<const PT *>(a.owner) + o * PS + u * UE;
        }
    };
    // request owner o into registers (modes 0, 1, 2); advances the running index
    auto load_owner = [&](uint32_t o, bool doit, PT(&dst)[KL]) {
        if (doit) {
            own_seek(o);
#pragma unroll
            for (int c = 0; c < NUL; c++) {
                const int u = own_unit(c);
                if (LPN == 1 || u < NU) ldg_unit(own_src(o, u), 0, dst + c * UE);
            }
        }
    };
    // mode 3: this group's staging slot behind the tile; stage_owner() copies the row into it with
    // cp.async (lane gl: units gl, gl + 8, ...), take_owner() waits for the copy and reads the
    // lane's units.  One slot is enough: the next copy is issued after every lane has read.
    constexpr int kStage = Cfg::stage_bytes(COLS, SPLIT);  // (per group, whatever G)
    const uint32_t stage_s = tile_s + tile_bytes + (uint32_t)gid * (uint32_t)kStage;
    auto stage_owner = [&](uint32_t o, bool doit) {
        if (doit) {
            own_seek(o);
#pragma unroll
            for (int u0 = 0; u0 < NU; u0 += G) {
                const int u = u0 + gl;
                if (u < NU)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(stage_s + u * 16),
                                 "l"(own_src(o, u)) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto take_owner = [&](PT(&dst)[KL]) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp(gmask);
#pragma unroll
        for (int c = 0; c < NUL; c++) {
            const int u = own_unit(c);
            if (LPN == 1 || u < NU) lds_unit(stage_s + u * 16, dst + c * UE);
        }
        __syncwarp(gmask);
    };
    // gather the tile row of packed entry v: this lane's units, in the order of its owner row
    auto gather = [&](uint32_t v, PT(&dst)[KL]) {
        if constexpr (SPLIT) {
            const uint32_t row = v & 0xffffu;
            const uint32_t ra = tileA_r + row * (uint32_t)(SA * 16);
            const uint32_t rb = tileB_r + row * (uint32_t)BSB;
#pragma unroll
            for (int c = 0; c < SA; c++) lds_unit(ra ^ (uint32_t)(c << 4), dst + c * UE);
#pragma unroll
            for (int c = 0; c < NUB; c++)
                lds_unit(kRotB ? (rb ^ (uint32_t)(c << 4)) : (rb + c * 16), dst + (SA + c) * UE);
        } else {
            const uint32_t raddr = tile_s + (v & 0xffffu) * (uint32_t)(PS * sizeof(PT));
#pragma unroll
            for (int c = 0; c < NUL; c++) {
                const int uu = LPN * c + hf;
                if (LPN == 1 || uu < NU) {
                    lds_unit(raddr + uu * 16, dst + c * UE);
                } else {
#pragma unroll
                    for (int j = 0; j < UE; j++) dst[c * UE + j] = 0;
                }
            }
        }
    };
    PT tr[KL];  // the gathered row; SPLIT: kept by hole entries (overwritten in full otherwise)
#pragma unroll
    for (int k = 0; k < KL; k++) tr[k] = 1;

    for (uint32_t ebase = e0; ebase < range_end;) {
        const uint32_t slab = ebase / NO;
        const uint32_t eend = min(range_end, (slab + 1) * NO);
        __syncthreads();
        if (threadIdx.x == 0) {
            mbar_expect_tx(&mbar, tile_bytes);
            bulk_g2s(tile, reinterpret_cast<const PT *>(a.tiles) + (int64_t)slab * a.T * PSS,
                     tile_bytes, &mbar);
        }
        // prime the group's pipeline while the tile lands: pointers and owners of its first two
        // segments, first quad and owner row of the first.  e runs over the POSITIONS of the
        // slab's segments in the stored order (a.seg[e] = owner row of position e): inside windows
        // of consecutive owners the segments are ordered by decreasing length, so that the four
        // groups of a warp, which run their chunk loops in lock step, get segments of (nearly
        // always) the same number of steps.
        uint32_t e = ebase + gid;
        // quad pointers of the current and the next segment; SPLIT: the start pointers carry the
        // number of all-hole steps at the end of their segment in the low 2 bits until it starts
        uint32_t beg = 0, end = 0, nb = 0, ne = 0;
        uint32_t og = 0, nog = 0;   // owner rows of the current and the next segment
        constexpr uint32_t kTag = SPLIT ? 3u : 0u;
        uint4 f0 = make_uint4(0u, 0u, 0u, 0u);
        PT ownn[KL];
#pragma unroll
        for (int k = 0; k < KL; k++) ownn[k] = 0;
        if (e < eend) {
            beg = __ldg(a.ptr4 + e);
            end = __ldg(a.ptr4 + e + 1) & ~kTag;
            og = __ldg(a.seg + e);
            if (e + kGroups < eend) {
                nb = __ldg(a.ptr4 + e + kGroups);
                ne = __ldg(a.ptr4 + e + kGroups + 1) & ~kTag;
                nog = __ldg(a.seg + e + kGroups);
            }
            const uint32_t b0 = beg & ~kTag;
            if (b0 + slot < end) f0 = ldcs_quad(ent4 + b0 + slot);
            if (kOwnMode == 1 || kOwnMode == 2) load_owner(og, b0 < end, ownn);
            if (kOwnMode == 3) stage_owner(og, b0 < end);
        }
        mbar_wait(&mbar, slab & 1u);
        while (e < eend) {
            const uint32_t en = e + kGroups;
            const uint32_t dead = beg & kTag;
            beg &= ~kTag;
            const uint32_t nbu = nb & ~kTag;
            const int nq = (int)(end - beg);
            const uint4 *eb = ent4 + beg;
            uint4 cur = f0;
            PT own[KL];
#pragma unroll
            for (int k = 0; k < KL; k++) own[k] = ownn[k];
            if (kOwnMode == 0) load_owner(og, nq > 0, own);
            if (kOwnMode == 3) {
                take_owner(own);   // (a segment without entries reads the previous row: unused)
                stage_owner(nog, en < eend && nbu < ne);
            }
            uint4 n1 = make_uint4(0u, 0u, 0u, 0u);
            if (NPG + slot < nq) n1 = ldcs_quad(eb + NPG + slot);
            // requests for the NEXT segment (pointers arrived during the previous one) and the
            // pointers of the one after it.  Mode 2: the next segment's first quad and the
            // pointers of the one after it are requested with its owner row, at the end of this
            // segment, instead of being held in registers through it (the first quad comes from
            // L2: the bulk prefetch includes it)
            constexpr uint32_t kPf = kOwnMode == 2 ? 0u : (uint32_t)NPG;  // first prefetched quad
            uint32_t nnb = 0, nne = 0, nnog = 0;
            auto load_ptrs = [&]() {
                if (en + kGroups < eend) {
                    nnb = __ldg(a.ptr4 + en + kGroups);
                    nne = __ldg(a.ptr4 + en + kGroups + 1) & ~kTag;
                    nnog = __ldg(a.seg + en + kGroups);
                }
            };
            if (kOwnMode != 2) f0 = make_uint4(0u, 0u, 0u, 0u);
            if (en < eend) {
                if (kOwnMode != 2) load_ptrs();
                if (kOwnMode != 2 && nbu + slot < ne) f0 = ldcs_quad(ent4 + nbu + slot);
                if (kOwnMode == 1) load_owner(nog, nbu < ne, ownn);
                if (gl == 0 && nbu + kPf < ne)
                    bulk_prefetch_l2(ent4 + nbu + kPf, (ne - nbu - kPf) * 16u);
            }
            PT acc[KL];
            PT xls = 0;
#pragma unroll
            for (int k = 0; k < KL; k++) acc[k] = 0;
            for (int c0 = 0; c0 < nq; c0 += NPG) {
                uint4 n2 = make_uint4(0u, 0u, 0u, 0u);
                if (c0 + 2 * NPG + slot < nq) n2 = ldcs_quad(eb + c0 + 2 * NPG + slot);
                PT pu[4], xu[4];   // fp32 cell-owner pass, LPN == 2
                // steps of this chunk that hold nonzeros (the last chunk of a segment may end in
                // all-hole steps)
                const int ulive = (SPLIT && VB_SKIP_DEAD && c0 + NPG >= nq) ? 4 - (int)dead : 4;
                // kLogProd: a count of the chunk has bits above the low kLpBits
                const bool big = ((cur.x | cur.y | cur.z | cur.w) >> (16 + kLpBits)) != 0u;
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    if (SPLIT && VB_SKIP_DEAD && u > 0 && u >= ulive) break;
                    const uint32_t v = u == 0 ? cur.x : u == 1 ? cur.y : u == 2 ? cur.z : cur.w;
                    const PT x = (PT)(int)(v >> 16);
                    // SPLIT: a hole keeps the previous row (no shared-memory traffic)
                    if (!SPLIT || !VB_SPLIT_PRED || (v >> 16)) gather(v, tr);
                    PT p = dot_rows<KL>(own, tr);
                    if (LPN == 2) p += __shfl_xor_sync(gmask, p, 1);
                    const PT q = x * rcp_t(p);
                    axpy_row<KL>(acc, tr, q);
                    if (kLogProd) {
                        // LPN == 2: both lanes of a pair hold p, each takes every other nonzero
                        if (LPN == 1 || (u & 1) == hf) lp.add(v, (double)p);
                    } else if (COLS) {
                        if (LPN == 1) xls = fma(x, log_t(p), xls);
                        else { pu[u] = p; xu[u] = x; }
                    }
                }
                if (kLogProd) lp.renorm();
                if (kLogProd && big) {
                    // (rare) the p of such a count is formed again from the tile row and the owner
                    // row, so that the steps keep nothing for it (both lanes of a pair hold the
                    // same entries and take this branch together)
                    const uint4 w = ldcs_quad(eb + c0 + slot);
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const uint32_t v = u == 0 ? w.x : u == 1 ? w.y : u == 2 ? w.z : w.w;
                        if (v >> (16 + kLpBits)) {
                            PT t[KL];
                            gather(v, t);
                            PT p = dot_rows<KL>(own, t);
                            if (LPN == 2) p += __shfl_xor_sync(pmask, p, 1);
                            if (LPN == 1 || (u & 1) == hf) lp.add_slow(v, (double)p);
                        }
                    }
                }
                if (COLS && !kLogProd && LPN == 2) {
#pragma unroll
                    for (int v = 0; v < 2; v++) {
                        const PT pm = hf ? pu[2 * v + 1] : pu[2 * v];
                        const PT xm = hf ? xu[2 * v + 1] : xu[2 * v];
                        xls = fma(xm, log_t(pm), xls);
                    }
                }
                cur = n1;
                n1 = n2;
            }
            if (kLogProd) lp.end_segment();
            else if (COLS) xl += (double)xls;
            if (kOwnMode == 2) {
                f0 = make_uint4(0u, 0u, 0u, 0u);
                if (en < eend) {
                    load_ptrs();
                    load_owner(nog, nbu < ne, ownn);
                    if (nbu + slot < ne) f0 = ldcs_quad(ent4 + nbu + slot);
                }
            }
            // sum over the lanes that hold the same rank entries (fp64), recursive halving
            double *out = a.Part + (int64_t)(slab * NO + og) * RS;
            double v0[KL];
#pragma unroll
            for (int k = 0; k < KL; k++) v0[k] = (double)acc[k];
            if constexpr (SPLIT) {
                // block A: register unit c of lane gl is rank unit c ^ (gl & (SA - 1)); the partner
                // gl ^ b holds the same rank unit in its register unit c ^ b
                if constexpr (SA == 8 && G == 4) {
                    // four lanes: register unit c of lane l8 is rank unit c ^ l8; halve over bits 1
                    // and 0 of the lane; the lane ends with rank units l8 and l8 ^ 4
                    double a1[8], a2[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {       // keep register units 0, 1, 4, 5
                        const int c = (u & 1) | ((u & 2) << 1);
#pragma unroll
                        for (int j = 0; j < 2; j++)
                            a1[2 * u + j] = v0[2 * c + j] + __shfl_xor_sync(gmask, v0[2 * (c ^ 2) + j], 2);
                    }
#pragma unroll
                    for (int u = 0; u < 2; u++) {       // keep register units 0, 4 (a1 units 0, 2)
#pragma unroll
                        for (int j = 0; j < 2; j++)
                            a2[2 * u + j] = a1[4 * u + j] + __shfl_xor_sync(gmask, a1[4 * u + 2 + j], 1);
                    }
                    *reinterpret_cast<double2 *>(out + 2 * l8) = make_double2(a2[0], a2[1]);
                    *reinterpret_cast<double2 *>(out + 2 * (l8 ^ 4)) = make_double2(a2[2], a2[3]);
                } else if constexpr (SA == 8) {
                    double a1[8], a2[4], a3[2];
#pragma unroll
                    for (int k = 0; k < 8; k++) a1[k] = v0[k] + __shfl_xor_sync(gmask, v0[k + 8], 4);
#pragma unroll
                    for (int k = 0; k < 4; k++) a2[k] = a1[k] + __shfl_xor_sync(gmask, a1[k + 4], 2);
#pragma unroll
                    for (int k = 0; k < 2; k++) a3[k] = a2[k] + __shfl_xor_sync(gmask, a2[k + 2], 1);
                    *reinterpret_cast<double2 *>(out + 2 * gl) = make_double2(a3[0], a3[1]);
                } else {
                    // SA == 4: halve over the four rotations, then add the two parity halves
                    double a1[4], a2[2];
#pragma unroll
                    for (int k = 0; k < 4; k++) a1[k] = v0[k] + __shfl_xor_sync(gmask, v0[k + 4], 2);
#pragma unroll
                    for (int k = 0; k < 2; k++) a2[k] = a1[k] + __shfl_xor_sync(gmask, a1[k + 2], 1);
#pragma unroll
                    for (int k = 0; k < 2; k++) a2[k] += __shfl_xor_sync(gmask, a2[k], 4);
                    if (gl < 4 && 2 * gl < RP)
                        *reinterpret_cast<double2 *>(out + 2 * gl) = make_double2(a2[0], a2[1]);
                }
                if constexpr (kRotB && G == 4) {
                    // all four lanes hold rank unit 8 + (c ^ h) in register unit c (h = bit 2 of
                    // l8 is the same for the group): plain halving of the four doubles
                    const int h = (l8 >> 2) & 1;
                    const bool hi1 = (gl & 2) != 0, hi0 = (gl & 1) != 0;
                    double b1[2];
#pragma unroll
                    for (int j = 0; j < 2; j++) {
                        const double keep = hi1 ? v0[2 * SA + 2 + j] : v0[2 * SA + j];
                        const double send = hi1 ? v0[2 * SA + j] : v0[2 * SA + 2 + j];
                        b1[j] = keep + __shfl_xor_sync(gmask, send, 2);
                    }
                    const double b2 = (hi0 ? b1[1] : b1[0]) + __shfl_xor_sync(gmask, hi0 ? b1[0] : b1[1], 1);
                    // register unit (bit 1 of gl) -> rank unit 8 + (that ^ h), double (bit 0 of gl)
                    const int kk = 2 * SA + 2 * ((hi1 ? 1 : 0) ^ h) + (hi0 ? 1 : 0);
                    if (kk < RP) out[kk] = b2;
                } else if constexpr (kRotB) {
                    // register unit c of lane gl is rank unit 8 + (c ^ h), h = bit 2 of gl: the
                    // partner gl ^ 4 holds my unit of register 0 in its register 1; then the four
                    // lanes of equal h hold the same unit and halve its two doubles
                    double b1[2];
#pragma unroll
                    for (int k = 0; k < 2; k++)
                        b1[k] = v0[2 * SA + k] + __shfl_xor_sync(gmask, v0[2 * SA + 2 + k], 4);
                    const bool hi2 = (gl & 2) != 0;
                    double b2 = (hi2 ? b1[1] : b1[0]) + __shfl_xor_sync(gmask, hi2 ? b1[0] : b1[1], 2);
                    b2 += __shfl_xor_sync(gmask, b2, 1);
                    // lane gl: rank entry 16 + 2 * h + (bit 1 of gl)
                    const int kk = 2 * SA + 2 * ((gl >> 2) & 1) + ((gl >> 1) & 1);
                    if ((gl & 1) == 0 && kk < RP) out[kk] = b2;
                } else if constexpr (NUB > 0 && G == 4) {
                    // (VB_G4_NU9) a plain unit of block B over four lanes
#pragma unroll
                    for (int k = 0; k < 2 * NUB; k++) {
                        double sB = v0[2 * SA + k];
                        sB += __shfl_xor_sync(gmask, sB, 2);
                        sB += __shfl_xor_sync(gmask, sB, 1);
                        if (gl == (k & 3) && 2 * SA + k < RP) out[2 * SA + k] = sB;
                    }
                } else if constexpr (NUB > 0) {
                    double vb[2 * NUB];
#pragma unroll
                    for (int k = 0; k < 2 * NUB; k++) vb[k] = v0[2 * SA + k];
                    halve_reduce_store<2 * NUB>(vb, gl, gmask, out + 2 * SA, RP - 2 * SA);
                }
            } else {
            constexpr int H1 = (KL + 1) / 2, H2 = (H1 + 1) / 2, H3 = (H2 + 1) / 2;
            double v1[H1], v2[H2];
            halve_step<KL, 4>(v0, v1, gl, gmask);
            halve_step<H1, 2>(v1, v2, gl, gmask);
            const int o1 = (gl & 4) ? H1 : 0, o2 = (gl & 2) ? H2 : 0;
            if (LPN == 1) {
                double v3[H3];
                halve_step<H2, 1>(v2, v3, gl, gmask);
                const int o3 = (gl & 1) ? H3 : 0;
#pragma unroll
                for (int k = 0; k < H3; k++) {
                    const int i2 = k + o3, i1 = i2 + o2, i0 = i1 + o1;  // entry index in acc[]
                    if (i2 < H2 && i1 < H1 && i0 < KL && i0 < RP) out[i0] = v3[k];
                }
            } else {
#pragma unroll
                for (int k = 0; k < H2; k++) {
                    const int i1 = k + o2, i0 = i1 + o1;
                    const int kk = (LPN * (i0 / UE) + hf) * UE + (i0 % UE);  // rank index
                    if (i1 < H1 && i0 < KL && kk < RP) out[kk] = v2[k];
                }
            }
            }
            e = en;
            beg = nb; end = ne; og = nog;
            nb = nnb; ne = nne; nog = nnog;
        }
        ebase = eend;
    }
    if (COLS) {
        if (kLogProd) xl = lp.total();
        xl = block_sum(xl, red);
        if (threadIdx.x == 0) a.xl_part[blockIdx.x] = xl;
    }
}

// ------------------------------------------------------------------------------------------
// Combine the per-slab partial statistics of a sweep pass in slab order and take the entropy-
// collapse term of the bound in the same pass (src/vbnmf_update.cpp:69-77):
//   SRaw[o][k] = sum_slab Part[slab][o][k];   out[0] = sum_{o,k<r} log(l_ok) l_ok SRaw[o][k]
// rows beyond the valid owners (layout padding) hold zeros in l and are skipped.
template <int RP>
__global__ void __launch_bounds__(kBlock)
combine_kernel(int64_t NO, int nslabs, int r, const double *__restrict__ Part,
               const double *__restrict__ l, double *__restrict__ SRaw, double *__restrict__ part,
               double *__restrict__ out, unsigned *counter, const double *__restrict__ xl_part,
               int nxl, const double *__restrict__ ctl, int tsplit) {
    constexpr int RS = row_stride(RP);
    __shared__ double sm[kWarpsPerBlock];
    if (ctl && ctl[kCtlDone] != 0.0) return;
    double ent = 0.0;
    const int64_t tot = NO * (RS / 2);
    for (int64_t u = (int64_t)blockIdx.x * kBlock + threadIdx.x; u < tot;
         u += (int64_t)gridDim.x * kBlock) {
        const int64_t o = u / (RS / 2);
        const int k2 = (int)(u - o * (RS / 2)) * 2;
        double2 s = make_double2(0.0, 0.0);
        for (int sl = 0; sl < nslabs; sl++) {
            const double2 v =
                __ldcs(reinterpret_cast<const double2 *>(Part + ((int64_t)sl * NO + o) * RS + k2));
            s.x += v.x;
            s.y += v.y;
        }
        if (k2 >= RP) s = make_double2(0.0, 0.0);
        *reinterpret_cast<double2 *>(SRaw + o * RS + k2) = s;
        // (a row of the split layout ends at RP: the padding columns of SRaw have no l)
        const double2 lv = k2 < RP ? *reinterpret_cast<const double2 *>(l + panel_ofs(o, k2, RS, tsplit))
                                   : make_double2(0.0, 0.0);
        if (k2 < r && lv.x > 0.0) ent += log(lv.x) * lv.x * s.x;
        if (k2 + 1 < r && lv.y > 0.0) ent += log(lv.y) * lv.y * s.y;
    }
    // per-CTA partial sums of x log p from the sweep ride along (out[1])
    double xl = 0.0;
    for (int i = blockIdx.x * kBlock + threadIdx.x; i < nxl; i += gridDim.x * kBlock)
        xl += xl_part[i];
    ent = block_sum(ent, sm);
    xl = block_sum(xl, sm);
    if (threadIdx.x == 0) {
        part[blockIdx.x * 2 + 0] = ent;
        part[blockIdx.x * 2 + 1] = xl;
    }
    last_block_reduce(part, 2, out, counter, sm);
}

// ------------------------------------------------------------------------------------------
// Posterior update of one side (W: rows = genes, H: rows = cells); identical algebra:
//   al = a + l o SRaw                                     src/vbnmf_update.cpp:38-39 / 48-49
//   be_k = a/b + osum_k   (osum = rowSums(eh_old) for W, colSums(ew_new) for H)   :40-43 / 50-53
//   e = al / be_k                                                                :44 / 54
//   l_new = max(exp(psi(al)) / be_k, fud)                                        :58-65
// and the reductions the bound and hyper_update need:
//   out[0..RS)   : sum over rows of e  (colSums(ew) / rowSums(eh))
//   out[RS+0]    : sum [ -(a/b) e + al (1 - log be_k) + lgamma(al) ]   (:84-86 / :88-89; the
//                  constant lga term is added on the host)
//   out[RS+1]    : sum log l_new                                       (R/bayesian.R:8-9)
//   out[RS+2]    : sum e                                               (R/bayesian.R:10-11)
// One thread per panel row.  Rows are in device order: row d = slab*T + local holds the item at
// sorted position local*S + slab, valid when that is < nvalid.  al is kept for ew/dw (eh/dh).
// Thread mapping: a CTA of kPostLanes * RS threads covers kPostRows consecutive panel rows; thread
// t always works on rank entry k = t % RS (so its be_k, log be_k and partial sums live in
// registers) of rows t / RS, t / RS + kPostLanes, ...  Loads and stores are fully coalesced and a
// panel of N rows exposes N * RS-way parallelism (the special functions dominate this kernel).
constexpr int kPostRows = 96;   // rows per CTA (posterior_kernel: at most; see post_rows_per_cta)
__host__ __device__ constexpr int post_lanes(int rs) {   // rows in flight per CTA
    return (1024 / rs) < 24 ? (1024 / rs) : 24;
}
__host__ __device__ constexpr int post_threads(int rs) {  // padded to whole warps
    return ((post_lanes(rs) * rs + 31) / 32) * 32;
}

// rows per CTA of posterior_kernel: kPostRows for large panels; small panels (the special
// functions of a row cost microseconds) are spread over about two CTAs per SM
__host__ __device__ inline int post_rows_per_cta(int64_t rows, int rs, int num_sms) {
    const int lanes = post_lanes(rs);
    const int64_t per = (rows + 2 * (int64_t)num_sms * lanes - 1) / (2 * (int64_t)num_sms * lanes);
    const int64_t r = per * lanes;
    return (int)(r < kPostRows ? (r < lanes ? lanes : r) : kPostRows);
}

template <int RP>
__global__ void __launch_bounds__(post_threads(row_stride(RP)))
posterior_kernel(int64_t rows, int T, int S, int64_t nvalid, int r, double a, double b, double fud,
                 const double *__restrict__ osum, const double *__restrict__ SRaw,
                 double *__restrict__ l, double *__restrict__ al_out, double *__restrict__ part,
                 double *__restrict__ out, unsigned *counter, float *__restrict__ l32,
                 const double *__restrict__ ctl, int hoff, int rows_per_cta, int tsplit) {
    constexpr int RS = row_stride(RP);
    constexpr int kPostLanes = post_lanes(RS);
    constexpr int NT = post_threads(RS);
    constexpr int W = RS + 3;
    if (ctl) {  // device-controlled loop: stop flag and the current hyper-parameters live on the GPU
        if (ctl[kCtlDone] != 0.0) return;
        a = ctl[kCtlHyper + hoff];
        b = ctl[kCtlHyper + hoff + 1];
    }
    __shared__ double sm[NT / 32];
    __shared__ double colbuf[4][NT];
    const int k = threadIdx.x % RS, lane_row = threadIdx.x / RS;  // lane_row >= kPostLanes: idle
    const bool kact = k < r;
    const double be = kact ? a / b + osum[k] : 1.0;
    const double lbe = log(be), aob = a / b;
    double es = 0.0, prior = 0.0, sll = 0.0;
    const int64_t row0 = (int64_t)blockIdx.x * rows_per_cta;
#pragma unroll 1
    for (int i = lane_row; i < rows_per_cta && lane_row < kPostLanes; i += kPostLanes) {
        const int64_t row = row0 + i;
        if (row >= rows) break;
        const int64_t slab = row / T, local = row - slab * T;
        const bool valid = local * S + slab < nvalid;
        double ln = 0.0, al = 0.0;
        const int64_t lo = panel_ofs(row, k, RS, tsplit);
        if (valid && kact) {
            al = a + l[lo] * SRaw[row * RS + k];
            const double e = al / be;
            double psi_al, lg_al;
            vb_psi_lgamma(al, &psi_al, &lg_al);
            const double tmp = exp(psi_al) / be;
            ln = tmp > fud ? tmp : fud;
            es += e;
            sll += log(ln);
            prior += -aob * e + al * (1.0 - lbe) + lg_al;
        }
        if (valid) {
            if (k < RP || tsplit == 0) l[lo] = ln;  // a row of the split layout ends at RP
            al_out[row * RS + k] = al;
            if (l32 && k < row_stride_f32(RP)) l32[row * row_stride_f32(RP) + k] = (float)ln;
        }
    }
    // per-rank-entry sums over the CTA's rows, in fixed order; then the three scalars
    colbuf[0][threadIdx.x] = es;
    colbuf[1][threadIdx.x] = prior;
    colbuf[2][threadIdx.x] = sll;
    __syncthreads();
    double *mypart = part + (size_t)blockIdx.x * W;
    if (threadIdx.x < RS) {
        double s0 = 0.0, s1 = 0.0, s2 = 0.0;
        for (int j = 0; j < kPostLanes; j++) {
            s0 += colbuf[0][threadIdx.x + j * RS];
            s1 += colbuf[1][threadIdx.x + j * RS];
            s2 += colbuf[2][threadIdx.x + j * RS];
        }
        mypart[threadIdx.x] = s0;
        colbuf[3][threadIdx.x] = s0;
        colbuf[1][threadIdx.x] = s1;
        colbuf[2][threadIdx.x] = s2;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double p = 0.0, q = 0.0, e = 0.0;
        for (int j = 0; j < RS; j++) { p += colbuf[1][j]; q += colbuf[2][j]; e += colbuf[3][j]; }
        mypart[RS + 0] = p;
        mypart[RS + 1] = q;
        mypart[RS + 2] = e;
    }
    last_block_reduce(part, W, out, counter, sm);
}

// ---- maximum-likelihood multiplicative updates (R/factorize.R:8-15 for h, :17-24 for w) ----
//   v_new = max(v o SRaw / osum_k, eps);  out[0..RS) = sum over rows of v_new
template <int RP>
__global__ void __launch_bounds__(post_threads(row_stride(RP)))
ml_update_kernel(int64_t rows, int T, int S, int64_t nvalid, int r, double eps,
                 const double *__restrict__ osum, const double *__restrict__ SRaw,
                 double *__restrict__ v, double *__restrict__ part, double *__restrict__ out,
                 unsigned *counter, float *__restrict__ l32, int tsplit,
                 const double *__restrict__ ctl) {
    constexpr int RS = row_stride(RP);
    constexpr int kPostLanes = post_lanes(RS);
    constexpr int NT = post_threads(RS);
    __shared__ double sm[NT / 32];
    __shared__ double colbuf[NT];
    if (ctl && ctl[kCtlDone] != 0.0) return;  // device-controlled loop: the run has ended
    const int k = threadIdx.x % RS, lane_row = threadIdx.x / RS;
    const bool kact = k < r;
    const double os = kact ? osum[k] : 1.0;
    double es = 0.0;
    const int64_t row0 = (int64_t)blockIdx.x * kPostRows;
#pragma unroll 1
    for (int i = lane_row; i < kPostRows && lane_row < kPostLanes; i += kPostLanes) {
        const int64_t row = row0 + i;
        if (row >= rows) break;
        const int64_t slab = row / T, local = row - slab * T;
        if (local * S + slab >= nvalid) continue;
        double x = 0.0;
        const int64_t lo = panel_ofs(row, k, RS, tsplit);
        if (kact) {
            x = v[lo] * SRaw[row * RS + k] / os;
            if (x < eps) x = eps;
            es += x;
        }
        if (k < RP || tsplit == 0) v[lo] = x;  // a row of the split layout ends at RP
        if (l32 && k < row_stride_f32(RP)) l32[row * row_stride_f32(RP) + k] = (float)x;
    }
    colbuf[threadIdx.x] = es;
    __syncthreads();
    if (threadIdx.x < RS) {
        double s0 = 0.0;
        for (int j = 0; j < kPostLanes; j++) s0 += colbuf[threadIdx.x + j * RS];
        part[(size_t)blockIdx.x * RS + threadIdx.x] = s0;
    }
    last_block_reduce(part, RS, out, counter, sm);
}

// fp32 mirror of a rows x RS panel (after set_state in VBNMF_FP32_STORAGE mode)
template <int RP>
__global__ void __launch_bounds__(kBlock)
mirror_kernel(int64_t rows, const double *__restrict__ v, float *__restrict__ v32) {
    const int64_t row = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (row >= rows) return;
#pragma unroll
    for (int k = 0; k < row_stride_f32(RP); k++)
        v32[row * row_stride_f32(RP) + k] = k < RP ? (float)v[row * row_stride(RP) + k] : 0.f;
}

// column sums of a rows x RS panel (padding rows hold zeros): out[k] = sum_row v[row][k]
template <int RP>
__global__ void __launch_bounds__(kBlock)
panel_colsum_kernel(int64_t rows, const double *__restrict__ v, double *__restrict__ part,
                    double *__restrict__ out, unsigned *counter, int tsplit) {
    constexpr int RS = row_stride(RP);
    __shared__ double sm[kWarpsPerBlock];
    const int64_t row = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    double lv[RP];
#pragma unroll
    for (int k = 0; k < RP; k++) lv[k] = 0.0;
    if (row < rows) {
#pragma unroll
        for (int k = 0; k < RP; k += 2) {
            const double2 t = __ldg(reinterpret_cast<const double2 *>(v + panel_ofs(row, k, RS, tsplit)));
            lv[k] = t.x;
            lv[k + 1] = t.y;
        }
    }
    double *mypart = part + (size_t)blockIdx.x * RS;
#pragma unroll
    for (int k = 0; k < RP; k++) {
        const double s = block_sum(lv[k], sm);
        if (threadIdx.x == 0) mypart[k] = s;
    }
    if (threadIdx.x == 0)
        for (int k = RP; k < RS; k++) mypart[k] = 0.0;
    last_block_reduce(part, RS, out, counter, sm);
}

}  // namespace vb
