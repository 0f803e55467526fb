// libvbnmf: host side of the B200-native VB Poisson-NMF engine and its C ABI (include/vbnmf.h).
//
// Replaces, for ccfindR's vb_factorize() path, the Rcpp step src/vbnmf_update.cpp:16-102 and the
// iteration loop R/bayesian.R:336-352 that calls it (plus hyper_update, R/bayesian.R:2-53), and
// for factorize() the loop R/factorize.R:189-212.  No CPU fallback: every entry point needs the
// CUDA device the handle was created on.
//
// Device data layout (DESIGN.md has the picture):
//   * genes and cells are renumbered: sorted by nonzero count (descending) and dealt round-robin
//     over S = ceil(count / T) slabs of T rows, device row = slab * T + local.  Slabs therefore
//     hold the same mix of dense and sparse rows, and neighbouring rows have similar lengths.
//   * panels lw, alw, SwRaw are (Sg*T) x RS, lh, alh, ShRaw are (Sc*T) x RS, row-major with the
//     rank index fastest; RS = row_stride(RP) doubles, padding rows/columns are zero.
//   * the count matrix is stored twice, once per sweep pass, slab-major in segments
//     (tile slab, owner row); see kernels.cuh sweep_tiled_kernel.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <time.h>

#include <algorithm>
#include <cmath>
#include <cub/cub.cuh>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <memory>
#include <numeric>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/vbnmf.h"
#include "kernels_common.cuh"
#include "svd_init.cuh"
#include "mtx_ingest.cuh"
#include "qc.cuh"
#include "shuffle.cuh"
#include "consensus.cuh"
#include "rp_ranks.h"
#include "rp_table.h"

namespace vb {
#define F(RP) extern const RpTable rp_table_##RP;
VB_RP_LIST(F)
#undef F
const RpTable *rp_table(int rp) {
    switch (rp) {
#define F(RP) \
    case RP:  \
        return &rp_table_##RP;
        VB_RP_LIST(F)
#undef F
    }
    return nullptr;
}
}  // namespace vb

namespace {

constexpr int kMaxRank = 64;
constexpr int64_t kGraphMaxNnz = 20000000;  // below this the iteration loop is replayed as a CUDA graph
// shared-memory budget of one staged slab: the 227 KB a CTA can opt in to minus the static part
constexpr int kTileBytes = 231424;
constexpr int kTileRowsMax = 4096, kTileRowsStep = 32;
constexpr int kSegWindow = 4096;  // owners per window of the length-sorted segment order (build_pass)
constexpr double kSplitKappa = 0.0;  // cost of a segment beyond its entries, in quads (split_p16_kernel)

thread_local std::string g_create_error;  // error text of the last failed create on this thread

// NVTX range around a phase of the iteration (visible in Nsight tools; header-only, no cost
// without a profiler attached)
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

// VBNMF_TIMING=1 prints host-side stage times (setup paths only) to stderr
struct StageTimer {
    const char *name;
    bool on;
    timespec t0;
    explicit StageTimer(const char *n) : name(n), on(getenv("VBNMF_TIMING") != nullptr) {
        if (on) clock_gettime(CLOCK_MONOTONIC, &t0);
    }
    ~StageTimer() {
        if (!on) return;
        cudaDeviceSynchronize();
        timespec t1;
        clock_gettime(CLOCK_MONOTONIC, &t1);
        fprintf(stderr, "[vbnmf] %-28s %8.2f ms\n", name,
                (t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6);
    }
};

struct NcclApi {
    void *lib = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    bool load(std::string &err) {
        if (lib) return true;
        // libnccl.so.2 resolves to the copy already mapped by the host process (e.g. torch's) if any
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) { err = std::string("cannot load libnccl: ") + dlerror(); return false; }
        GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
        AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
        AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
        CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
        GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy) {
            err = "libnccl lacks a required symbol";
            return false;
        }
        return true;
    }
};
NcclApi g_nccl;

// one pass of the tiled count-matrix layout
struct PassLayout {
    int64_t E = 0;              // segments = tile slabs * owners
    int64_t nent = 0;           // entries stored (nonzeros, plus the schedule holes of packed-16)
    int64_t *d_ptr = nullptr;   // E + 1
    int32_t *d_idx = nullptr;   // nnz (double counts only)
    void *d_val = nullptr;      // nnz (double counts only)
    void *d_ent = nullptr;      // nnz packed {int32 tile row, float count} (float counts), or
                                // the padded {count << 16 | tile row} words of the packed-16 layout
    uint32_t *d_ptr4 = nullptr; // packed-16 layout: E + 1 segment pointers in quads (16 bytes),
                                // indexed by the POSITION of a segment in the stored order
    uint32_t *d_seg = nullptr;  // packed-16 layout: owner row of position pos (inside windows of
                                // kSegWindow owners the segments are stored by decreasing length)
    int64_t *d_split = nullptr; // grid + 1
    void release(cudaStream_t s) {
        void *ps[] = {d_ptr, d_idx, d_val, d_ent, d_ptr4, d_seg, d_split};
        for (void *q : ps)
            if (q) cudaFreeAsync(q, s);
        d_ptr = nullptr; d_idx = nullptr; d_val = nullptr; d_ent = nullptr; d_ptr4 = nullptr;
        d_seg = nullptr; d_split = nullptr;
    }
};

// tiled layout for tile height T (cached per T; the rank only enters through T)
struct Layout {
    int T = 0, Sg = 0, Sc = 0;
    int npg = 0;  // packed-16 layout: nonzeros per group step it was ordered for (0: 8-byte layout)
    int kmult = 4;  // packed-16 layout: the schedule's step count is a multiple of this (4 or 1)
    int mode = 0;  // packed-16 layout: schedule mode (vb::kSchedPlain / kSchedSbs / kSchedCls4)
    int64_t NG = 0, NC = 0;
    int32_t *d_gene_dev = nullptr, *d_cell_dev = nullptr;  // original index -> device row
    PassLayout cols, rows;
    int grid = 0;
    void release(cudaStream_t s) {
        cols.release(s); rows.release(s);
        if (d_gene_dev) cudaFreeAsync(d_gene_dev, s);
        if (d_cell_dev) cudaFreeAsync(d_cell_dev, s);
        d_gene_dev = d_cell_dev = nullptr;
    }
};

}  // namespace

struct vbnmf_comm {
    int nranks = 1, rank = 0, device = 0;
    ncclComm_t comm = nullptr;
};

struct vbnmf_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int num_sms = 148;
    int64_t n = 0, m = 0, nnz = 0, m_global = 0, nnz_global = 0;
    int r = 0, rp = 0, rs = 0;
    int precision = VBNMF_FP64;
    bool val_float = true;
    bool p16 = false;  // all counts are integers < 2^16: packed-16 layouts (sweep_p16_kernel)
    bool borrowed = false;
    // Scratch arena of the first layout build (5 * nnz 32-bit words), reserved when the handle is
    // created, BEFORE the smaller GB-sized buffers: the memory pool then hands the same blocks to
    // the same requests at every handle creation instead of splitting the big block and mapping
    // new memory for the arena later (tens of ms, varying from run to run).
    uint32_t *d_arena = nullptr;
    // the count matrix as given (CSC); the tiled layouts are derived from it
    int64_t *d_colptr = nullptr;
    int32_t *d_rowidx = nullptr;
    void *d_val = nullptr;
    // entries with a non-zero value per gene (n) and per cell (m); the gene counts are global once
    // the cells are sharded (vbnmf_attach_comm)
    unsigned long long *d_cnt = nullptr;
    bool colof_in_arena = false;  // d_arena[0, nnz) holds the column of every entry (scan_matrix)
    int64_t empty_rows = 0, empty_cols = 0;
    std::vector<Layout *> layouts;
    Layout *L = nullptr;
    const vb::RpTable *tab = nullptr;
    int smem_bytes = 0;
    // panels in device order
    double *d_lw = nullptr, *d_lh = nullptr, *d_alw = nullptr, *d_alh = nullptr;
    float *d_lw32 = nullptr, *d_lh32 = nullptr;  // fp32 mirrors read by the sweep (fp32-storage mode)
    int rsf = 0, panel_precision = -1;
    int split_kind = 0;  // 0 plain rows, 1 split layout, 2 split layout + 4-lane groups (rp_table.h)
    int tsplit = 0;  // layout of d_lw / d_lh: 0 row-major, else the tile height T of the split
                     // layout (kernels.cuh panel_ofs) read by the split variant of the p16 sweep
    // d_red = [SwRaw NG*rs | ehsum rs | hprior, sumloglh, sumeh | enth, xlogp | entw, - | pad]
    double *d_red = nullptr;
    double *d_ShRaw = nullptr, *d_Part1 = nullptr, *d_Part2 = nullptr, *d_xl = nullptr;
    double *d_scal = nullptr;  // [ewsum rs | wprior, sumloglw, sumew | pad]
    double *h_scal = nullptr;  // pinned mirror: [d_scal (rs+8) | tail of d_red (rs+8)]
    double *d_partW = nullptr, *d_partH = nullptr, *d_partC = nullptr;
    unsigned *d_counters = nullptr;
    double *d_ctl = nullptr, *h_ctl = nullptr;  // device loop control block and its pinned mirror
    const double *ctl = nullptr;                // = d_ctl while a device-controlled loop is running
    int gridC = 0;
    double lgx = 0.0, mlconst = 0.0;  // global sums over nonzeros
    // host copies of the small vectors
    double ehsum[kMaxRank], ewsum[kMaxRank], bew[kMaxRank], beh[kMaxRank];
    double wacc[3], hacc[3], xlogp = 0, enth = 0, entw = 0;
    bool stats_valid = false, has_posterior = false;
    // NCCL
    int nranks = 1, rank = 0;
    ncclComm_t comm = nullptr;
    // exchange region of the peer-memory all-reduce (kernels_common.cuh): own allocation, the
    // peers' regions mapped through CUDA IPC, sequence number of the last all-reduce
    unsigned long long *d_xchg = nullptr;
    unsigned long long *xchg_peer[vb::kXchgFlags] = {};
    int64_t xchg_stride = 0;
    unsigned long long xchg_seq = 0;
    bool peer_ok = false;
    int64_t launches = 0;
    std::string err;
};

namespace {

using H = vbnmf_handle;

#define CK(call)                                                                         \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                 \
            return VBNMF_ERR_CUDA;                                                       \
        }                                                                                \
    } while (0)

#define CKN(call)                                                                        \
    do {                                                                                 \
        ncclResult_t e_ = (call);                                                        \
        if (e_ != ncclSuccess) {                                                         \
            h->err = std::string(#call) + ": " +                                         \
                     (g_nccl.GetErrorString ? g_nccl.GetErrorString(e_) : "nccl error"); \
            return VBNMF_ERR_NCCL;                                                       \
        }                                                                                \
    } while (0)

int fail(H *h, int code, const std::string &msg) {
    h->err = msg;
    return code;
}
int check_rank(H *h, int r) {
    return r < 1 || r > kMaxRank ? fail(h, VBNMF_ERR_ARG, "rank must be in 1..64") : 0;
}
int check_state(H *h) {
    return h->d_lw ? 0 : fail(h, VBNMF_ERR_STATE, "vbnmf_set_state has not been called");
}

// Device memory comes from the stream-ordered pool (cudaMallocAsync) with a high release
// threshold: the many GB-sized buffers of a handle are recycled instead of being mapped and
// unmapped by the driver at every create/destroy (which cost more than the factorization itself).
template <typename T>
cudaError_t vmalloc(H *h, T **p, size_t bytes) {
    return cudaMallocAsync((void **)p, bytes ? bytes : 16, h->stream);
}
inline void vfree(cudaStream_t s, void *p) {
    if (p) cudaFreeAsync(p, s);
}

// Scratch device memory of one scope: every buffer taken with get() is freed (stream-ordered)
// when the scope ends, on every return path.  free() returns one earlier, where keeping it until
// the end would raise the peak; keep() hands one over to an owner that outlives the scope.
struct ScopedBufs {
    H *h;
    cudaStream_t s;
    std::vector<void *> p;
    explicit ScopedBufs(H *h_) : h(h_), s(h_->stream) {}
    ScopedBufs(const ScopedBufs &) = delete;
    ScopedBufs &operator=(const ScopedBufs &) = delete;
    ~ScopedBufs() { for (void *q : p) vfree(s, q); }
    template <typename T>
    cudaError_t get(T **x, size_t bytes) {
        *x = nullptr;
        const cudaError_t e = vmalloc(h, x, bytes);
        if (e == cudaSuccess) p.push_back((void *)*x);
        return e;
    }
    void hold(void *x) { p.push_back(x); }  // x (allocated elsewhere) is freed with the scope
    template <typename T>
    void free(T *&x) {
        vfree(s, keep(x));
        x = nullptr;
    }
    template <typename T>
    T *keep(T *x) {
        p.erase(std::remove(p.begin(), p.end(), (void *)x), p.end());
        return x;
    }
};

// A device-controlled loop: while this lives the kernels read the stop flag and the hypers from the
// control block (h->d_ctl); the host-controlled mode is restored on every exit path.
struct DeviceControl {
    H *h;
    explicit DeviceControl(H *h_) : h(h_) { h->ctl = h->d_ctl; }
    ~DeviceControl() { h->ctl = nullptr; }
};

// f(float()) or f(double()): the stored type of the counts as a template argument
template <typename F>
auto with_val_type(bool as_float, F &&f) {
    return as_float ? f(float()) : f(double());
}

inline cudaError_t copy_sync(H *h, void *dst, const void *src, size_t bytes, cudaMemcpyKind kind) {
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, h->stream);
    return e != cudaSuccess ? e : cudaStreamSynchronize(h->stream);
}

inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
inline int pad_rank(int r) {
    int rp = (r + 1) & ~1;
    if (rp < 2) rp = 2;
    if (rp > 32) rp = (rp + 7) & ~7;
    return rp;
}
inline int64_t tail_off(const H *h) { return h->L->NG * h->rs; }
inline int64_t red_len(const H *h) { return h->L->NG * h->rs + h->rs + 8; }

int choose_tile_rows(const H *h, int row_bytes, int stage_bytes) {
    // largest multiple of 32 rows that fits beside the owner staging slots of the packed-16 sweeps
    // (ranks with the same row stride share a layout)
    int T = ((kTileBytes - stage_bytes) / row_bytes / kTileRowsStep) * kTileRowsStep;
    T = std::max(kTileRowsStep, std::min(T, kTileRowsMax));
    // every rank of a sharded factorization must arrive at the same T (the gene panels are
    // all-reduced in device order): only global quantities enter
    const int64_t big = std::max(h->n, h->m_global);
    const int64_t cap = std::max<int64_t>(128, ((big + 127) / 128) * 128);
    T = (int)std::min<int64_t>(T, cap);
    // Small problems: the largest tile leaves too few segments to occupy the 148 x 64 eight-lane
    // groups (a pass over the 1,000 x 200 plumbing case is 200 segments).  Shrink the tile until a
    // pass has about four segments per group, but keep ~40 nonzeros per segment (below that the
    // per-segment overhead wins).  Measured: 1,000 x 200 r=3 0.072 -> 0.059 ms per iteration,
    // 5,000 x 3,000 r=8 0.091 -> 0.075; C2 and larger keep the largest tile.
    // (sharded: the same formula on the global matrix divided evenly over the ranks)
    const int64_t nnz_all = h->nranks > 1 ? h->nnz_global : h->nnz;
    if (nnz_all > 0) {
        const double density = (double)nnz_all / ((double)h->n * (double)h->m_global);
        const int tmin = std::max(64, (int)((40.0 / density + 31.0) / 32.0) * 32);
        const int64_t want = 4 * (int64_t)h->num_sms * 64;
        const int64_t m_eff = (h->m_global + h->nranks - 1) / h->nranks;
        auto segments = [&](int t) {
            return std::min((int64_t)cdiv(h->n, t) * m_eff, (int64_t)cdiv(m_eff, t) * h->n);
        };
        while (T - kTileRowsStep >= tmin && segments(T) < want) T -= kTileRowsStep;
    }
    if (const char *env = getenv("VBNMF_TILE_ROWS")) {  // experiments: force a smaller tile
        const int t = atoi(env);
        if (t >= 32 && t <= T) T = (t / 32) * 32;
    }
    return T;
}

int allreduce(H *h, double *buf, int64_t count) {
    if (h->nranks <= 1) return 0;
    NvtxRange nv("vbnmf:allreduce");
    CKN(g_nccl.AllReduce(buf, buf, (size_t)count, ncclFloat64, ncclSum, h->comm, h->stream));
    h->launches += 1;
    return 0;
}

// ---- all-reduce over NVLink peer memory (one process per GPU, CUDA IPC) -------------------------
void free_xchg(H *h) {
    if (!h->d_xchg) return;
    for (int p = 0; p < h->nranks && p < vb::kXchgFlags; p++)
        if (p != h->rank && h->xchg_peer[p]) cudaIpcCloseMemHandle(h->xchg_peer[p]);
    cudaFree(h->d_xchg);
    h->d_xchg = nullptr;
    for (auto &q : h->xchg_peer) q = nullptr;
    h->peer_ok = false;
}

// Collective over the ranks of the communicator (called from alloc_panels, which every rank runs
// with the same rank argument).  Any failure on any rank -> every rank keeps the NCCL all-reduce.
int setup_xchg(H *h) {
    free_xchg(h);
    if (h->nranks <= 1) return 0;
    // Opt-in (VBNMF_PEER_ALLREDUCE=1, the same environment on every rank): measured on 8 B200s at
    // C2 the NCCL all-reduce of the 1.6 MB vector (in-switch reduction) is 20 us per iteration
    // FASTER than the two peer-memory launches (1.490 vs 1.510 ms per iteration, bitwise identical
    // results), and equal on 2 GPUs (profiles/r01_peer_allreduce_ab.txt).
    if (!getenv("VBNMF_PEER_ALLREDUCE")) return 0;
    const bool want = h->nranks <= vb::kXchgFlags && g_nccl.AllGather;
    int bad = want ? 0 : 1;
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof(mine));
    h->xchg_stride = (((int64_t)red_len(h) * 8 + 255) / 256) * 256;
    const size_t bytes = (size_t)2 * vb::kXchgFlags * 8 + 4 * (size_t)h->xchg_stride;
    if (!bad) {
        if (cudaMalloc((void **)&h->d_xchg, bytes) != cudaSuccess) { h->d_xchg = nullptr; bad = 1; }
        else if (cudaMemset(h->d_xchg, 0, bytes) != cudaSuccess) bad = 1;
        else if (cudaIpcGetMemHandle(&mine, h->d_xchg) != cudaSuccess) bad = 1;
        cudaGetLastError();
    }
    // all-gather the 64-byte handles (+ the per-rank failure flag in a 65th... kept separate below)
    const int hb = (int)sizeof(cudaIpcMemHandle_t);
    ScopedBufs B(h);
    char *d_all = nullptr;
    CK(B.get(&d_all, (size_t)hb * (h->nranks + 1)));
    CK(cudaMemcpyAsync(d_all + (size_t)hb * h->nranks, &mine, hb, cudaMemcpyHostToDevice, h->stream));
    if (g_nccl.AllGather) {
        CKN(g_nccl.AllGather(d_all + (size_t)hb * h->nranks, d_all, (size_t)hb, ncclInt8, h->comm,
                             h->stream));
    }
    std::vector<cudaIpcMemHandle_t> all((size_t)h->nranks);
    CK(cudaMemcpyAsync(all.data(), d_all, (size_t)hb * h->nranks, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    B.free(d_all);
    if (!bad) {
        h->xchg_peer[h->rank] = h->d_xchg;
        for (int p = 0; p < h->nranks && !bad; p++) {
            if (p == h->rank) continue;
            void *q = nullptr;
            if (cudaIpcOpenMemHandle(&q, all[(size_t)p], cudaIpcMemLazyEnablePeerAccess) !=
                cudaSuccess) {
                cudaGetLastError();
                bad = 1;
            } else {
                h->xchg_peer[p] = (unsigned long long *)q;
            }
        }
    }
    // agree: the sum of the failure flags over the ranks must be zero
    double *d_flag = nullptr, flag = (double)bad;
    CK(B.get(&d_flag, 8));
    CK(cudaMemcpyAsync(d_flag, &flag, 8, cudaMemcpyHostToDevice, h->stream));
    int rc = allreduce(h, d_flag, 1);
    if (rc) return rc;
    CK(cudaMemcpyAsync(&flag, d_flag, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    B.free(d_flag);
    if (flag != 0.0) { free_xchg(h); return 0; }
    h->peer_ok = true;
    h->xchg_seq = 0;
    return 0;
}

// all-reduce of d_red (the W-side statistics and the scalars of the bound) inside the device-
// controlled loop: peer memory when it is set up, NCCL otherwise
int allreduce_red(H *h) {
    if (h->nranks <= 1) return 0;
    if (!h->peer_ok) return allreduce(h, h->d_red, red_len(h));
    NvtxRange nv("vbnmf:allreduce(peer)");
    vb::XchgArgs a;
    for (int p = 0; p < vb::kXchgFlags; p++) a.peer[p] = h->xchg_peer[p];
    a.nranks = h->nranks; a.rank = h->rank;
    a.seq = ++h->xchg_seq;
    a.n2 = red_len(h) / 2;
    a.buf_stride = h->xchg_stride;
    a.ctl = h->ctl;
    vb::xchg_publish_kernel<<<64, vb::kBlock, 0, h->stream>>>(
        a, reinterpret_cast<const double2 *>(h->d_red), h->d_counters + 8);
    vb::xchg_reduce_kernel<<<std::min(128, h->num_sms), vb::kBlock, 0, h->stream>>>(
        a, reinterpret_cast<double2 *>(h->d_red), h->d_counters + 9);
    h->launches += 2;
    return 0;
}

// every rank has left its device loop: nobody reads this rank's exchange region any more
int peer_exit_barrier(H *h) {
    if (!h->peer_ok) return 0;
    CKN(g_nccl.AllReduce(h->d_counters + 12, h->d_counters + 12, 1, ncclInt32, ncclSum, h->comm,
                         h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// ---- building the tiled layouts ---------------------------------------------------------------
// device row of every item: stable sort by descending count (cub radix sort of 2^31-1-count),
// then sorted position pos -> slab pos % S, local row pos / S.  scratch: 4 * count uint32.
int deal_device(H *h, const unsigned long long *d_cnt, int64_t count, int T, int S,
                int32_t *d_dev, uint32_t *scratch) {
    uint32_t *k_in = scratch, *k_out = scratch + count, *v_in = scratch + 2 * count,
             *v_out = scratch + 3 * count;
    const int g = cdiv(count, vb::kBlock);
    vb::order_keys_kernel<<<g, vb::kBlock, 0, h->stream>>>(count, d_cnt, k_in, v_in, nullptr);
    size_t tmp_bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in, k_out, v_in, v_out, count, 0, 31,
                                       h->stream));
    ScopedBufs B(h);
    void *d_tmp = nullptr;
    CK(B.get(&d_tmp, tmp_bytes));
    CK(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, k_in, k_out, v_in, v_out, count, 0, 31,
                                       h->stream));
    vb::deal_kernel<<<g, vb::kBlock, 0, h->stream>>>(count, S, T, v_out, d_dev);
    return 0;
}

// scratch: 4 * nnz uint32 (sort keys/payloads in and out), owned by get_layout.  One arena instead
// of a handful of GB-sized stream-ordered allocations per pass: the pool then sees the same few
// sizes at every handle creation and hands the blocks back without mapping new memory (the
// separate buffers cost 20-200 ms per layout, varying from run to run).
template <typename VT>
int build_pass(H *h, Layout *L, bool cols_pass, const int32_t *d_colof, uint32_t *scratch) {
    StageTimer tm(cols_pass ? "build_pass(cols)" : "build_pass(rows)");
    PassLayout &P = cols_pass ? L->cols : L->rows;
    const int64_t nnz = h->nnz;
    const int64_t NO = cols_pass ? L->NC : L->NG;
    const int nslabs = cols_pass ? L->Sg : L->Sc;
    P.E = (int64_t)nslabs * NO;
    // (the sweep kernels also step 32-bit segment positions by up to two group strides past E)
    if (P.E >= (int64_t)UINT32_MAX - 1024)
        return fail(h, VBNMF_ERR_ARG, "matrix too large for 32-bit segment keys on one GPU");
    const int g = h->num_sms * 8;
    uint32_t *k_in = scratch, *k_out = scratch + nnz, *p_in = scratch + 2 * nnz,
             *p_out = scratch + 3 * nnz;
    { StageTimer t1("  make_keys");
    vb::make_keys_kernel<VT><<<g, vb::kBlock, 0, h->stream>>>(
        nnz, h->d_rowidx, d_colof, L->d_gene_dev, L->d_cell_dev, L->T, NO, cols_pass,
        L->npg > 0 ? (const VT *)h->d_val : nullptr, k_in, p_in); }
    int bits = 1;
    while (((int64_t)1 << bits) < P.E) bits++;
    size_t tmp_bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in, k_out, p_in, p_out, nnz, 0, bits,
                                       h->stream));
    // the segment pointers stay with the 8-byte layout; the packed-16 layout needs them only
    // until its segments are built
    ScopedBufs B(h);
    void *d_tmp = nullptr;
    int64_t *d_ptr = nullptr;
    CK(B.get(&d_tmp, tmp_bytes));
    { StageTimer t1("  radix_sort");
    CK(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, k_in, k_out, p_in, p_out, nnz, 0, bits,
                                       h->stream)); }
    CK(B.get(&d_ptr, (size_t)(P.E + 1) * 8));
    { StageTimer t1("  segment_ptr");
    vb::segment_ptr_kernel<<<g, vb::kBlock, 0, h->stream>>>(P.E, nnz, k_out, d_ptr); }
    CK(cudaStreamSynchronize(h->stream));
    B.free(d_tmp);
    if (L->npg > 0) {
        // packed-16 layout: pad every segment to whole quads, scan the quad counts into ptr4
        uint32_t *d_len4 = nullptr;
        uint8_t *d_dead = nullptr;
        CK(B.get(&d_len4, (size_t)(P.E + 1) * 4));
        if (L->kmult == 1) CK(B.get(&d_dead, (size_t)P.E));
        CK(vmalloc(h, &P.d_ptr4, (size_t)(P.E + 1) * 4));
        const uint32_t *d_words = p_out;  // the sorted payloads are the packed words
        { StageTimer t1("  plan(p16)");
        vb::plan_p16_kernel<<<g, vb::kBlock, 0, h->stream>>>(P.E, d_ptr, d_words, L->npg,
                                                             L->kmult, L->mode, d_len4, d_dead); }
        // order the segments by decreasing number of steps inside windows of W owners
        // (seg_order_keys_kernel; VBNMF_SEG_WINDOW: experiments, 0 = owner order)
        int W = kSegWindow;
        if (const char *wenv = getenv("VBNMF_SEG_WINDOW")) W = atoi(wenv);
        uint32_t *d_len4p = nullptr, *d_okey = nullptr, *d_oval = nullptr;
        uint8_t *d_deadp = nullptr;
        CK(B.get(&d_len4p, (size_t)(P.E + 1) * 4));
        if (d_dead) CK(B.get(&d_deadp, (size_t)P.E));
        CK(vmalloc(h, &P.d_seg, (size_t)P.E * 4));
        { StageTimer t1("  order segments");
        const int ge = cdiv(P.E + 1, vb::kBlock);
        void *d_otmp = nullptr;
        if (W > 0) {
            CK(B.get(&d_okey, (size_t)P.E * 4 * 4));  // keys in/out, values in/out
            d_oval = d_okey + 2 * P.E;
            vb::seg_order_keys_kernel<<<ge, vb::kBlock, 0, h->stream>>>(P.E, NO, W, d_len4, d_dead,
                                                                        L->npg, d_okey, d_oval);
            const int64_t nwin_all = (int64_t)nslabs * ((NO + W - 1) / W);
            if (nwin_all >= ((int64_t)1 << 22))
                return fail(h, VBNMF_ERR_ARG, "too many segment windows for 32-bit sort keys");
            int obits = 10;
            while (((int64_t)1 << obits) < nwin_all * 1024) obits++;
            size_t ob = 0;
            CK(cub::DeviceRadixSort::SortPairs(nullptr, ob, d_okey, d_okey + P.E, d_oval,
                                               d_oval + P.E, P.E, 0, obits, h->stream));
            CK(B.get(&d_otmp, ob));
            CK(cub::DeviceRadixSort::SortPairs(d_otmp, ob, d_okey, d_okey + P.E, d_oval,
                                               d_oval + P.E, P.E, 0, obits, h->stream));
        }
        vb::seg_permute_kernel<<<ge, vb::kBlock, 0, h->stream>>>(
            P.E, NO, W > 0 ? d_oval + P.E : nullptr, d_len4, d_dead, d_len4p, d_deadp, P.d_seg);
        B.free(d_otmp); }
        size_t scan_bytes = 0;
        CK(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, d_len4p, P.d_ptr4, P.E + 1, h->stream));
        void *d_scan = nullptr;
        CK(B.get(&d_scan, scan_bytes));
        CK(cub::DeviceScan::ExclusiveSum(d_scan, scan_bytes, d_len4p, P.d_ptr4, P.E + 1, h->stream));
        if (2 * nnz + 32 * P.E >= ((int64_t)1 << 34))
            return fail(h, VBNMF_ERR_ARG, "matrix too large for 32-bit quad pointers on one GPU");
        uint32_t quads = 0;
        CK(cudaMemcpyAsync(&quads, P.d_ptr4 + P.E, 4, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        B.free(d_len4); B.free(d_scan);
        B.free(d_len4p); B.free(d_okey);
        CK(vmalloc(h, &P.d_ent, (size_t)quads * 16));
        P.nent = (int64_t)quads * 4;
        { StageTimer t1("  build_segments(p16)");
        vb::build_segments_p16_kernel<<<g, vb::kBlock, 0, h->stream>>>(
            P.E, NO, d_ptr, P.d_ptr4, P.d_seg, d_words, L->npg, L->kmult, L->mode,
            cols_pass ? h->n : h->m, cols_pass ? L->Sg : L->Sc, (uint32_t *)P.d_ent); }
        CK(vmalloc(h, &P.d_split, (size_t)(L->grid + 1) * 8));
        // per-segment overhead in quads (VBNMF_SPLIT_KAPPA: tuning)
        const char *kenv = getenv("VBNMF_SPLIT_KAPPA");
        const double kappa = kenv ? atof(kenv) : kSplitKappa;
        vb::split_p16_kernel<<<cdiv(L->grid + 1, 128), 128, 0, h->stream>>>(L->grid, P.E, P.d_ptr4,
                                                                           kappa, P.d_split);
        if (d_deadp)
            vb::tag_dead_kernel<<<cdiv(P.E, vb::kBlock), vb::kBlock, 0, h->stream>>>(P.E, d_deadp,
                                                                                    P.d_ptr4);
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaGetLastError());
        return 0;
    }
    P.nent = nnz;
    if (sizeof(VT) == 4) {
        CK(vmalloc(h, &P.d_ent, (size_t)nnz * 8));
    } else {
        CK(vmalloc(h, &P.d_idx, (size_t)nnz * 4));
        CK(vmalloc(h, &P.d_val, (size_t)nnz * sizeof(VT)));
    }
    { StageTimer t1("  build_segments");
    vb::build_segments_kernel<VT><<<g, vb::kBlock, 0, h->stream>>>(
        P.E, d_ptr, p_out, h->d_rowidx, d_colof, L->d_gene_dev, L->d_cell_dev,
        (const VT *)h->d_val, L->T, cols_pass, P.d_idx, (VT *)P.d_val, (int2 *)P.d_ent); }
    CK(vmalloc(h, &P.d_split, (size_t)(L->grid + 1) * 8));
    vb::split_kernel<<<cdiv(L->grid + 1, 128), 128, 0, h->stream>>>(L->grid, P.E, nnz, d_ptr,
                                                                   P.d_split);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    P.d_ptr = B.keep(d_ptr);
    return 0;
}

template <typename VT>
void launch_expand_cols(H *h, int32_t *d_colof, unsigned long long *d_cnt, unsigned *d_bad) {
    vb::expand_cols_kernel<VT><<<h->num_sms * 8, vb::kBlock, 0, h->stream>>>(
        h->m, h->n, h->d_colptr, h->d_rowidx, (const VT *)h->d_val, d_colof, d_cnt,
        d_cnt ? d_cnt + h->n : nullptr, d_bad);
}

int get_layout(H *h, int T, int npg, int kmult, int mode, Layout **out) {
    if (!h->p16) npg = 0;
    if (npg != 8 && mode != vb::kSchedOne4) { kmult = 4; mode = vb::kSchedPlain; }
    for (Layout *l : h->layouts)
        if (l->T == T && l->npg == npg && l->kmult == kmult && l->mode == mode) { *out = l; return 0; }
    StageTimer tm("get_layout(total)");
    Layout *L = new Layout();
    L->T = T;
    L->npg = npg;
    L->kmult = kmult;
    L->mode = mode;
    L->Sg = cdiv(h->n, T);
    L->Sc = cdiv(h->m, T);
    L->NG = (int64_t)L->Sg * T;
    L->NC = (int64_t)L->Sc * T;
    L->grid = h->num_sms;
    auto bail = [&](int rc) { L->release(h->stream); delete L; return rc; };
    auto body = [&]() -> int {
        CK(vmalloc(h, &L->d_gene_dev, (size_t)h->n * 4));
        CK(vmalloc(h, &L->d_cell_dev, (size_t)h->m * 4));
        // one arena: [colof | 4 sort buffers], nnz 32-bit words each (also the scratch of the
        // two small sorts that renumber the genes and the cells)
        const int64_t words = std::max<int64_t>(h->nnz * 5, 4 * std::max(h->n, h->m));
        ScopedBufs B(h);
        uint32_t *arena = h->d_arena;
        const bool have_colof = arena && h->colof_in_arena;
        h->d_arena = nullptr;
        h->colof_in_arena = false;
        if (arena) B.hold(arena);
        else CK(B.get(&arena, (size_t)words * 4));
        int32_t *d_colof = (int32_t *)arena;
        uint32_t *scratch = arena + h->nnz;
        int rc = 0;
        { StageTimer t1("  deal(device sort)");
        // (the scratch of the small sorts must not overlap colof: needs 4 * max(n, m) words)
        uint32_t *dscr = scratch;
        uint32_t *own = nullptr;
        if (4 * std::max(h->n, h->m) > 4 * h->nnz) {
            CK(B.get(&own, (size_t)4 * std::max(h->n, h->m) * 4));
            dscr = own;
        }
        rc = deal_device(h, h->d_cnt, h->n, T, L->Sg, L->d_gene_dev, dscr);
        if (!rc) rc = deal_device(h, h->d_cnt + h->n, h->m, T, L->Sc, L->d_cell_dev, dscr);
        B.free(own); }
        if (rc) return rc;
        return with_val_type(h->val_float, [&](auto v) -> int {
            using VT = decltype(v);
            if (!have_colof) {
                StageTimer t1("  expand_cols");
                launch_expand_cols<VT>(h, d_colof, nullptr, nullptr);
            }
            int rc2 = build_pass<VT>(h, L, true, d_colof, scratch);
            if (!rc2) rc2 = build_pass<VT>(h, L, false, d_colof, scratch);
            StageTimer t1("  free(arena)");
            B.free(arena);
            return rc2;
        });
    };
    int rc = body();
    if (rc) return bail(rc);
    h->layouts.push_back(L);
    *out = L;
    return 0;
}

void drop_layouts(H *h) {
    for (Layout *l : h->layouts) { l->release(h->stream); delete l; }
    h->layouts.clear();
    h->L = nullptr;
}

// nonzero counts per gene / cell (kept on the device), validation, the constants over the nonzeros
template <typename VT>
int scan_matrix_t(H *h) {
    StageTimer tm("scan_matrix");
    const int64_t n = h->n, m = h->m, nnz = h->nnz;
    const int gridK = h->num_sms * 8;
    ScopedBufs B(h);
    double *d_part = nullptr, *d_out = nullptr;
    unsigned *d_flags = nullptr;  // [bad row index, empty rows, empty cols]
    CK(B.get(&d_part, (size_t)gridK * 4 * 8));
    CK(B.get(&d_out, 4 * 8));
    CK(B.get(&d_flags, 4 * sizeof(unsigned)));
    CK(cudaMemsetAsync(d_flags, 0, 4 * sizeof(unsigned), h->stream));
    vb::count_constants_kernel<VT><<<gridK, vb::kBlock, 0, h->stream>>>(
        nnz, (const VT *)h->d_val, d_part, d_out, h->d_counters + 4);
    double consts[4];
    unsigned flags[4];
    CK(cudaMemcpyAsync(consts, d_out, 32, cudaMemcpyDeviceToHost, h->stream));
    // the column of every entry goes into the arena the first layout build sorts in (so that it
    // is expanded once), or into a temporary when the handle has no arena
    int32_t *d_colof = (int32_t *)h->d_arena;
    if (!d_colof) CK(B.get(&d_colof, (size_t)nnz * 4));
    CK(vmalloc(h, &h->d_cnt, (size_t)(n + m) * 8));
    CK(cudaMemsetAsync(h->d_cnt, 0, (size_t)(n + m) * 8, h->stream));
    launch_expand_cols<VT>(h, d_colof, h->d_cnt, d_flags);
    h->colof_in_arena = h->d_arena != nullptr;
    // empty genes / cells: counted by the kernel that makes the sort keys (scratch discarded)
    uint32_t *d_scr = nullptr;
    CK(B.get(&d_scr, (size_t)2 * std::max(n, m) * 4));
    vb::order_keys_kernel<<<cdiv(n, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        n, h->d_cnt, d_scr, d_scr + std::max(n, m), d_flags + 1);
    vb::order_keys_kernel<<<cdiv(m, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        m, h->d_cnt + n, d_scr, d_scr + std::max(n, m), d_flags + 2);
    CK(cudaMemcpyAsync(flags, d_flags, sizeof(flags), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    if (flags[0]) return fail(h, VBNMF_ERR_ARG, "row index out of range");
    if (consts[3] != 0.0)
        return fail(h, VBNMF_ERR_ARG, "counts must be finite and non-negative");
    h->empty_rows = flags[1];
    h->empty_cols = flags[2];
    // R/bayesian.R:244-247: refused when a factorization is set up (alloc_panels), not here -- a
    // handle made by vbnmf_create_from_mtx may hold a matrix the front end has yet to filter
    // (read_10x drops empty genes / cells, R/utils.R:52), and the empty genes of ONE shard are
    // legal (vbnmf_attach_comm repeats the test on the all-reduced gene counts).
    h->lgx = consts[0];
    h->mlconst = consts[1];
    // VBNMF_NO_P16=1 keeps the 8-byte entries (A/B measurements, tests of that path)
    h->p16 = h->val_float && consts[2] == 0.0 && !getenv("VBNMF_NO_P16");
    return 0;
}

// ---- panels -------------------------------------------------------------------------------------
void free_panels(H *h) {
    free_xchg(h);
    double **ps[] = {&h->d_lw, &h->d_lh, &h->d_alw, &h->d_alh, &h->d_red, &h->d_ShRaw,
                     &h->d_Part1, &h->d_Part2, &h->d_xl, &h->d_scal, &h->d_partW, &h->d_partH,
                     &h->d_partC};
    for (auto p : ps) {
        vfree(h->stream, *p);
        *p = nullptr;
    }
    if (h->h_scal) cudaFreeHost(h->h_scal);
    h->h_scal = nullptr;
    vfree(h->stream, h->d_lw32); vfree(h->stream, h->d_lh32);
    h->d_lw32 = h->d_lh32 = nullptr;
}

int alloc_panels(H *h, int r) {
    const int rp = pad_rank(r);
    const vb::RpTable *tab = vb::rp_table(rp);
    if (!tab) return fail(h, VBNMF_ERR_ARG, "no kernels compiled for this rank");
    const int rs = tab->rs;
    const bool f32 = h->precision == VBNMF_FP32_STORAGE;
    // R/bayesian.R:244-245 (for a sharded matrix the test was made on the global gene counts)
    if (!getenv("VBNMF_ALLOW_EMPTY")) {
        if (h->empty_rows) return fail(h, VBNMF_ERR_EMPTY, "Input matrix contains empty rows");
        if (h->empty_cols) return fail(h, VBNMF_ERR_EMPTY, "Input matrix contains empty columns");
    }
    // split layout + rotated gathers: fp64 panels, packed-16 entries, rows of 4..10 units
    // (tab->split64 = units of block A: 8 for ranks 16..20, 4 for ranks 8..14)
    // The 4-unit variant is opt-in (VBNMF_SPLIT4=1): measured at C2 (r = 10) it is SLOWER than the
    // lock-step layout (1.48 vs 1.41 ms per iteration) although it saves ~11 % of the gather
    // wavefronts -- with rows of 5 units the pass is bound by issue slots and latency as much as by
    // the LSU pipe, and the rotated addresses add one LOP3 per unit.
    const bool split = !f32 && h->p16 && tab->split64 && !getenv("VBNMF_NO_SPLIT") &&
                       (tab->split64 == 8 || getenv("VBNMF_SPLIT4"));
    // a slab row of the split layout is block A + a dense block B (kernels.cuh split_ps)
    const int row_bytes = f32 ? tab->rsf * 4 : (split ? vb::split_ps(rp) * 8 : rs * 8);
    // 4-lane groups: split layout with an 8-unit block A (ranks 15..20); VBNMF_NO_G4=1 keeps the
    // 8-lane groups (A/B measurements)
    const bool g4 = split && tab->stage64_g4 >= 0 && !getenv("VBNMF_NO_G4");
    const int stage_bytes = h->p16 ? (f32 ? tab->stage32 : (g4 ? tab->stage64_g4 : tab->stage64)) : 0;
    const int T = choose_tile_rows(h, row_bytes, stage_bytes);
    Layout *L = nullptr;
    int kmult = split ? 1 : 4;
    if (const char *e = getenv("VBNMF_KMULT")) kmult = atoi(e) == 1 ? 1 : 4;  // experiments
    // schedule of block B: parity classes side by side (4-unit block A), four classes of two
    // lanes (8-unit block A + two dense units: ranks 19, 20), else eight residue classes
    int mode = vb::kSchedPlain;
    if (split && tab->split64 == 4) mode = vb::kSchedSbs;
    else if (split && vb::split_bs(rp) == 4 && !getenv("VBNMF_NO_CLS4")) mode = vb::kSchedCls4;
    if (g4) mode = vb::kSchedOne4;
    int rc = get_layout(h, T, f32 ? tab->npg32 : (g4 ? 4 : tab->npg64), kmult, mode, &L);
    if (rc) return rc;
    if (rp == h->rp && L == h->L && h->d_lw && h->panel_precision == h->precision &&
        h->split_kind == (split ? (g4 ? 2 : 1) : 0)) {
        h->r = r;
        return 0;
    }
    free_panels(h);
    h->tab = tab;
    h->L = L;
    h->tsplit = split ? vb::make_tsplit(T, rp) : 0;
    h->split_kind = split ? (g4 ? 2 : 1) : 0;
    h->r = r; h->rp = rp; h->rs = rs; h->rsf = tab->rsf;
    h->panel_precision = h->precision;
    h->smem_bytes = T * row_bytes + stage_bytes;
    // The opt-in is per kernel and device, i.e. shared by every handle of the process: always ask
    // for the largest tile so that a second handle with a smaller tile cannot lower the limit
    // under this one.
    if (tab->sweep_prepare(kTileBytes))
        return fail(h, VBNMF_ERR_CUDA, "cannot opt in to the shared-memory tile size");
    const size_t gr = (size_t)L->NG * rs * 8, cr = (size_t)L->NC * rs * 8;
    CK(vmalloc(h, &h->d_lw, gr));
    CK(vmalloc(h, &h->d_alw, gr));
    CK(vmalloc(h, &h->d_lh, cr));
    CK(vmalloc(h, &h->d_alh, cr));
    CK(vmalloc(h, &h->d_ShRaw, cr));
    CK(vmalloc(h, &h->d_red, (size_t)red_len(h) * 8));
    CK(vmalloc(h, &h->d_Part1, (size_t)L->Sg * cr));
    CK(vmalloc(h, &h->d_Part2, (size_t)L->Sc * gr));
    CK(vmalloc(h, &h->d_xl, (size_t)L->grid * 8));
    CK(vmalloc(h, &h->d_scal, (size_t)(rs + 8) * 8));
    h->gridC = h->num_sms * 4;
    // per-CTA partial rows of the posterior / ML / column-sum kernels (the larger of the two grids)
    const int64_t gw = std::max(cdiv(L->NG, vb::post_rows_per_cta(L->NG, rs, h->num_sms)),
                                std::max(cdiv(L->NG, vb::kPostRows), cdiv(L->NG, vb::kBlock)));
    const int64_t gh = std::max(cdiv(L->NC, vb::post_rows_per_cta(L->NC, rs, h->num_sms)),
                                std::max(cdiv(L->NC, vb::kPostRows), cdiv(L->NC, vb::kBlock)));
    CK(vmalloc(h, &h->d_partW, (size_t)gw * (rs + 3) * 8));
    CK(vmalloc(h, &h->d_partH, (size_t)gh * (rs + 3) * 8));
    CK(vmalloc(h, &h->d_partC, (size_t)h->gridC * 2 * 8));
    CK(cudaMallocHost(&h->h_scal, (size_t)2 * (rs + 8) * 8));
    CK(cudaMemsetAsync(h->d_red, 0, (size_t)red_len(h) * 8, h->stream));
    CK(cudaMemsetAsync(h->d_scal, 0, (size_t)(rs + 8) * 8, h->stream));
    CK(cudaMemsetAsync(h->d_ShRaw, 0, cr, h->stream));
    if (f32) {
        CK(vmalloc(h, &h->d_lw32, (size_t)L->NG * h->rsf * 4));
        CK(vmalloc(h, &h->d_lh32, (size_t)L->NC * h->rsf * 4));
    }
    return setup_xchg(h);
}

// panels for rank r with all four zeroed (their padding rows and columns must read 0)
int zeroed_panels(H *h, int r) {
    int rc = alloc_panels(h, r);
    if (rc) return rc;
    const size_t gr = (size_t)h->L->NG * h->rs * 8, cr = (size_t)h->L->NC * h->rs * 8;
    CK(cudaMemsetAsync(h->d_lw, 0, gr, h->stream));
    CK(cudaMemsetAsync(h->d_alw, 0, gr, h->stream));
    CK(cudaMemsetAsync(h->d_lh, 0, cr, h->stream));
    CK(cudaMemsetAsync(h->d_alh, 0, cr, h->stream));
    return 0;
}

// fp32-storage mode: refresh the mirrors from the fp64 panels (after an upload)
int refresh_mirrors(H *h) {
    if (h->precision != VBNMF_FP32_STORAGE) return 0;
    h->tab->mirror(h->L->NG, h->d_lw, h->d_lw32, h->stream);
    h->tab->mirror(h->L->NC, h->d_lh, h->d_lh32, h->stream);
    h->launches += 2;
    CK(cudaGetLastError());
    return 0;
}

// rowSums(eh) of the state just loaded (alh holds eh before the first update), over all shards,
// into the tail of the reduce buffer and the host vectors
int initial_ehsum(H *h) {
    const Layout *L = h->L;
    const int rs = h->rs, r = h->r;
    int rc;
    double *tail = h->d_red + tail_off(h);
    CK(cudaMemsetAsync(tail, 0, (size_t)(rs + 8) * 8, h->stream));
    vb::ColsumArgs ca{L->NC, h->d_alh, h->d_partH, tail, h->d_counters + 1, 0};
    h->tab->colsum(ca, h->stream);
    h->launches += 1;
    if ((rc = allreduce(h, tail, rs + 8))) return rc;
    double s[kMaxRank + 16];  // rs + 8 <= 66 + 8
    CK(cudaMemcpyAsync(s, tail, (size_t)(rs + 8) * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    for (int k = 0; k < kMaxRank; k++) {
        h->ehsum[k] = k < r ? s[k] : 0.0;
        h->ewsum[k] = 0.0;
        h->bew[k] = h->beh[k] = 1.0;
    }
    h->stats_valid = false;
    h->has_posterior = false;
    return 0;
}

// a state just written into the panels: the fp32 mirrors and rowSums(eh)
int loaded_state(H *h) {
    int rc = refresh_mirrors(h);
    return rc ? rc : initial_ehsum(h);
}

// caller's matrix (n x r column-major for the W side, r x m for the H side) -> device panel(s) in
// device order, zero padded.  The matrix goes up as it is (staged through pinned memory by the
// worker pool) and is permuted on the device.
int upload_panel(H *h, double *dst1, double *dst2, const double *src, bool wside, int r);

// ---- one iteration --------------------------------------------------------------------------------
inline int entry_format(const H *h) {
    return h->L->npg > 0 ? vb::kEntP16 : (h->val_float ? vb::kEntF32 : vb::kEntF64);
}
int launch_posterior(H *h, bool wside, double a, double b, double fud) {
    NvtxRange nv(wside ? "vbnmf:posterior_W" : "vbnmf:posterior_H");
    const Layout *L = h->L;
    double *tail = h->d_red + tail_off(h);
    vb::PosteriorArgs p;
    p.rows = wside ? L->NG : L->NC;
    p.T = L->T;
    p.S = wside ? L->Sg : L->Sc;
    p.nvalid = wside ? h->n : h->m;
    p.r = h->r;
    p.a = a; p.b = b; p.fud = fud;
    p.osum = wside ? tail : h->d_scal;
    p.SRaw = wside ? h->d_red : h->d_ShRaw;
    p.l = wside ? h->d_lw : h->d_lh;
    p.al_out = wside ? h->d_alw : h->d_alh;
    p.part = wside ? h->d_partW : h->d_partH;
    p.out = wside ? h->d_scal : tail;
    p.counter = h->d_counters + (wside ? 0 : 1);
    p.l32 = wside ? h->d_lw32 : h->d_lh32;  // nullptr in fp64 mode
    p.ctl = h->ctl;
    p.hoff = wside ? 0 : 2;
    p.rows_per_cta = vb::post_rows_per_cta(p.rows, h->rs, h->num_sms);
    p.tsplit = h->tsplit;
    h->tab->posterior(p, h->stream);
    h->launches += 1;
    return 0;
}

// cell-owner pass: ShRaw, enth -> tail[rs+3], xlogp -> tail[rs+4]
int launch_sweep_cols(H *h) {
    NvtxRange nv("vbnmf:sweep_cell_owner");
    const Layout *L = h->L;
    double *tail = h->d_red + tail_off(h);
    const bool f32 = h->precision == VBNMF_FP32_STORAGE;
    vb::SweepTiledArgs a{L->NC, L->T, L->cols.d_split, L->cols.d_ptr, L->cols.d_ent,
                         L->cols.d_idx, (const double *)L->cols.d_val,
                         f32 ? (const void *)h->d_lh32 : (const void *)h->d_lh,
                         f32 ? (const void *)h->d_lw32 : (const void *)h->d_lw, h->d_Part1, h->d_xl,
                         h->ctl, L->cols.d_ptr4, L->cols.d_seg};
    h->tab->sweep(a, true, entry_format(h), f32, h->split_kind, L->grid, h->smem_bytes, h->stream);
    vb::CombineArgs c{L->NC, L->Sg, h->r, h->d_Part1, h->d_lh, h->d_ShRaw, h->d_partC,
                      tail + h->rs + 3, h->d_counters + 2, h->d_xl, L->grid, h->gridC, h->ctl,
                      h->tsplit};
    h->tab->combine(c, h->stream);
    h->launches += 2;
    return 0;
}

// gene-owner pass: SwRaw (local part) -> d_red, entw (local part) -> tail[rs+5]
int launch_sweep_rows(H *h) {
    NvtxRange nv("vbnmf:sweep_gene_owner");
    const Layout *L = h->L;
    double *tail = h->d_red + tail_off(h);
    const bool f32 = h->precision == VBNMF_FP32_STORAGE;
    vb::SweepTiledArgs a{L->NG, L->T, L->rows.d_split, L->rows.d_ptr, L->rows.d_ent,
                         L->rows.d_idx, (const double *)L->rows.d_val,
                         f32 ? (const void *)h->d_lw32 : (const void *)h->d_lw,
                         f32 ? (const void *)h->d_lh32 : (const void *)h->d_lh, h->d_Part2, nullptr,
                         h->ctl, L->rows.d_ptr4, L->rows.d_seg};
    h->tab->sweep(a, false, entry_format(h), f32, h->split_kind, L->grid, h->smem_bytes, h->stream);
    vb::CombineArgs c{L->NG, L->Sc, h->r, h->d_Part2, h->d_lw, h->d_red, h->d_partC,
                      tail + h->rs + 5, h->d_counters + 3, nullptr, 0, h->gridC, h->ctl,
                      h->tsplit};
    h->tab->combine(c, h->stream);
    h->launches += 2;
    return 0;
}

// statistics at the current lw, lh: ShRaw, SwRaw (global), xlogp, enth, entw
int sweep(H *h) {
    int rc;
    if ((rc = launch_sweep_cols(h))) return rc;
    if ((rc = launch_sweep_rows(h))) return rc;
    if ((rc = allreduce(h, h->d_red, red_len(h)))) return rc;
    CK(cudaGetLastError());
    h->stats_valid = true;
    return 0;
}

// the statistics at the loaded state when they are stale; the H-side sums already in the reduce
// buffer must survive the pass
int ensure_stats(H *h) {
    if (h->stats_valid) return 0;
    std::vector<double> keep((size_t)h->rs + 8, 0.0);
    for (int k = 0; k < h->r; k++) keep[k] = h->ehsum[k];
    int rc = sweep(h);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h->d_red + tail_off(h), keep.data(), (size_t)h->rs * 8,
                       cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int fetch_scalars(H *h) {
    const int w = h->rs + 8;
    CK(cudaMemcpyAsync(h->h_scal, h->d_scal, w * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->h_scal + w, h->d_red + tail_off(h), w * sizeof(double),
                       cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// host half of an iteration: take the freshly fetched scalars, refresh the small host vectors and
// assemble the lower bound (src/vbnmf_update.cpp:67-90 in its nonzero-only form, see DESIGN.md)
double absorb_scalars(H *h, const double *hyper) {
    const double aw = hyper[0], bw = hyper[1], ah = hyper[2], bh = hyper[3];
    const int rs = h->rs, r = h->r, w = rs + 8;
    const double *ws = h->h_scal, *hs = h->h_scal + w;
    for (int k = 0; k < r; k++) {
        h->bew[k] = aw / bw + h->ehsum[k];  // rowSums(eh_old), :42-43
        h->ewsum[k] = ws[k];
        h->beh[k] = ah / bh + h->ewsum[k];  // colSums(ew_new), :52-53
    }
    for (int k = 0; k < r; k++) h->ehsum[k] = hs[k];
    for (int c = 0; c < 3; c++) { h->wacc[c] = ws[rs + c]; h->hacc[c] = hs[rs + c]; }
    h->enth = hs[rs + 3];
    h->xlogp = hs[rs + 4];
    h->entw = hs[rs + 5];
    const double nr = (double)h->n * r, mr = (double)h->m_global * r;
    double U = 0.0;
    for (int k = 0; k < r; k++) U -= h->ewsum[k] * h->ehsum[k];       // -sum(ew.eh), :78
    U -= h->entw + h->enth - h->xlogp;                                // -x((A+B)/wth - log wth), :74-78
    U -= h->lgx;                                                      // -lgamma(x+1), :81
    U += h->wacc[0] + nr * (-lgamma(aw) + aw * log(aw / bw));         // :82-86
    U += h->hacc[0] + mr * (-lgamma(ah) + ah * log(ah / bh));         // :87-89
    h->has_posterior = true;
    return U / ((double)h->n * (double)h->m_global);                  // :90 (in double, not int)
}

// One reference iteration given valid statistics: posterior update (W then H), sweep at the new
// factors, lower bound.  src/vbnmf_update.cpp:38-90.
int iterate(H *h, const double *hyper, double fud, double *lkh) {
    int rc;
    if ((rc = launch_posterior(h, true, hyper[0], hyper[1], fud))) return rc;
    if ((rc = launch_posterior(h, false, hyper[2], hyper[3], fud))) return rc;
    if ((rc = sweep(h))) return rc;
    if ((rc = fetch_scalars(h))) return rc;
    *lkh = absorb_scalars(h, hyper);
    return 0;
}

void means_of(const H *h, double *means) {
    const double nr = (double)h->n * h->r, mr = (double)h->m_global * h->r;
    means[0] = h->wacc[1] / nr;
    means[1] = h->hacc[1] / mr;
    means[2] = h->wacc[2] / nr;
    means[3] = h->hacc[2] / mr;
}

// ---- host worker pool ---------------------------------------------------------------------------
// Persistent threads that copy / convert host arrays into the pinned staging buffers (creating
// and joining threads per 32 MB chunk cost more than the conversion).  The number of workers is
// min(16, hardware threads), VBNMF_HOST_THREADS, or vbnmf_set_host_threads(): with one process
// per GPU the host side should pass cores / processes.
class WorkerPool {
public:
    void set_threads(int n) {
        std::lock_guard<std::mutex> lk(mu_);
        want_ = std::max(1, std::min(n, 64));
    }
    int threads() {
        std::lock_guard<std::mutex> lk(mu_);
        return want_;
    }
    // fn(part, nparts) for part in [0, nparts), nparts = current number of workers; returns when
    // all parts are done.  The calling thread runs part 0.
    void run(const std::function<void(int, int)> &fn) {
        std::unique_lock<std::mutex> lk(mu_);
        const int np = want_;
        while ((int)th_.size() < np - 1) {
            const int id = (int)th_.size() + 1;
            th_.emplace_back([this, id] { loop(id); });
        }
        fn_ = &fn;
        nparts_ = np;
        pending_ = np - 1;
        gen_++;
        lk.unlock();
        cv_.notify_all();
        fn(0, np);
        lk.lock();
        done_.wait(lk, [this] { return pending_ == 0; });
        fn_ = nullptr;
    }
    WorkerPool() {
        unsigned hw = std::thread::hardware_concurrency();
        want_ = (int)std::max(1u, std::min(16u, hw ? hw : 1u));
        if (const char *e = getenv("VBNMF_HOST_THREADS")) want_ = std::max(1, std::min(atoi(e), 64));
    }
    ~WorkerPool() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
            gen_++;
        }
        cv_.notify_all();
        for (auto &t : th_) t.join();
    }

private:
    void loop(int id) {
        uint64_t seen = 0;
        for (;;) {
            std::unique_lock<std::mutex> lk(mu_);
            cv_.wait(lk, [&] { return gen_ != seen; });
            seen = gen_;
            if (stop_) return;
            if (id >= nparts_ || !fn_) continue;
            const std::function<void(int, int)> *fn = fn_;
            const int np = nparts_;
            lk.unlock();
            (*fn)(id, np);
            lk.lock();
            if (--pending_ == 0) done_.notify_all();
        }
    }
    std::mutex mu_;
    std::condition_variable cv_, done_;
    std::vector<std::thread> th_;
    const std::function<void(int, int)> *fn_ = nullptr;
    int want_ = 1, nparts_ = 0, pending_ = 0;
    uint64_t gen_ = 0;
    bool stop_ = false;
};
WorkerPool &pool() {
    static WorkerPool *p = new WorkerPool();  // leaked on purpose: no join at process exit
    return *p;
}

// Host -> device upload of a large array through pinned staging buffers: the pool converts /
// validates a chunk into one buffer while the copy engine drains the others.  `conv` maps
// src[i] -> dst element and returns false for an invalid element.
struct Staging {
    static constexpr size_t kBytes = (size_t)32 << 20;
    static constexpr int kSlots = 3;
    void *buf[kSlots] = {};
    cudaEvent_t ev[kSlots];
    bool ok = false;
    bool init() {
        if (ok) return true;
        for (int i = 0; i < kSlots; i++) {
            if (cudaMallocHost(&buf[i], kBytes) != cudaSuccess) return false;
            if (cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) != cudaSuccess) return false;
        }
        ok = true;
        return true;
    }
};
Staging g_staging;
std::mutex g_staging_mu;  // the staging buffers and the pool are shared by all handles of the process

template <typename Src, typename Dst, typename Conv>
int staged_upload(H *h, Dst *d_dst, const Src *src, int64_t count, Conv conv, bool *all_ok) {
    std::lock_guard<std::mutex> lock(g_staging_mu);
    if (!g_staging.init()) return fail(h, VBNMF_ERR_CUDA, "cannot allocate pinned staging buffers");
    const int64_t per = (int64_t)(Staging::kBytes / sizeof(Dst));
    std::atomic<int> bad{0};
    int slot = 0;
    for (int64_t lo = 0; lo < count; lo += per, slot = (slot + 1) % Staging::kSlots) {
        const int64_t len = std::min(per, count - lo);
        CK(cudaEventSynchronize(g_staging.ev[slot]));  // the copy that last used this buffer is done
        Dst *out = (Dst *)g_staging.buf[slot];
        const Src *in = src + lo;
        pool().run([&](int t, int nt) {
            const int64_t a = len * t / nt, b = len * (t + 1) / nt;
            bool okk = true;
            for (int64_t i = a; i < b; i++) okk &= conv(in[i], out[i]);
            if (!okk) bad.store(1, std::memory_order_relaxed);
        });
        CK(cudaMemcpyAsync(d_dst + lo, out, (size_t)len * sizeof(Dst), cudaMemcpyHostToDevice,
                           h->stream));
        CK(cudaEventRecord(g_staging.ev[slot], h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    *all_ok = bad.load() == 0;
    return 0;
}

// device -> host of a large array into pageable memory, through the same pinned buffers
int staged_download(H *h, double *dst, const double *d_src, int64_t count) {
    std::lock_guard<std::mutex> lock(g_staging_mu);
    if (!g_staging.init()) return fail(h, VBNMF_ERR_CUDA, "cannot allocate pinned staging buffers");
    const int64_t per = (int64_t)(Staging::kBytes / 8);
    const int64_t nch = (count + per - 1) / per;
    auto drain = [&](int64_t c) -> int {
        const int sl = (int)(c % Staging::kSlots);
        const int64_t lo = c * per, len = std::min(per, count - lo);
        CK(cudaEventSynchronize(g_staging.ev[sl]));
        const double *in = (const double *)g_staging.buf[sl];
        pool().run([&](int t, int nt) {
            const int64_t a = len * t / nt, b = len * (t + 1) / nt;
            memcpy(dst + lo + a, in + a, (size_t)(b - a) * 8);
        });
        return 0;
    };
    for (int64_t c = 0; c < nch; c++) {
        const int sl = (int)(c % Staging::kSlots);
        if (c >= Staging::kSlots) {  // the slot still holds chunk c - kSlots: move it out first
            int rc = drain(c - Staging::kSlots);
            if (rc) return rc;
        }
        const int64_t lo = c * per, len = std::min(per, count - lo);
        CK(cudaMemcpyAsync(g_staging.buf[sl], d_src + lo, (size_t)len * 8, cudaMemcpyDeviceToHost,
                           h->stream));
        CK(cudaEventRecord(g_staging.ev[sl], h->stream));
    }
    for (int64_t c = std::max<int64_t>(0, nch - Staging::kSlots); c < nch; c++) {
        int rc = drain(c);
        if (rc) return rc;
    }
    return 0;
}

int upload_panel(H *h, double *dst1, double *dst2, const double *src, bool wside, int r) {
    const Layout *L = h->L;
    const int64_t cnt = wside ? h->n : h->m;
    ScopedBufs B(h);
    double *d_raw = nullptr;
    CK(B.get(&d_raw, (size_t)cnt * r * 8));
    bool ok = true;
    int rc = staged_upload(h, d_raw, src, cnt * r, [](double v, double &o) { o = v; return true; },
                           &ok);
    if (rc) return rc;
    vb::scatter_panel_kernel<<<cdiv(cnt * r, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        cnt, r, h->rs, wside ? L->d_gene_dev : L->d_cell_dev, d_raw, wside, dst1, dst2, h->tsplit);
    return 0;
}

int init_common(H *h, int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail(h, VBNMF_ERR_CUDA, "no CUDA device available (libvbnmf has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(h, VBNMF_ERR_ARG, "bad device ordinal");
    h->device = device;
    CK(cudaSetDevice(device));
    // (cudaGetDeviceProperties fills ~100 fields and takes milliseconds; one attribute is enough)
    CK(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device));
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->own_stream = true;
    {   // Keep freed blocks in the device's default pool.  With a finite threshold a large
        // factorization (the layout build of a 2e9-nonzero matrix cycles through ~60 GB of
        // scratch) has the driver unmap and remap tens of GB at every synchronisation: measured
        // 2 s for ONE free and 3.5 s per layout build against 0.4 s of kernels.  Default: keep
        // everything (VBNMF_POOL_KEEP_GB sets a limit; vbnmf_trim_pool() returns the memory).
        cudaMemPool_t mp;
        if (cudaDeviceGetDefaultMemPool(&mp, device) == cudaSuccess) {
            const char *env = getenv("VBNMF_POOL_KEEP_GB");
            uint64_t keep = env ? (uint64_t)(atof(env) * 1073741824.0) : UINT64_MAX;
            cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    CK(vmalloc(h, &h->d_counters, 16 * sizeof(unsigned)));
    CK(cudaMemsetAsync(h->d_counters, 0, 16 * sizeof(unsigned), h->stream));
    CK(vmalloc(h, &h->d_ctl, vb::kCtlLen * sizeof(double)));
    CK(cudaMallocHost(&h->h_ctl, vb::kCtlLen * sizeof(double)));
    CK(cudaStreamSynchronize(h->stream));
    h->m_global = h->m;
    h->nnz_global = h->nnz;
    return 0;
}

// ---- handle creation ---------------------------------------------------------------------------
// the matrix one GPU holds: int32 row / column indices, fewer than 2^32-1 entries
int set_dims(H *h, int64_t n, int64_t m, int64_t nnz) {
    if (n > INT32_MAX || m > INT32_MAX)
        return fail(h, VBNMF_ERR_ARG, "n and m must be below 2^31 (int32 row/column indices)");
    if (nnz >= (int64_t)UINT32_MAX) return fail(h, VBNMF_ERR_ARG, "nnz per GPU must be < 2^32-1");
    h->n = n; h->m = m; h->nnz = nnz;
    return 0;
}

// the CSC arrays of h->nnz entries, after the scratch arena of the first layout build (the
// allocation order vbnmf_handle::d_arena explains); the values follow (store_values)
int alloc_csc(H *h) {
    CK(vmalloc(h, &h->d_arena, (size_t)std::max<int64_t>(h->nnz * 5, 4 * std::max(h->n, h->m)) * 4));
    CK(vmalloc(h, &h->d_colptr, (size_t)(h->m + 1) * 8));
    CK(vmalloc(h, &h->d_rowidx, (size_t)h->nnz * 4));
    return 0;
}

// The counts into h->d_val: fp32 when fill(float *dst, bool *exact) finds every one exactly
// representable, else fp64 through fill(double *dst, bool *exact).  The fp32 buffer is returned
// before the fp64 one is taken.
template <typename Fill>
int store_values(H *h, Fill &&fill) {
    ScopedBufs B(h);
    float *dv = nullptr;
    CK(B.get(&dv, (size_t)h->nnz * 4));
    bool exact = true;
    int rc = fill(dv, &exact);
    if (rc) return rc;
    h->val_float = exact;
    if (exact) {
        h->d_val = B.keep(dv);
        return 0;
    }
    B.free(dv);
    double *dd = nullptr;
    CK(B.get(&dd, (size_t)h->nnz * 8));
    if ((rc = fill(dd, &exact))) return rc;
    h->d_val = B.keep(dd);
    return 0;
}

// Every handle is made here.  check(h) validates the arguments and sets n, m, nnz without touching
// the device, so that a bad argument is reported as one on a machine without a GPU; fill(h) puts
// the count matrix on the device, which is then scanned.  On failure the error text is kept for
// vbnmf_last_error(NULL) and the handle is destroyed.  out = NULL: a temporary handle for a
// handle-free entry point (no matrix, no scan), destroyed when fill returns.
template <typename Check, typename Fill>
int create_handle(vbnmf_handle **out, int device, Check &&check, Fill &&fill) {
    H *h = new H();
    int rc = check(h);
    if (!rc) rc = init_common(h, device);
    if (!rc) rc = fill(h);
    if (!rc && out)
        rc = with_val_type(h->val_float, [h](auto v) { return scan_matrix_t<decltype(v)>(h); });
    if (rc || !out) {
        g_create_error = h->err;
        vbnmf_destroy(h);
        return rc;
    }
    *out = h;
    return 0;
}

// ---- vb_init(initializer = 'svd2' and 'svd') on the device (svd_init.cuh) ---------------------------

template <typename VT>
struct SvdCtx {
    H *h;
    int k;
    double *d_part = nullptr, *d_G = nullptr, *d_M = nullptr, *d_tmp = nullptr;
    int gblocks;
    // G (k x k, host) = A^T A summed over the rows of all shards
    int gram(const double *A, int64_t rows, std::vector<double> &G) {
        const int kk = k * k;
        vb::gram_part_kernel<<<gblocks, vb::kBlock, (size_t)vb::kGramRows * k * 8, h->stream>>>(
            rows, k, A, d_part);
        vb::gram_sum_kernel<<<cdiv(kk, vb::kBlock), vb::kBlock, 0, h->stream>>>(gblocks, kk, d_part, d_G);
        h->launches += 2;
        int rc = allreduce(h, d_G, kk);
        if (rc) return rc;
        G.resize((size_t)kk);
        CK(cudaMemcpyAsync(G.data(), d_G, (size_t)kk * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return 0;
    }
    // A <- A M (M k x kout on the host); d_tmp must hold rows x kout
    int right_mult(double *A, int64_t rows, const std::vector<double> &M, int kout, double *out) {
        CK(cudaMemcpyAsync(d_M, M.data(), (size_t)k * kout * 8, cudaMemcpyHostToDevice, h->stream));
        vb::right_mult_kernel<<<cdiv(rows * kout, vb::kBlock), vb::kBlock, 0, h->stream>>>(
            rows, k, kout, A, d_M, out);
        h->launches += 1;
        return 0;
    }
    // orthonormalise the columns of A (sum over all shards' rows): Cholesky-QR, twice
    int orth(double *A, int64_t rows, bool *ok) {
        std::vector<double> G, R, Ri;
        *ok = true;
        for (int pass = 0; pass < 2; pass++) {
            int rc = gram(A, rows, G);
            if (rc) return rc;
            if (!svdhost::cholesky_upper(k, G, R)) { *ok = false; return 0; }
            svdhost::invert_upper(k, R, Ri);
            if ((rc = right_mult(A, rows, Ri, k, d_tmp))) return rc;
            CK(cudaMemcpyAsync(A, d_tmp, (size_t)rows * k * 8, cudaMemcpyDeviceToDevice, h->stream));
        }
        return 0;
    }
    int xt(const double *Q, double *out) {  // out (m x k) = X^T Q
        vb::spmm_xt_kernel<VT><<<h->num_sms * 8, vb::kBlock, 0, h->stream>>>(
            h->m, k, h->d_colptr, h->d_rowidx, (const VT *)h->d_val, Q, out);
        h->launches += 1;
        return 0;
    }
    int x(const double *Z, double *Y) {     // Y (n x k) = X Z, summed over the shards
        CK(cudaMemsetAsync(Y, 0, (size_t)h->n * k * 8, h->stream));
        vb::spmm_x_kernel<VT><<<h->num_sms * 8, vb::kBlock, 0, h->stream>>>(
            h->m, k, h->d_colptr, h->d_rowidx, (const VT *)h->d_val, Z, Y);
        h->launches += 1;
        return allreduce(h, Y, h->n * (int64_t)k);
    }
};

// Rank-r truncated SVD of the resident matrix from a sketch of k columns, then
// finish(U, T, ok) while the buffers live: U (n x r) and T = V diag(d) (m x r, the local cells),
// both row-major on the device, components in decreasing order of d.  *ok = false when a Gram
// matrix is not positive definite (the sketch is rank-deficient).
template <typename VT, typename Finish>
int truncated_svd_t(H *h, int r, uint64_t seed, int64_t cell_offset, int k, int power_iters,
                    bool *ok, Finish &&finish) {
    const int64_t n = h->n, m = h->m, big = std::max(n, m);
    SvdCtx<VT> c;
    c.h = h; c.k = k;
    c.gblocks = h->num_sms * 2;
    ScopedBufs B(h);
    double *d_Y = nullptr, *d_Z = nullptr;
    CK(B.get(&d_Y, (size_t)n * k * 8));
    CK(B.get(&d_Z, (size_t)m * k * 8));
    CK(B.get(&c.d_tmp, (size_t)big * k * 8));
    CK(B.get(&c.d_part, (size_t)c.gblocks * k * k * 8));
    CK(B.get(&c.d_G, (size_t)k * k * 8));
    CK(B.get(&c.d_M, (size_t)k * k * 8));
    int rc;
    vb::gauss_fill_kernel<<<cdiv(m * k, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        m, k, (unsigned long long)seed, cell_offset, d_Z);
    h->launches += 1;
    if ((rc = c.x(d_Z, d_Y))) return rc;                 // Y = X Omega
    if ((rc = c.orth(d_Y, n, ok)) || !*ok) return rc;
    // subspace iteration Y <- X X^T Y, re-orthonormalised, until the r leading Ritz values
    // (eigenvalues of Y^T X X^T Y = gram(X^T Y)) stop moving: their error is the square of the
    // error of the vectors, so 1e-13 relative leaves the singular vectors good to ~1e-7
    std::vector<double> Gz, evz, Vz, prev;
    for (int q = 0; q < power_iters; q++) {
        if ((rc = c.xt(d_Y, d_Z))) return rc;
        if ((rc = c.gram(d_Z, m, Gz))) return rc;
        svdhost::jacobi_eigen(k, Gz, evz, Vz);
        bool conv = q >= 2 && !prev.empty();
        for (int a = 0; a < r && conv; a++)
            conv = std::fabs(evz[(size_t)a] - prev[(size_t)a]) <= 1e-13 * std::fabs(evz[(size_t)a]);
        prev = evz;
        if (conv) break;
        if ((rc = c.orth(d_Z, m, ok)) || !*ok) return rc;
        if ((rc = c.x(d_Z, d_Y))) return rc;
        if ((rc = c.orth(d_Y, n, ok)) || !*ok) return rc;
    }
    if ((rc = c.xt(d_Y, d_Z))) return rc;                // B^T = X^T Q  (m x k)
    std::vector<double> G, ev, V;
    if ((rc = c.gram(d_Z, m, G))) return rc;             // B B^T
    svdhost::jacobi_eigen(k, G, ev, V);                  // = U_B diag(d^2) U_B^T
    std::vector<double> M1((size_t)k * r);               // first r eigenvectors
    for (int a = 0; a < k; a++)
        for (int q = 0; q < r; q++) M1[(size_t)a * r + q] = V[(size_t)a * k + q];
    // U = Q U_B (n x r), T = B^T U_B = (diag(d) V^T)^T (m x r)
    double *d_U = c.d_tmp;
    if ((rc = c.right_mult(d_Y, n, M1, r, d_U))) return rc;
    double *d_T = nullptr;
    CK(B.get(&d_T, (size_t)m * r * 8));
    if ((rc = c.right_mult(d_Z, m, M1, r, d_T))) return rc;
    return finish(d_U, d_T, ok);
}

// 'svd2' from U and T: w = |U| / scale, h = |T| * scale, scale = bh / mean(|T|) over all cells
int svd2_finish(H *h, int r, double bh, const double *d_U, const double *d_T, bool *ok) {
    const Layout *L = h->L;
    const int64_t n = h->n, m = h->m;
    ScopedBufs B(h);
    double *d_sum = nullptr, *d_spart = nullptr;
    CK(B.get(&d_sum, 8));
    CK(B.get(&d_spart, (size_t)h->num_sms * 4 * 8));
    int rc;
    // scale <- bh / mean(h), h = |T|^T over all cells
    vb::abs_sum_kernel<<<h->num_sms * 4, vb::kBlock, 0, h->stream>>>(m * r, d_T, d_spart, d_sum,
                                                                   h->d_counters + 5);
    h->launches += 1;
    if ((rc = allreduce(h, d_sum, 1))) return rc;
    double sum = 0.0;
    CK(cudaMemcpyAsync(&sum, d_sum, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const double mean_h = sum / ((double)r * (double)h->m_global);
    if (!(mean_h > 0.0) || !std::isfinite(mean_h)) { *ok = false; return 0; }
    const double scale = bh / mean_h;                    // :156
    vb::svd_store_kernel<<<cdiv(n * r, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        n, r, h->rs, L->d_gene_dev, d_U, 1.0 / scale, h->d_lw, h->d_alw, h->tsplit);   // w / scale
    vb::svd_store_kernel<<<cdiv(m * r, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        m, r, h->rs, L->d_cell_dev, d_T, scale, h->d_lh, h->d_alh, h->tsplit);         // h * scale
    h->launches += 2;
    CK(cudaGetLastError());
    return 0;
}

// 'svd' from U and T (the rule of vbnmf_init_svd in vbnmf.h).  With v_k = T_k / d_k:
//   k = 0:  w = sgn' sqrt(d_0) u_0, h = sgn sqrt(d_0) v_0 = sgn T_0 / sqrt(d_0), sgn = sign(u_00),
//           sgn' = -1 if sgn < 0 else 1 (:120-124, literally);
//   k >= 1: P = |u+| |v+|, N = |u-| |v-|; s = -1 if N > P else 1; with the oriented pair
//           w = sqrt(d P) u+ / |u+| = sqrt(|T+| / |u+|) u+, h = sqrt(d P) v+ / |v+| = sqrt(|u+| / |T+|) T+
//           (d_k cancels: |v+| = |T+| / d_k).
// Only the 4r sums of squares, u_00 and the 4r factors cross the bus.
int svd_finish(H *h, int r, const double *d_U, const double *d_T, bool *ok) {
    const Layout *L = h->L;
    const int64_t n = h->n, m = h->m;
    const int nb = h->num_sms * 2;
    ScopedBufs B(h);
    double *d_part = nullptr, *d_sq = nullptr, *d_fs = nullptr;
    CK(B.get(&d_part, (size_t)nb * 2 * r * 8));
    CK(B.get(&d_sq, (size_t)4 * r * 8));           // U: (pos, neg) x r, then T: (pos, neg) x r
    CK(B.get(&d_fs, (size_t)4 * r * 8));           // f_w, s_w, f_h, s_h
    int rc;
    vb::signed_sq_part_kernel<<<nb, vb::kBlock, 0, h->stream>>>(n, r, d_U, d_part);
    vb::gram_sum_kernel<<<1, vb::kBlock, 0, h->stream>>>(nb, 2 * r, d_part, d_sq);
    vb::signed_sq_part_kernel<<<nb, vb::kBlock, 0, h->stream>>>(m, r, d_T, d_part);
    vb::gram_sum_kernel<<<1, vb::kBlock, 0, h->stream>>>(nb, 2 * r, d_part, d_sq + 2 * r);
    h->launches += 4;
    if ((rc = allreduce(h, d_sq + 2 * r, 2 * r))) return rc;   // T: sums over all cells
    std::vector<double> sq((size_t)4 * r), fs((size_t)4 * r);
    double u00 = 0.0;
    CK(cudaMemcpyAsync(sq.data(), d_sq, (size_t)4 * r * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&u00, d_U, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    double *fw = fs.data(), *sw = fw + r, *fh = sw + r, *sh = fh + r;
    const double d0 = std::sqrt(sq[2 * r] + sq[2 * r + 1]);   // |T_0| = d_0
    const double sgn = u00 > 0.0 ? 1.0 : (u00 < 0.0 ? -1.0 : 0.0);
    fw[0] = std::sqrt(d0);
    sw[0] = sgn < 0.0 ? -1.0 : 1.0;
    fh[0] = 1.0 / std::sqrt(d0);
    sh[0] = sgn;
    if (!(d0 > 0.0) || !std::isfinite(d0)) { *ok = false; return 0; }
    for (int q = 1; q < r; q++) {
        const double up = std::sqrt(sq[2 * q]), un = std::sqrt(sq[2 * q + 1]);
        const double tp = std::sqrt(sq[2 * r + 2 * q]), tn = std::sqrt(sq[2 * r + 2 * q + 1]);
        const bool flip = un * tn > up * tp;
        const double nu = flip ? un : up, nt = flip ? tn : tp;
        // P = N = 0 cannot happen for a nonnegative matrix and d_k > 0 (u^T X v would be <= 0)
        if (!(nu > 0.0 && nt > 0.0) || !std::isfinite(nu * nt)) { *ok = false; return 0; }
        fw[q] = std::sqrt(nt / nu);
        fh[q] = std::sqrt(nu / nt);
        sw[q] = sh[q] = flip ? -1.0 : 1.0;
    }
    CK(cudaMemcpyAsync(d_fs, fs.data(), (size_t)4 * r * 8, cudaMemcpyHostToDevice, h->stream));
    vb::svd_pos_store_kernel<<<cdiv(n * r, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        n, r, h->rs, L->d_gene_dev, d_U, d_fs, d_fs + r, h->d_lw, h->d_alw, h->tsplit);
    vb::svd_pos_store_kernel<<<cdiv(m * r, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        m, r, h->rs, L->d_cell_dev, d_T, d_fs + 2 * r, d_fs + 3 * r, h->d_lh, h->d_alh, h->tsplit);
    h->launches += 2;
    CK(cudaGetLastError());
    return 0;
}

// The two SVD initialisers: zeroed panels, the truncated SVD with oversampling 20 (a rank-deficient
// sketch, where Cholesky fails, falls back to none) and at most 60 subspace iterations, then
// finish(U, T, ok), the mirrors and rowSums(eh).
template <typename Finish>
int svd_init(H *h, int r, uint64_t seed, int64_t cell_offset, const char *name, Finish finish) {
    int rc;
    if ((rc = zeroed_panels(h, r))) return rc;
    const int kmax = (int)std::min<int64_t>(std::min(h->n, h->m_global), vb::kSvdMaxK);
    for (int k : {std::min(r + 20, kmax), r}) {
        bool ok = true;
        rc = with_val_type(h->val_float, [&](auto v) {
            return truncated_svd_t<decltype(v)>(h, r, seed, cell_offset, k, 60, &ok, finish);
        });
        if (rc) return rc;
        if (ok) return loaded_state(h);
    }
    return fail(h, VBNMF_ERR_ARG, std::string(name) + " initializer: the matrix has numerical rank below `rank`");
}

}  // namespace

// ---- cell / gene QC (qc.cuh) ---------------------------------------------------------------------
namespace {

// the kept entries of src into h's CSC (h->d_colptr already holds the new column pointers)
template <typename OT>
void launch_subset_compact(H *h, const H *src, const int32_t *d_cols, const int32_t *d_rowmap,
                           const double *d_scale, OT *out_val, unsigned *d_bad) {
    with_val_type(src->val_float, [&](auto v) {
        using VT = decltype(v);
        vb::qc_subset_compact_kernel<VT, OT><<<h->num_sms * 8, vb::kBlock, 0, h->stream>>>(
            h->m, d_cols, src->d_colptr, src->d_rowidx, (const VT *)src->d_val, d_rowmap,
            d_scale, h->d_colptr, h->d_rowidx, out_val, d_bad);
    });
}

}  // namespace

// ---- column shuffle (shuffle.cuh) ---------------------------------------------------------------
namespace {

// the shuffled CSC of src into h's arrays (h->d_colptr already holds src's column pointers)
template <typename VT>
int launch_shuffle(H *h, const H *src, uint64_t seed, unsigned *d_bad) {
    const int64_t per_warp = vb::shuffle_words(h->n) * 2 * 4;
    const int warps = (int)std::min<int64_t>(vb::kShuffleWarps, vb::kShuffleSmemMax / per_warp);
    const int smem = (int)(warps * per_warp);
    auto kern = vb::shuffle_columns_kernel<VT>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem));
    const int grid = (int)std::min<int64_t>((int64_t)h->num_sms * std::max(per_sm, 1),
                                            cdiv(h->m, warps));
    kern<<<grid, warps * 32, smem, h->stream>>>(h->n, h->m, seed, src->d_colptr,
                                                (const VT *)src->d_val, h->d_rowidx, (VT *)h->d_val,
                                                d_bad);
    h->launches += 1;
    CK(cudaGetLastError());
    return 0;
}

}  // namespace

// ---- consensus measures (consensus.cuh) ---------------------------------------------------------
namespace {

inline int64_t choose2(unsigned long long x) { return (int64_t)(x * (x - 1) / 2); }

// S1 = sum over runs t of sum_c C(n^t_c, 2) (the tables of the pairs (t, t) are diagonal);
// S2 = S1 + 2 sum_{t < u} sum_{c, c'} C(M^tu_cc', 2).  Pairs go in batches whose tables fit 256 MB.
int consensus_moments(H *h, int64_t m, int nrun, int K, const int32_t *d_lab, int64_t moments[2]) {
    const int KK = K * K;
    const int64_t npairs = (int64_t)nrun * (nrun + 1) / 2;
    std::vector<int32_t> pt, pu;
    for (int t = 0; t < nrun; t++)
        for (int u = t; u < nrun; u++) { pt.push_back(t); pu.push_back(u); }
    const int64_t batch = std::max<int64_t>(1, std::min<int64_t>({npairs, 65535,
                                                                 (256ll << 20) / ((int64_t)KK * 8)}));
    ScopedBufs B(h);
    int32_t *d_pt = nullptr, *d_pu = nullptr;
    unsigned long long *d_tab = nullptr;
    CK(B.get(&d_pt, (size_t)npairs * 4));
    CK(B.get(&d_pu, (size_t)npairs * 4));
    CK(B.get(&d_tab, (size_t)batch * KK * 8));
    CK(cudaMemcpyAsync(d_pt, pt.data(), (size_t)npairs * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d_pu, pu.data(), (size_t)npairs * 4, cudaMemcpyHostToDevice, h->stream));
    const int smem = KK * 4;
    CK(cudaFuncSetAttribute(vb::pair_contingency_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            std::max(smem, 1)));
    std::vector<unsigned long long> tab((size_t)batch * KK);
    int64_t s1 = 0, cross = 0;
    for (int64_t p0 = 0; p0 < npairs; p0 += batch) {
        const int64_t np = std::min(batch, npairs - p0);
        CK(cudaMemsetAsync(d_tab, 0, (size_t)np * KK * 8, h->stream));
        const int gx = (int)std::max<int64_t>(1, std::min<int64_t>(cdiv(m, vb::kBlock),
                                                                   cdiv(4 * h->num_sms, np)));
        vb::pair_contingency_kernel<<<dim3(gx, (unsigned)np), vb::kBlock, smem, h->stream>>>(
            m, nrun, K, d_lab, d_pt + p0, d_pu + p0, d_tab);
        h->launches += 1;
        CK(cudaGetLastError());
        CK(copy_sync(h, tab.data(), d_tab, (size_t)np * KK * 8, cudaMemcpyDeviceToHost));
        for (int64_t p = 0; p < np; p++) {
            int64_t sum = 0;
            for (int i = 0; i < KK; i++) sum += choose2(tab[(size_t)(p * KK + i)]);
            (pt[(size_t)(p0 + p)] == pu[(size_t)(p0 + p)] ? s1 : cross) += sum;
        }
    }
    moments[0] = s1;
    moments[1] = s1 + 2 * cross;
    return 0;
}

// Groups of cells with equal label tuples, in lexicographic order of (L[0], L[1], ...): their
// count G, sizes (G) and tuples (G x W words, 4 labels per word).  d_size / d_tup are allocated
// in the caller's scope `out`.
int consensus_groups(H *h, ScopedBufs &out, int64_t m, int nrun, int K, const int32_t *d_lab, int W,
                     int64_t *G_out, int64_t **d_size, uint32_t **d_tup) {
    cudaStream_t s = h->stream;
    ScopedBufs B(h);
    uint32_t *d_k0, *d_k1;
    int32_t *d_p0, *d_p1, *d_flag, *d_gid;
    CK(B.get(&d_k0, (size_t)m * 4));
    CK(B.get(&d_k1, (size_t)m * 4));
    CK(B.get(&d_p0, (size_t)m * 4));
    CK(B.get(&d_p1, (size_t)m * 4));
    int bits = 1;
    while ((1 << bits) < K) bits++;
    cub::DoubleBuffer<uint32_t> keys(d_k0, d_k1);
    cub::DoubleBuffer<int32_t> vals(d_p0, d_p1);
    size_t sort_bytes = 0, scan_bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, keys, vals, (int)m, 0, bits, s));
    CK(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, d_p0, d_p1, (int)m, s));
    void *d_tmp = nullptr;
    CK(B.get(&d_tmp, std::max(sort_bytes, scan_bytes)));
    std::vector<int32_t> iota((size_t)m);
    std::iota(iota.begin(), iota.end(), 0);
    CK(cudaMemcpyAsync(vals.Current(), iota.data(), (size_t)m * 4, cudaMemcpyHostToDevice, s));
    const int gm = cdiv(m, vb::kBlock);
    for (int t = nrun - 1; t >= 0; t--) {  // LSD: cub's radix sort is stable
        vb::group_gather_key_kernel<<<gm, vb::kBlock, 0, s>>>(m, d_lab + (int64_t)t * m,
                                                             vals.Current(), keys.Current());
        CK(cub::DeviceRadixSort::SortPairs(d_tmp, sort_bytes, keys, vals, (int)m, 0, bits, s));
        h->launches += 2;
    }
    const int32_t *d_perm = vals.Current();
    d_flag = (int32_t *)d_k0;  // the key buffers are free now
    d_gid = (int32_t *)d_k1;
    vb::group_flag_kernel<<<gm, vb::kBlock, 0, s>>>(m, nrun, d_lab, d_perm, d_flag);
    CK(cub::DeviceScan::InclusiveSum(d_tmp, scan_bytes, d_flag, d_gid, (int)m, s));
    int32_t G32 = 0;
    CK(copy_sync(h, &G32, d_gid + m - 1, 4, cudaMemcpyDeviceToHost));
    const int64_t G = G32;
    int64_t *d_start;
    CK(B.get(&d_start, (size_t)G * 8));
    CK(out.get(d_size, (size_t)G * 8));
    CK(out.get(d_tup, (size_t)G * W * 4));
    vb::group_start_kernel<<<gm, vb::kBlock, 0, s>>>(m, nrun, W, d_lab, d_perm, d_flag, d_gid,
                                                     d_start, *d_tup);
    vb::group_size_kernel<<<cdiv(G, vb::kBlock), vb::kBlock, 0, s>>>(G, m, d_start, *d_size);
    h->launches += 4;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s));
    *G_out = G;
    return 0;
}

// bytes the pool can still hand out: the driver's free memory plus what the pool keeps cached
size_t device_bytes_available(H *h) {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return 0;
    cudaMemPool_t mp;
    uint64_t reserved = 0, used = 0;
    if (cudaDeviceGetDefaultMemPool(&mp, h->device) == cudaSuccess &&
        cudaMemPoolGetAttribute(mp, cudaMemPoolAttrReservedMemCurrent, &reserved) == cudaSuccess &&
        cudaMemPoolGetAttribute(mp, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess &&
        reserved > used)
        free_b += (size_t)(reserved - used);
    return free_b;
}

// the packed IP triangle, the row cache and the merge loop; merges (G - 1) x 5 on the host
int consensus_tree(H *h, int64_t G, int nrun, int W, const int64_t *d_size0, const uint32_t *d_tup,
                   int64_t *merges, int64_t *rescans) {
    cudaStream_t s = h->stream;
    ScopedBufs B(h);
    vb::MergeArgs A;
    A.G = G;
    A.nrun = nrun;
    const int64_t ntri = G * (G - 1) / 2;
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, vb::merge_loop_kernel, vb::kMergeBlock, 0));
    const int grid = h->num_sms * std::max(per_sm, 1);
    CK(B.get(&A.ip, (size_t)ntri * 8));
    CK(B.get(&A.size, (size_t)G * 8));
    CK(B.get(&A.bq, (size_t)G * 8));
    CK(B.get(&A.bb, (size_t)G * 4));
    CK(B.get(&A.merges, (size_t)(G - 1) * 5 * 8));
    CK(B.get(&A.resc, (size_t)G * 4));
    CK(B.get(&A.nresc, 16));
    CK(B.get(&A.part_q, (size_t)grid * 8));
    CK(B.get(&A.part_a, (size_t)grid * 8));
    CK(B.get(&A.rescans, 8));
    CK(cudaMemcpyAsync(A.size, d_size0, (size_t)G * 8, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemsetAsync(A.rescans, 0, 8, s));
    const int pad = 4 * W - nrun;
    const dim3 fill_grid(cdiv(G, 64), (unsigned)std::min<int64_t>(cdiv(G, 4), 65535));
    vb::ip_fill_kernel<<<fill_grid, vb::kBlock, 0, s>>>(G, W, pad, d_tup, A.size, A.ip);
    vb::row_best_kernel<<<(int)std::min<int64_t>(G, 1 << 20), vb::kMergeBlock, 0, s>>>(
        G, nrun, A.ip, A.size, A.bq, A.bb);
    h->launches += 2;
    CK(cudaGetLastError());
    void *args[] = {&A};
    CK(cudaLaunchCooperativeKernel((void *)vb::merge_loop_kernel, grid, vb::kMergeBlock, args, 0, s));
    h->launches += 1;
    CK(cudaMemcpyAsync(merges, A.merges, (size_t)(G - 1) * 5 * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(rescans, A.rescans, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    return 0;
}

}  // namespace

extern "C" {

const char *vbnmf_last_error(const vbnmf_handle *h) {
    return h ? h->err.c_str() : g_create_error.c_str();
}

void vbnmf_destroy(vbnmf_handle *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    free_panels(h);
    drop_layouts(h);
    if (!h->borrowed) {
        vfree(h->stream, h->d_colptr); vfree(h->stream, h->d_rowidx); vfree(h->stream, h->d_val);
    }
    vfree(h->stream, h->d_arena);
    vfree(h->stream, h->d_cnt);
    vfree(h->stream, h->d_counters);
    vfree(h->stream, h->d_ctl);
    if (h->h_ctl) cudaFreeHost(h->h_ctl);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int vbnmf_set_host_threads(int nthreads) {
    if (nthreads < 1) return VBNMF_ERR_ARG;
    pool().set_threads(nthreads);
    return 0;
}

int vbnmf_trim_pool(int device) {
    cudaMemPool_t mp;
    if (cudaSetDevice(device) != cudaSuccess) return VBNMF_ERR_CUDA;
    if (cudaDeviceSynchronize() != cudaSuccess) return VBNMF_ERR_CUDA;
    if (cudaDeviceGetDefaultMemPool(&mp, device) != cudaSuccess) return VBNMF_ERR_CUDA;
    return cudaMemPoolTrimTo(mp, 0) == cudaSuccess ? 0 : VBNMF_ERR_CUDA;
}

int vbnmf_create(vbnmf_handle **out, int64_t n, int64_t m, int64_t nnz, const int32_t *colptr32,
                 const int64_t *colptr64, const int32_t *rowidx, const double *values, int device) {
    if (!out) return VBNMF_ERR_ARG;
    *out = nullptr;
    StageTimer tm("vbnmf_create(total)");
    auto check = [&](H *h) -> int {
        if (n <= 0 || m <= 0 || nnz <= 0 || (!colptr32 == !colptr64) || !rowidx || !values)
            return fail(h, VBNMF_ERR_ARG, "vbnmf_create: bad arguments");
        return set_dims(h, n, m, nnz);
    };
    return create_handle(out, device, check, [&](H *h) -> int {
        StageTimer tu("  upload (staged, pinned)");
        int rc = alloc_csc(h);
        if (rc) return rc;
        // column pointers: widened to 64 bits and checked on the way (first = 0, last = nnz,
        // non-decreasing: element j is compared with element j + 1, which the caller's array holds)
        auto colptr_up = [&](const auto *cp) -> int {
            if (cp[0] != 0 || (int64_t)cp[m] != nnz) return fail(h, VBNMF_ERR_ARG, "colptr does not span nnz");
            bool ok = true;
            int rc2 = staged_upload(h, h->d_colptr, cp, m + 1,
                                    [](const auto &v, int64_t &o) { o = v; return true; }, &ok);
            if (rc2) return rc2;
            std::atomic<int> unsorted{0};
            pool().run([&](int t, int nt) {
                bool g = true;
                for (int64_t j = m * t / nt; j < m * (t + 1) / nt; j++) g &= cp[j] <= cp[j + 1];
                if (!g) unsorted.store(1);
            });
            return unsorted.load() ? fail(h, VBNMF_ERR_ARG, "colptr is not non-decreasing") : 0;
        };
        if ((rc = colptr64 ? colptr_up(colptr64) : colptr_up(colptr32))) return rc;
        // row indices: plain copy, range-checked on the device (scan_matrix)
        bool ok = true;
        rc = staged_upload(h, h->d_rowidx, rowidx, nnz,
                           [](int32_t v, int32_t &o) { o = v; return true; }, &ok);
        if (rc) return rc;
        // NaN compares unequal: it takes the fp64 path and is refused by scan_matrix
        return store_values(h, [&](auto *dv, bool *exact) {
            using VT = std::remove_pointer_t<decltype(dv)>;
            return staged_upload(h, dv, values, nnz, [](double v, VT &o) {
                o = (VT)v;
                return sizeof(VT) == 8 || (double)o == v;
            }, exact);
        });
    });
}

int vbnmf_create_from_device(vbnmf_handle **out, int64_t n, int64_t m, int64_t nnz,
                             const int64_t *d_colptr, const int32_t *d_rowidx, const float *d_values,
                             int device) {
    if (!out) return VBNMF_ERR_ARG;
    *out = nullptr;
    auto check = [&](H *h) -> int {
        if (n <= 0 || m <= 0 || nnz <= 0 || !d_colptr || !d_rowidx || !d_values)
            return fail(h, VBNMF_ERR_ARG, "vbnmf_create_from_device: bad arguments");
        return set_dims(h, n, m, nnz);
    };
    return create_handle(out, device, check, [&](H *h) -> int {
        h->borrowed = true;
        h->val_float = true;
        h->d_colptr = const_cast<int64_t *>(d_colptr);
        h->d_rowidx = const_cast<int32_t *>(d_rowidx);
        h->d_val = const_cast<float *>(d_values);
        return 0;
    });
}

int vbnmf_create_from_mtx(vbnmf_handle **out, const char *path, int device, int64_t dims[3]) {
    if (!out || !path) return VBNMF_ERR_ARG;
    *out = nullptr;
    StageTimer tm("vbnmf_create_from_mtx(total)");
    std::unique_ptr<FILE, int (*)(FILE *)> file(nullptr, fclose);
    int64_t nbytes = 0;
    // header (host): banner, comments, the size line
    auto check = [&](H *h) -> int {
        FILE *fp = fopen(path, "rb");
        if (!fp) return fail(h, VBNMF_ERR_ARG, std::string("cannot open ") + path);
        file.reset(fp);
        char line[1024];
        if (!fgets(line, sizeof(line), fp) || strncmp(line, "%%MatrixMarket", 14) != 0)
            return fail(h, VBNMF_ERR_ARG, "not a MatrixMarket file");
        std::string banner(line);
        for (auto &ch : banner) ch = (char)tolower((unsigned char)ch);
        if (banner.find("matrix") == std::string::npos || banner.find("coordinate") == std::string::npos ||
            banner.find("general") == std::string::npos ||
            (banner.find("real") == std::string::npos && banner.find("integer") == std::string::npos))
            return fail(h, VBNMF_ERR_ARG,
                        "MatrixMarket: only 'matrix coordinate real|integer general' is supported");
        long long n = 0, m = 0, nnz = 0;
        for (;;) {
            if (!fgets(line, sizeof(line), fp))
                return fail(h, VBNMF_ERR_ARG, "MatrixMarket: missing size line");
            if (line[0] == '%' || line[0] == '\n' || line[0] == '\r') continue;
            if (sscanf(line, "%lld %lld %lld", &n, &m, &nnz) != 3)
                return fail(h, VBNMF_ERR_ARG, "MatrixMarket: malformed size line");
            break;
        }
        if (n <= 0 || m <= 0 || nnz <= 0 || set_dims(h, n, m, nnz))
            return fail(h, VBNMF_ERR_ARG, "MatrixMarket: dimensions out of range");
        const long off = ftell(fp);
        fseek(fp, 0, SEEK_END);
        nbytes = (int64_t)ftell(fp) - off;
        fseek(fp, off, SEEK_SET);
        if (nbytes <= 0) return fail(h, VBNMF_ERR_ARG, "MatrixMarket: no entries");
        return 0;
    };
    const int rc = create_handle(out, device, check, [&](H *h) -> int {
        const int64_t n = h->n, m = h->m, nnz = h->nnz;
        ScopedBufs B(h);
        char *d_buf = nullptr;
        uint8_t *d_flag = nullptr;
        int64_t *d_start = nullptr, *d_num = nullptr;
        unsigned long long *d_key = nullptr, *d_key2 = nullptr;
        double *d_v = nullptr, *d_v2 = nullptr;
        unsigned *d_bad = nullptr;
        void *d_tmp = nullptr;
        CK(B.get(&d_buf, (size_t)nbytes));
        {   // file bytes -> device through the pinned staging buffers
            std::lock_guard<std::mutex> lock(g_staging_mu);
            if (!g_staging.init()) return fail(h, VBNMF_ERR_CUDA, "cannot allocate pinned staging buffers");
            int slot = 0;
            for (int64_t lo = 0; lo < nbytes; lo += (int64_t)Staging::kBytes, slot = (slot + 1) % Staging::kSlots) {
                const size_t len = (size_t)std::min<int64_t>((int64_t)Staging::kBytes, nbytes - lo);
                CK(cudaEventSynchronize(g_staging.ev[slot]));
                if (fread(g_staging.buf[slot], 1, len, file.get()) != len)
                    return fail(h, VBNMF_ERR_ARG, "MatrixMarket: short read");
                CK(cudaMemcpyAsync(d_buf + lo, g_staging.buf[slot], len, cudaMemcpyHostToDevice, h->stream));
                CK(cudaEventRecord(g_staging.ev[slot], h->stream));
            }
            CK(cudaStreamSynchronize(h->stream));
        }
        file.reset();
        // line starts
        CK(B.get(&d_flag, (size_t)nbytes));
        CK(B.get(&d_start, (size_t)(nnz + 1) * 8));
        CK(B.get(&d_num, 8));
        CK(B.get(&d_bad, 4 * sizeof(unsigned)));
        CK(cudaMemsetAsync(d_bad, 0, 4 * sizeof(unsigned), h->stream));
        vb::mtx_line_flags_kernel<<<h->num_sms * 8, vb::kBlock, 0, h->stream>>>(nbytes, d_buf, d_flag);
        // count first (the output must not overflow when the file has more lines than declared)
        size_t tb = 0;
        cub::CountingInputIterator<int64_t> iota(0);
        int64_t *d_cnt = d_num;
        CK(cub::DeviceReduce::Sum(nullptr, tb, d_flag, d_cnt, nbytes, h->stream));
        CK(B.get(&d_tmp, tb));
        CK(cub::DeviceReduce::Sum(d_tmp, tb, d_flag, d_cnt, nbytes, h->stream));
        int64_t nlines = 0;
        CK(cudaMemcpyAsync(&nlines, d_cnt, 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        B.free(d_tmp);
        if (nlines != nnz)
            return fail(h, VBNMF_ERR_ARG, "MatrixMarket: number of entry lines differs from the size line");
        CK(cub::DeviceSelect::Flagged(nullptr, tb, iota, d_flag, d_start, d_num, nbytes, h->stream));
        CK(B.get(&d_tmp, tb));
        CK(cub::DeviceSelect::Flagged(d_tmp, tb, iota, d_flag, d_start, d_num, nbytes, h->stream));
        B.free(d_tmp);
        // parse, sort by (column, row)
        CK(B.get(&d_key, (size_t)nnz * 8));
        CK(B.get(&d_key2, (size_t)nnz * 8));
        CK(B.get(&d_v, (size_t)nnz * 8));
        CK(B.get(&d_v2, (size_t)nnz * 8));
        vb::mtx_parse_kernel<<<cdiv(nnz, vb::kBlock), vb::kBlock, 0, h->stream>>>(
            nnz, nbytes, d_buf, d_start, n, m, d_key, d_v, d_bad);
        int cbits = 1;
        while ((1ll << cbits) < m) cbits++;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, d_key, d_key2, d_v, d_v2, nnz, 0, 32 + cbits, h->stream));
        CK(B.get(&d_tmp, tb));
        CK(cub::DeviceRadixSort::SortPairs(d_tmp, tb, d_key, d_key2, d_v, d_v2, nnz, 0, 32 + cbits, h->stream));
        int rc = alloc_csc(h);
        if (rc) return rc;
        vb::mtx_colptr_kernel<<<cdiv(m + 1, vb::kBlock), vb::kBlock, 0, h->stream>>>(m, nnz, d_key2,
                                                                                   h->d_colptr);
        // the fp32 pass also flags malformed lines and duplicates; the fp64 pass writes its flags
        // apart, from d_bad + 3
        return store_values(h, [&](auto *dv, bool *exact) -> int {
            using VT = std::remove_pointer_t<decltype(dv)>;
            vb::mtx_unpack_kernel<VT><<<cdiv(nnz, vb::kBlock), vb::kBlock, 0, h->stream>>>(
                nnz, d_key2, d_v2, h->d_rowidx, dv, sizeof(VT) == 4 ? d_bad : d_bad + 3);
            unsigned bad[4];
            CK(cudaMemcpyAsync(bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            CK(cudaGetLastError());
            if (bad[0]) return fail(h, VBNMF_ERR_ARG, "MatrixMarket: malformed entry line or index out of range");
            if (bad[1]) return fail(h, VBNMF_ERR_ARG, "MatrixMarket: duplicate entries");
            *exact = !bad[2];
            return 0;
        });
    });
    if (!rc && dims) { dims[0] = (*out)->n; dims[1] = (*out)->m; dims[2] = (*out)->nnz; }
    return rc;
}

/* the CSC arrays a handle holds, back on the host (colptr m+1 int64, rowidx nnz int32, values nnz
 * doubles; any may be NULL) */
int vbnmf_get_csc(vbnmf_handle *h, int64_t *colptr, int32_t *rowidx, double *values) {
    if (!h) return VBNMF_ERR_ARG;
    CK(cudaSetDevice(h->device));
    if (colptr) CK(cudaMemcpyAsync(colptr, h->d_colptr, (size_t)(h->m + 1) * 8, cudaMemcpyDeviceToHost, h->stream));
    if (rowidx) CK(cudaMemcpyAsync(rowidx, h->d_rowidx, (size_t)h->nnz * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (values) {
        if (h->val_float) {
            std::vector<float> tmp((size_t)h->nnz);
            CK(copy_sync(h, tmp.data(), h->d_val, (size_t)h->nnz * 4, cudaMemcpyDeviceToHost));
            for (int64_t t = 0; t < h->nnz; t++) values[t] = (double)tmp[(size_t)t];
        } else {
            CK(copy_sync(h, values, h->d_val, (size_t)h->nnz * 8, cudaMemcpyDeviceToHost));
        }
    }
    return 0;
}

int vbnmf_qc_stats(vbnmf_handle *h, double *cell_sum, double *gene_sum, double *gene_sumsq,
                   int64_t *gene_cells, int64_t *cell_genes) {
    if (!h) return VBNMF_ERR_ARG;
    if (h->nranks > 1)
        return fail(h, VBNMF_ERR_STATE, "vbnmf_qc_stats: the handle holds one shard of the cells "
                                        "(vbnmf_attach_comm); its gene statistics would be partial");
    CK(cudaSetDevice(h->device));
    const int64_t n = h->n, m = h->m;
    if (cell_sum || gene_sum || gene_sumsq) {
        ScopedBufs B(h);
        double *d = nullptr;  // [cell_sum m | gene_sum n | gene_sumsq n]
        CK(B.get(&d, (size_t)(m + 2 * n) * 8));
        CK(cudaMemsetAsync(d + m, 0, (size_t)2 * n * 8, h->stream));
        with_val_type(h->val_float, [&](auto v) {
            using VT = decltype(v);
            vb::qc_stats_kernel<VT><<<h->num_sms * 8, vb::kBlock, 0, h->stream>>>(
                m, h->d_colptr, h->d_rowidx, (const VT *)h->d_val, d, d + m, d + m + n);
        });
        CK(cudaGetLastError());
        if (cell_sum) CK(cudaMemcpyAsync(cell_sum, d, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
        if (gene_sum) CK(cudaMemcpyAsync(gene_sum, d + m, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
        if (gene_sumsq)
            CK(cudaMemcpyAsync(gene_sumsq, d + m + n, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    // entries with a non-zero value: the counts scan_matrix keeps on the device
    static_assert(sizeof(unsigned long long) == sizeof(int64_t), "d_cnt is copied as int64");
    if (gene_cells) CK(cudaMemcpyAsync(gene_cells, h->d_cnt, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    if (cell_genes) CK(cudaMemcpyAsync(cell_genes, h->d_cnt + n, (size_t)m * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int vbnmf_create_subset(vbnmf_handle **out, vbnmf_handle *src, const uint8_t *keep_rows,
                        const uint8_t *keep_cols, const double *col_scale) {
    if (!out) return VBNMF_ERR_ARG;
    *out = nullptr;
    StageTimer tm("vbnmf_create_subset(total)");
    auto check = [&](H *h) -> int {
        if (!src || !keep_rows || !keep_cols)
            return fail(h, VBNMF_ERR_ARG, "vbnmf_create_subset: bad arguments");
        // the gene statistics and the empty-gene test of one shard are partial: refused, not guessed
        if (src->nranks > 1)
            return fail(h, VBNMF_ERR_STATE, "vbnmf_create_subset: the source holds one shard of "
                                            "the cells (vbnmf_attach_comm)");
        int64_t n = 0, m = 0;
        for (int64_t i = 0; i < src->n; i++) n += keep_rows[i] != 0;
        for (int64_t j = 0; j < src->m; j++) m += keep_cols[j] != 0;
        if (n == 0 || m == 0)
            return fail(h, VBNMF_ERR_ARG, "vbnmf_create_subset: no rows or no columns selected");
        h->n = n; h->m = m;
        return 0;
    };
    return create_handle(out, src ? src->device : 0, check, [&](H *h) -> int {
        const int64_t n0 = src->n, m0 = src->m, m = h->m;
        ScopedBufs B(h);
        uint8_t *d_mask = nullptr;  // [rows n0 | columns m0]
        double *d_scale = nullptr;
        int32_t *d_rowmap = nullptr, *d_cols = nullptr, *d_nsel = nullptr;
        int64_t *d_ptr = nullptr;
        unsigned *d_bad = nullptr;
        void *d_tmp = nullptr;
        // src's arrays are read on this handle's stream: src's own work on them must be complete
        CK(cudaStreamSynchronize(src->stream));
        cudaStream_t s = h->stream;
        CK(B.get(&d_mask, (size_t)(n0 + m0)));
        CK(cudaMemcpyAsync(d_mask, keep_rows, (size_t)n0, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(d_mask + n0, keep_cols, (size_t)m0, cudaMemcpyHostToDevice, s));
        if (col_scale) {
            CK(B.get(&d_scale, (size_t)m0 * 8));
            CK(cudaMemcpyAsync(d_scale, col_scale, (size_t)m0 * 8, cudaMemcpyHostToDevice, s));
        }
        CK(B.get(&d_rowmap, (size_t)n0 * 4));
        CK(B.get(&d_cols, (size_t)m * 4));
        CK(B.get(&d_nsel, 4));
        CK(B.get(&d_ptr, (size_t)(m + 1) * 8));
        cub::CountingInputIterator<int32_t> iota(0);
        size_t tb1 = 0, tb2 = 0, tb3 = 0;
        CK(cub::DeviceScan::ExclusiveSum(nullptr, tb1, d_rowmap, d_rowmap, n0, s));
        CK(cub::DeviceSelect::Flagged(nullptr, tb2, iota, d_mask + n0, d_cols, d_nsel, m0, s));
        CK(cub::DeviceScan::ExclusiveSum(nullptr, tb3, d_ptr, d_ptr, m + 1, s));
        CK(B.get(&d_tmp, std::max(tb1, std::max(tb2, tb3))));
        // kept rows renumbered in order (exclusive scan of the row mask), dropped rows -> -1
        vb::qc_mask_kernel<<<cdiv(n0, vb::kBlock), vb::kBlock, 0, s>>>(n0, d_mask, d_rowmap);
        CK(cub::DeviceScan::ExclusiveSum(d_tmp, tb1, d_rowmap, d_rowmap, n0, s));
        vb::qc_rowmap_kernel<<<cdiv(n0, vb::kBlock), vb::kBlock, 0, s>>>(n0, d_mask, d_rowmap);
        // kept columns in order; per kept column its kept entries; the scan gives the new colptr
        CK(cub::DeviceSelect::Flagged(d_tmp, tb2, iota, d_mask + n0, d_cols, d_nsel, m0, s));
        vb::qc_subset_count_kernel<<<h->num_sms * 8, vb::kBlock, 0, s>>>(
            m, d_cols, src->d_colptr, src->d_rowidx, d_rowmap, d_ptr);
        CK(cudaMemsetAsync(d_ptr + m, 0, 8, s));
        CK(cub::DeviceScan::ExclusiveSum(d_tmp, tb3, d_ptr, d_ptr, m + 1, s));
        int64_t nnz = 0;
        CK(cudaMemcpyAsync(&nnz, d_ptr + m, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        if (nnz == 0) return fail(h, VBNMF_ERR_ARG, "vbnmf_create_subset: the selection holds no entries");
        h->nnz = h->nnz_global = nnz;
        int rc = alloc_csc(h);
        if (rc) return rc;
        CK(cudaMemcpyAsync(h->d_colptr, d_ptr, (size_t)(m + 1) * 8, cudaMemcpyDeviceToDevice, s));
        CK(B.get(&d_bad, 4));
        CK(cudaMemsetAsync(d_bad, 0, 4, s));
        // the kept (scaled) values
        return store_values(h, [&](auto *dv, bool *exact) -> int {
            launch_subset_compact(h, src, d_cols, d_rowmap, d_scale, dv, d_bad);
            unsigned bad = 0;
            CK(copy_sync(h, &bad, d_bad, 4, cudaMemcpyDeviceToHost));
            CK(cudaGetLastError());
            *exact = !bad;
            return 0;
        });
    });
}

int vbnmf_create_shuffled(vbnmf_handle **out, vbnmf_handle *src, uint64_t seed) {
    if (!out) return VBNMF_ERR_ARG;
    *out = nullptr;
    StageTimer tm("vbnmf_create_shuffled(total)");
    auto check = [&](H *h) -> int {
        if (!src) return fail(h, VBNMF_ERR_ARG, "vbnmf_create_shuffled: bad arguments");
        // the draw is keyed by the column index: a shard would need its global column offset
        if (src->nranks > 1)
            return fail(h, VBNMF_ERR_STATE, "vbnmf_create_shuffled: the source holds one shard of "
                                            "the cells (vbnmf_attach_comm)");
        if (src->n > vb::kShuffleMaxRows)
            return fail(h, VBNMF_ERR_ARG,
                        "vbnmf_create_shuffled: n = " + std::to_string(src->n) + " rows; at most " +
                            std::to_string(vb::kShuffleMaxRows) +
                            " (a column's row bitmap must fit one CTA's shared memory)");
        h->n = src->n; h->m = src->m; h->nnz = src->nnz;
        h->val_float = src->val_float;
        return 0;
    };
    return create_handle(out, src ? src->device : 0, check, [&](H *h) -> int {
        int optin = 0;
        CK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
        if (optin < vb::shuffle_words(h->n) * 2 * 4)
            return fail(h, VBNMF_ERR_ARG, "vbnmf_create_shuffled: the row bitmap of a column does "
                                          "not fit this device's shared memory");
        // src's arrays are read on this handle's stream: src's own work on them must be complete
        CK(cudaStreamSynchronize(src->stream));
        cudaStream_t s = h->stream;
        int rc = alloc_csc(h);
        if (rc) return rc;
        CK(cudaMemcpyAsync(h->d_colptr, src->d_colptr, (size_t)(h->m + 1) * 8,
                           cudaMemcpyDeviceToDevice, s));
        CK(vmalloc(h, &h->d_val, (size_t)h->nnz * (h->val_float ? 4 : 8)));
        ScopedBufs B(h);
        unsigned *d_bad = nullptr;
        CK(B.get(&d_bad, 4));
        CK(cudaMemsetAsync(d_bad, 0, 4, s));
        rc = with_val_type(h->val_float, [&](auto v) {
            return launch_shuffle<decltype(v)>(h, src, seed, d_bad);
        });
        if (rc) return rc;
        unsigned bad = 0;
        CK(copy_sync(h, &bad, d_bad, 4, cudaMemcpyDeviceToHost));
        CK(cudaGetLastError());
        if (bad)
            return fail(h, VBNMF_ERR_ARG, "vbnmf_create_shuffled: a column holds more entries than "
                                          "there are rows (repeated entries)");
        return 0;
    });
}

int vbnmf_consensus(int device, int64_t m, int nrun, int nlabels, const int32_t *labels,
                    int64_t max_groups, int64_t moments[2], int64_t *ngroups, int64_t *merges,
                    int64_t merge_cap, int64_t *rescans) {
    auto arg = [](H *h, const std::string &msg) {
        return fail(h, VBNMF_ERR_ARG, "vbnmf_consensus: " + msg);
    };
    if (ngroups) *ngroups = 0;
    if (rescans) *rescans = 0;
    auto check = [&](H *h) -> int {
        if (!labels || !moments || (merges && (!ngroups || !rescans)))
            return arg(h, "labels and moments are required, ngroups and rescans with merges");
        if (nrun < 1 || m < 1 || m > INT32_MAX) return arg(h, "needs nrun >= 1 and 1 <= m < 2^31");
        if (nlabels < 1 || nlabels > vb::kConsensusMaxLabels)
            return arg(h, "nlabels = " + std::to_string(nlabels) + "; 1 ... " +
                              std::to_string(vb::kConsensusMaxLabels) +
                              " (a K x K table of counters must fit one CTA's shared memory)");
        const unsigned __int128 half = (unsigned __int128)((m + 1) / 2);
        if ((unsigned __int128)nrun * half * half >= ((unsigned __int128)1 << 53))
            return arg(h, "nrun * ceil(m / 2)^2 must be below 2^53 (exact IP values and their fp64 ratios)");
        for (int64_t i = 0; i < (int64_t)nrun * m; i++)
            if (labels[i] < 0 || labels[i] >= nlabels)
                return arg(h, "label " + std::to_string(labels[i]) + " outside 0 ... nlabels - 1");
        return 0;
    };
    return create_handle(nullptr, device, check, [&](H *h) -> int {
        StageTimer tm("vbnmf_consensus(total)");
        const int W = (nrun + 3) / 4;
        ScopedBufs B(h);
        int32_t *d_lab = nullptr;
        CK(B.get(&d_lab, (size_t)nrun * m * 4));
        CK(cudaMemcpyAsync(d_lab, labels, (size_t)nrun * m * 4, cudaMemcpyHostToDevice, h->stream));
        int rc = consensus_moments(h, m, nrun, nlabels, d_lab, moments);
        if (rc || !merges) return rc;
        int64_t G = 0, *d_size = nullptr;
        uint32_t *d_tup = nullptr;
        if ((rc = consensus_groups(h, B, m, nrun, nlabels, d_lab, W, &G, &d_size, &d_tup))) return rc;
        B.free(d_lab);
        *ngroups = G;
        if (merge_cap < G - 1)
            return fail(h, VBNMF_ERR_ARG, "vbnmf_consensus: merge_cap = " + std::to_string(merge_cap) +
                                              " below G - 1 = " + std::to_string(G - 1));
        if (G <= 1) return 0;
        // the triangle, the row cache, the merge list and the sizes; 256 MB left for the rest
        const double need = 8.0 * G * (G - 1) / 2 + 64.0 * G + (256 << 20);
        if (max_groups > 0 && G > max_groups)
            return fail(h, VBNMF_ERR_MEMORY, "vbnmf_consensus: G = " + std::to_string(G) +
                                                 " groups above max_groups = " + std::to_string(max_groups));
        if (cudaStreamSynchronize(h->stream) != cudaSuccess || need > (double)device_bytes_available(h))
            return fail(h, VBNMF_ERR_MEMORY, "vbnmf_consensus: G = " + std::to_string(G) + " groups need " +
                                                 std::to_string((int64_t)(need / 1e9)) +
                                                 " GB of device memory for the IP triangle");
        return consensus_tree(h, G, nrun, W, d_size, d_tup, merges, rescans);
    });
}

int vbnmf_set_precision(vbnmf_handle *h, int precision) {
    if (!h) return VBNMF_ERR_ARG;
    if (precision != VBNMF_FP64 && precision != VBNMF_FP32_STORAGE)
        return fail(h, VBNMF_ERR_ARG, "precision must be VBNMF_FP64 or VBNMF_FP32_STORAGE");
    if (precision != h->precision) {
        h->precision = precision;  // takes effect at the next vbnmf_set_state / mlnmf_run
        h->stats_valid = false;
    }
    return 0;
}

int vbnmf_set_stream(vbnmf_handle *h, void *cuda_stream) {
    if (!h) return VBNMF_ERR_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->own_stream) cudaStreamDestroy(h->stream);
    h->stream = (cudaStream_t)cuda_stream;
    h->own_stream = false;
    return 0;
}

int vbnmf_nccl_unique_id(void *uid128) {
    std::string err;
    if (!uid128 || !g_nccl.load(err)) { g_create_error = err; return VBNMF_ERR_NCCL; }
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) return VBNMF_ERR_NCCL;
    static_assert(sizeof(id) == 128, "ncclUniqueId is 128 bytes");
    memcpy(uid128, &id, 128);
    return 0;
}

int vbnmf_comm_create(vbnmf_comm **out, int nranks, int rank, const void *uid128, int device) {
    if (!out || nranks < 1 || rank < 0 || rank >= nranks || !uid128) return VBNMF_ERR_ARG;
    *out = nullptr;
    if (!g_nccl.load(g_create_error)) return VBNMF_ERR_NCCL;
    if (cudaSetDevice(device) != cudaSuccess) {
        g_create_error = "vbnmf_comm_create: bad device";
        return VBNMF_ERR_CUDA;
    }
    vbnmf_comm *c = new vbnmf_comm();
    c->nranks = nranks; c->rank = rank; c->device = device;
    ncclUniqueId id;
    memcpy(&id, uid128, 128);
    ncclResult_t e = g_nccl.CommInitRank(&c->comm, nranks, id, rank);
    if (e != ncclSuccess) {
        g_create_error = std::string("ncclCommInitRank: ") +
                         (g_nccl.GetErrorString ? g_nccl.GetErrorString(e) : "error");
        delete c;
        return VBNMF_ERR_NCCL;
    }
    *out = c;
    return 0;
}

void vbnmf_comm_destroy(vbnmf_comm *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    delete c;
}

int vbnmf_attach_comm(vbnmf_handle *h, vbnmf_comm *c) {
    if (!h || !c) return VBNMF_ERR_ARG;
    if (c->device != h->device) return fail(h, VBNMF_ERR_ARG, "communicator is on another device");
    if (h->nranks > 1) return fail(h, VBNMF_ERR_STATE, "a communicator is already attached");
    if (c->nranks == 1) return 0;
    CK(cudaSetDevice(h->device));
    h->comm = c->comm;
    h->nranks = c->nranks;
    h->rank = c->rank;
    // global quantities: total cells, the sums over nonzeros, and the per-gene nonzero counts
    // (every rank must derive the same gene renumbering)
    // ... and whether EVERY shard holds 16-bit integer counts: the packed-16 layout decides the
    // tile height (split layout, staging slots), which all ranks must share -- the gene panels
    // are all-reduced in device order
    double hv[5] = {(double)h->m, h->lgx, h->mlconst, (double)h->nnz, h->p16 ? 0.0 : 1.0};
    ScopedBufs B(h);
    double *dv = nullptr;
    unsigned *d_flag = nullptr;
    uint32_t *d_scr = nullptr;
    CK(B.get(&dv, 5 * 8));
    CK(B.get(&d_flag, 4));
    CK(B.get(&d_scr, (size_t)2 * h->n * 4));
    CK(cudaMemsetAsync(d_flag, 0, 4, h->stream));
    CK(cudaMemcpyAsync(dv, hv, 5 * 8, cudaMemcpyHostToDevice, h->stream));
    int rc = allreduce(h, dv, 5);
    if (rc) return rc;
    CKN(g_nccl.AllReduce(h->d_cnt, h->d_cnt, (size_t)h->n, ncclUint64, ncclSum, h->comm, h->stream));
    vb::order_keys_kernel<<<cdiv(h->n, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        h->n, h->d_cnt, d_scr, d_scr + h->n, d_flag);
    unsigned nzero = 0;
    CK(cudaMemcpyAsync(hv, dv, 5 * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&nzero, d_flag, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    B.free(dv); B.free(d_flag); B.free(d_scr);
    h->m_global = (int64_t)llround(hv[0]);
    h->lgx = hv[1];
    h->mlconst = hv[2];
    h->nnz_global = (int64_t)llround(hv[3]);
    if (hv[4] != 0.0) h->p16 = false;
    h->empty_rows = nzero;  // of the whole matrix now (R/bayesian.R:244); tested at set_state
    free_panels(h);
    drop_layouts(h);
    h->stats_valid = false;
    return 0;
}

int vbnmf_set_state(vbnmf_handle *h, int r, const double *lw, const double *lh, const double *ew,
                    const double *eh) {
    if (!h || !lw || !lh) return VBNMF_ERR_ARG;
    int rc;
    if ((rc = check_rank(h, r))) return rc;
    CK(cudaSetDevice(h->device));
    StageTimer tm("vbnmf_set_state(total)");
    if ((rc = zeroed_panels(h, r))) return rc;
    // before the first update ew/eh are whatever the caller holds (vb_init: ew = w, eh = h); a
    // matrix passed twice goes up once
    const bool ew_same = !ew || ew == lw, eh_same = !eh || eh == lh;
    if ((rc = upload_panel(h, h->d_lw, ew_same ? h->d_alw : nullptr, lw, true, r))) return rc;
    if (!ew_same && (rc = upload_panel(h, h->d_alw, nullptr, ew, true, r))) return rc;
    if ((rc = upload_panel(h, h->d_lh, eh_same ? h->d_alh : nullptr, lh, false, r))) return rc;
    if (!eh_same && (rc = upload_panel(h, h->d_alh, nullptr, eh, false, r))) return rc;
    return loaded_state(h);
}

int vbnmf_init_random(vbnmf_handle *h, int r, const double hyper[4], uint64_t seed,
                      int64_t cell_offset) {
    if (!h || !hyper) return VBNMF_ERR_ARG;
    int rc;
    if ((rc = check_rank(h, r))) return rc;
    if (!(hyper[0] > 0 && hyper[1] > 0 && hyper[2] > 0 && hyper[3] > 0) || cell_offset < 0)
        return fail(h, VBNMF_ERR_ARG, "hyper-parameters must be positive");
    CK(cudaSetDevice(h->device));
    StageTimer tm("vbnmf_init_random(total)");
    if ((rc = zeroed_panels(h, r))) return rc;
    const Layout *L = h->L;
    const int rs = h->rs;
    // w ~ Gamma(aw, scale bw/aw), h ~ Gamma(ah, scale bh/ah); lw = ew = w, lh = eh = h (:111-115,170)
    vb::init_random_kernel<<<cdiv(h->n * r, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        h->n, r, rs, L->d_gene_dev, 0, 0, (unsigned long long)seed, hyper[0], hyper[1] / hyper[0],
        h->d_lw, h->d_alw, h->tsplit);
    vb::init_random_kernel<<<cdiv(h->m * r, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        h->m, r, rs, L->d_cell_dev, 1, cell_offset, (unsigned long long)seed, hyper[2],
        hyper[3] / hyper[2], h->d_lh, h->d_alh, h->tsplit);
    h->launches += 2;
    return loaded_state(h);
}

int vbnmf_init_svd2(vbnmf_handle *h, int r, const double hyper[4], uint64_t seed,
                    int64_t cell_offset) {
    if (!h || !hyper) return VBNMF_ERR_ARG;
    if (int rc = check_rank(h, r)) return rc;
    if (!(hyper[3] > 0) || cell_offset < 0) return fail(h, VBNMF_ERR_ARG, "bh must be positive");
    if (r > std::min(h->n, h->m_global)) return fail(h, VBNMF_ERR_ARG, "rank exceeds min(n, m)");
    CK(cudaSetDevice(h->device));
    StageTimer tm("vbnmf_init_svd2(total)");
    const double bh = hyper[3];
    return svd_init(h, r, seed, cell_offset, "svd2", [h, r, bh](const double *U, const double *T, bool *ok) {
        return svd2_finish(h, r, bh, U, T, ok);
    });
}

int vbnmf_init_svd(vbnmf_handle *h, int r, uint64_t seed, int64_t cell_offset) {
    if (!h) return VBNMF_ERR_ARG;
    if (int rc = check_rank(h, r)) return rc;
    if (cell_offset < 0) return fail(h, VBNMF_ERR_ARG, "cell_offset must be >= 0");
    if (r > std::min(h->n, h->m_global)) return fail(h, VBNMF_ERR_ARG, "rank exceeds min(n, m)");
    CK(cudaSetDevice(h->device));
    StageTimer tm("vbnmf_init_svd(total)");
    return svd_init(h, r, seed, cell_offset, "svd", [h, r](const double *U, const double *T, bool *ok) {
        return svd_finish(h, r, U, T, ok);
    });
}

int vbnmf_step(vbnmf_handle *h, const double hyper[4], double fudge, double *lkh) {
    if (!h || !hyper || !lkh) return VBNMF_ERR_ARG;
    int rc;
    if ((rc = check_state(h))) return rc;
    CK(cudaSetDevice(h->device));
    if ((rc = ensure_stats(h))) return rc;
    return iterate(h, hyper, fudge, lkh);
}

// The it-loop of vb_iterate with the loop control on the device: iterations are enqueued in
// batches without a host round trip; control_kernel applies hyper_update, the NaN and convergence
// rules after every iteration and raises the stop flag that turns the rest of the batch into
// no-ops.  VBNMF_HOST_LOOP=1 selects the host-controlled loop (one sync per iteration) instead.
static int run_device_loop(H *h, const vbnmf_cfg *cfg, double hyper[4], double *lkh_trace,
                           double *hyper_trace, int *niter, double *lml, int *stop_reason,
                           cudaEvent_t *ev /*optional: 4 events per iteration, bench*/) {
    CK(cudaSetDevice(h->device));
    int rc;
    const int rs = h->rs, r = h->r, itmax = cfg->itmax;
    if ((rc = ensure_stats(h))) return rc;
    // control block: hypers, lk0 = 0 (R/bayesian.R:336), rowSums(eh) of the loaded state
    double *c = h->h_ctl;
    for (int i = 0; i < vb::kCtlLen; i++) c[i] = 0.0;
    for (int q = 0; q < 4; q++) c[vb::kCtlHyper + q] = hyper[q];
    for (int k = 0; k < r; k++) c[vb::kCtlEhsum + k] = h->ehsum[k];
    CK(cudaMemcpyAsync(h->d_ctl, c, vb::kCtlLen * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    ScopedBufs B(h);
    double *d_trace = nullptr, *d_htrace = nullptr;
    CK(B.get(&d_trace, (size_t)itmax * 8));
    CK(B.get(&d_htrace, (size_t)itmax * 32));
    vb::ControlArgs ca;
    ca.ctl = h->d_ctl;
    ca.scal = h->d_scal;
    ca.tail = h->d_red + tail_off(h);
    ca.trace = d_trace;
    ca.htrace = d_htrace;
    ca.n = (double)h->n; ca.m_global = (double)h->m_global; ca.lgx = h->lgx; ca.tol = cfg->tol;
    ca.r = r; ca.rs = rs; ca.itmax = itmax; ca.n0 = cfg->n0; ca.dn = cfg->dn;
    for (int q = 0; q < 4; q++) ca.flags[q] = cfg->hyper_update[q];
    // from here on the kernels read the stop flag and the hypers from the control block
    DeviceControl dc(h);
    const int batch = 8;
    int launched = 0, it = 0;
    bool done = false;
    // Small problems are launch-bound (an iteration of the 1,000 x 200 plumbing case is ~8 kernels
    // of a few microseconds): there one batch of iterations is captured into a CUDA graph and
    // replayed.  Every kernel argument is the same in every iteration (hypers and the stop flag
    // live in the control block), and iterations replayed past the stop are no-ops.
    struct GraphGuard {
        cudaGraph_t g = nullptr;
        cudaGraphExec_t x = nullptr;
        ~GraphGuard() {
            if (x) cudaGraphExecDestroy(x);
            if (g) cudaGraphDestroy(g);
        }
    } gg;
    const bool use_graph = !ev && h->nranks == 1 && itmax >= 4 * batch && h->nnz <= kGraphMaxNnz &&
                           !getenv("VBNMF_NO_GRAPH");
    auto enqueue = [&](int gi) -> int {
        if ((rc = launch_posterior(h, true, 0, 0, cfg->fudge))) return rc;
        if ((rc = launch_posterior(h, false, 0, 0, cfg->fudge))) return rc;
        if (ev) CK(cudaEventRecord(ev[4 * gi + 0], h->stream));
        if ((rc = launch_sweep_cols(h))) return rc;
        if (ev) CK(cudaEventRecord(ev[4 * gi + 1], h->stream));
        if (ev) CK(cudaEventRecord(ev[4 * gi + 2], h->stream));
        if ((rc = launch_sweep_rows(h))) return rc;
        if (ev) CK(cudaEventRecord(ev[4 * gi + 3], h->stream));
        if ((rc = allreduce_red(h))) return rc;
        vb::control_kernel<<<1, 32, 0, h->stream>>>(ca);
        h->launches += 1;
        return 0;
    };
    int64_t launches_per_batch = 0;
    if (use_graph) {
        const int64_t l0 = h->launches;
        CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        rc = 0;
        for (int b = 0; b < batch && !rc; b++) rc = enqueue(b);
        cudaError_t ce = cudaStreamEndCapture(h->stream, &gg.g);
        launches_per_batch = h->launches - l0;
        h->launches = l0;
        if (rc) return rc;
        CK(ce);
        CK(cudaGraphInstantiate(&gg.x, gg.g, 0));
    }
    while (!done && launched < itmax) {
        const int nb = use_graph ? batch : std::min(batch, itmax - launched);
        if (use_graph) {
            CK(cudaGraphLaunch(gg.x, h->stream));
            h->launches += launches_per_batch;
        } else {
            for (int b = 0; b < nb; b++)
                if ((rc = enqueue(launched + b))) return rc;
        }
        launched += nb;
        CK(cudaMemcpyAsync(c, h->d_ctl, vb::kCtlLen * sizeof(double), cudaMemcpyDeviceToHost,
                           h->stream));
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaGetLastError());
        done = c[vb::kCtlDone] != 0.0;
        it = (int)c[vb::kCtlIt];
    }
    // results and the small host-side vectors the export functions use
    if (lkh_trace && it > 0)
        CK(cudaMemcpyAsync(lkh_trace, d_trace, (size_t)it * 8, cudaMemcpyDeviceToHost, h->stream));
    if (hyper_trace && it > 0)
        CK(cudaMemcpyAsync(hyper_trace, d_htrace, (size_t)it * 32, cudaMemcpyDeviceToHost,
                           h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if ((rc = peer_exit_barrier(h))) return rc;
    for (int k = 0; k < r; k++) {
        h->bew[k] = c[vb::kCtlBew + k];
        h->beh[k] = c[vb::kCtlBeh + k];
        h->ehsum[k] = c[vb::kCtlEhsum + k];
    }
    for (int q = 0; q < 3; q++) { h->wacc[q] = c[vb::kCtlAcc + q]; h->hacc[q] = c[vb::kCtlAcc + 3 + q]; }
    for (int q = 0; q < 4; q++) hyper[q] = c[vb::kCtlHyper + q];
    h->has_posterior = it > 0;
    // iterations enqueued past the stop were no-ops except for the all-reduce of stale statistics
    h->stats_valid = (launched == it || h->nranks == 1) && c[vb::kCtlHyperErr] == 0.0;
    *niter = it;
    *lml = c[vb::kCtlLk0];                                                  // R/bayesian.R:379
    *stop_reason = (int)c[vb::kCtlReason];
    if (c[vb::kCtlHyperErr] != 0.0)
        return fail(h, VBNMF_ERR_HYPER, "Hyper-parameter update failed to converge");
    return 0;
}

int vbnmf_run(vbnmf_handle *h, const vbnmf_cfg *cfg, double hyper[4], double *lkh_trace,
              double *hyper_trace, int *niter, double *lml, int *stop_reason) {
    if (!h || !cfg || !hyper || !niter || !lml || !stop_reason) return VBNMF_ERR_ARG;
    if (int rc = check_state(h)) return rc;
    if (cfg->itmax < 1 || cfg->dn < 1) return fail(h, VBNMF_ERR_ARG, "itmax and dn must be >= 1");
    if (!getenv("VBNMF_HOST_LOOP"))
        return run_device_loop(h, cfg, hyper, lkh_trace, hyper_trace, niter, lml, stop_reason,
                               nullptr);
    double lk0 = 0.0, lkh = 0.0;  // R/bayesian.R:336
    int it, reason = VBNMF_STOP_ITMAX, rc = 0;
    for (it = 1; it <= cfg->itmax; it++) {                                  // :337
        if ((rc = vbnmf_step(h, hyper, cfg->fudge, &lkh))) return rc;       // :339
        if (it > cfg->n0 && it % cfg->dn == 0) {                            // :342-344
            double mn[4];
            means_of(h, mn);
            if ((rc = vb_hyper_update(cfg->hyper_update, mn, hyper, 100, 1e-3)))
                return fail(h, rc, "Hyper-parameter update failed to converge");
        }
        if (lkh_trace) lkh_trace[it - 1] = lkh;
        if (hyper_trace) memcpy(hyper_trace + 4 * (it - 1), hyper, 4 * sizeof(double));
        if (std::isnan(lkh)) { reason = VBNMF_STOP_NAN; break; }            // :345
        if (it > 1 && it > cfg->n0 && lkh >= lk0 && fabs(1 - lkh / lk0) < cfg->tol) {  // :346-347
            reason = VBNMF_STOP_CONVERGED;
            break;
        }
        lk0 = lkh;                                                          // :348
    }
    if (it > cfg->itmax) it = cfg->itmax;
    *niter = it;
    *lml = lk0;                                                             // :379
    *stop_reason = reason;
    return 0;
}

int vbnmf_get_means(vbnmf_handle *h, double means[4]) {
    if (!h || !means) return VBNMF_ERR_ARG;
    if (!h->has_posterior) return fail(h, VBNMF_ERR_STATE, "no update has been run yet");
    means_of(h, means);
    return 0;
}

int vbnmf_get_state(vbnmf_handle *h, double *lw, double *lh, double *ew, double *eh, double *dw,
                    double *dh) {
    if (!h) return VBNMF_ERR_ARG;
    if (int rc = check_state(h)) return rc;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    StageTimer tm("vbnmf_get_state(total)");
    // the panels are brought into the caller's layout (and divided by bew / beh, :44,46,54,56) on
    // the device, then copied out
    const int r = h->r;
    const int64_t n = h->n, m = h->m;
    const Layout *L = h->L;
    ScopedBufs B(h);
    double *d_be = nullptr, *d_tmp = nullptr;
    CK(B.get(&d_be, 2 * kMaxRank * 8));
    CK(B.get(&d_tmp, (size_t)std::max(n, m) * r * 8));
    CK(cudaMemcpyAsync(d_be, h->bew, kMaxRank * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(d_be + kMaxRank, h->beh, kMaxRank * 8, cudaMemcpyHostToDevice, h->stream));
    auto one = [&](const double *panel, bool wside, int mode, double *out) -> int {
        if (!out) return 0;
        const int64_t cnt = wside ? n : m;
        if (mode == 2 && !h->has_posterior) {  // dw = dh = 0 before the first update (vb_init)
            memset(out, 0, (size_t)cnt * r * 8);
            return 0;
        }
        vb::gather_panel_kernel<<<cdiv(cnt * r, vb::kBlock), vb::kBlock, 0, h->stream>>>(
            cnt, r, h->rs, wside ? L->d_gene_dev : L->d_cell_dev, panel, wside,
            wside ? d_be : d_be + kMaxRank, mode, d_tmp, mode == 0 ? h->tsplit : 0);
        if (cnt * r * 8 >= (int64_t)(8 << 20)) return staged_download(h, out, d_tmp, cnt * r);
        CK(cudaMemcpyAsync(out, d_tmp, (size_t)cnt * r * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return 0;
    };
    int rc;
    if ((rc = one(h->d_lw, true, 0, lw)) || (rc = one(h->d_alw, true, 1, ew)) ||
        (rc = one(h->d_alw, true, 2, dw)) || (rc = one(h->d_lh, false, 0, lh)) ||
        (rc = one(h->d_alh, false, 1, eh)) || (rc = one(h->d_alh, false, 2, dh)))
        return rc;
    CK(cudaGetLastError());
    return 0;
}

int vbnmf_cluster_id(vbnmf_handle *h, int32_t *cid) {
    if (!h || !cid) return VBNMF_ERR_ARG;
    if (int rc = check_state(h)) return rc;
    CK(cudaSetDevice(h->device));
    const Layout *L = h->L;
    ScopedBufs B(h);
    double *d_beh = nullptr;
    int32_t *d_cid = nullptr, *d_out = nullptr;
    CK(B.get(&d_beh, kMaxRank * 8));
    CK(B.get(&d_cid, (size_t)L->NC * 4));
    CK(B.get(&d_out, (size_t)h->m * 4));
    CK(cudaMemcpyAsync(d_beh, h->beh, kMaxRank * 8, cudaMemcpyHostToDevice, h->stream));
    vb::cluster_id_kernel<<<cdiv(L->NC, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        L->NC, h->rs, h->r, h->d_alh, d_beh, d_cid);
    vb::gather_i32_kernel<<<cdiv(h->m, vb::kBlock), vb::kBlock, 0, h->stream>>>(
        h->m, L->d_cell_dev, d_cid, d_out);
    CK(cudaMemcpyAsync(cid, d_out, (size_t)h->m * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    return 0;
}

int vbnmf_uniform_columns(vbnmf_handle *h, double tol, int32_t *flags) {
    if (!h || !flags) return VBNMF_ERR_ARG;
    if (int rc = check_state(h)) return rc;
    CK(cudaSetDevice(h->device));
    const Layout *L = h->L;
    ScopedBufs B(h);
    double *d_bew = nullptr;
    int32_t *d_fl = nullptr;
    CK(B.get(&d_bew, kMaxRank * 8));
    CK(B.get(&d_fl, kMaxRank * 4));
    CK(cudaMemcpyAsync(d_bew, h->bew, kMaxRank * 8, cudaMemcpyHostToDevice, h->stream));
    vb::uniform_columns_kernel<<<h->r, vb::kBlock, 0, h->stream>>>(
        L->NG, L->T, L->Sg, h->n, h->rs, h->d_alw, d_bew, tol, d_fl);
    CK(cudaMemcpyAsync(flags, d_fl, (size_t)h->r * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    return 0;
}

int vbnmf_bench_iterations(vbnmf_handle *h, double hyper[4], double fudge, int iters,
                           int hyper_on, double ms[4], int64_t *launches, double *lkh_last) {
    if (!h || !hyper || !ms || iters < 1) return VBNMF_ERR_ARG;
    if (int rc = check_state(h)) return rc;
    CK(cudaSetDevice(h->device));
    int rc;
    double lkh = 0.0;
    if (!h->stats_valid && (rc = vbnmf_step(h, hyper, fudge, &lkh))) return rc;
    // exactly `iters` iterations of the product loop (run_device_loop) with a tolerance that never
    // triggers, CUDA events around the two sweep passes.  hyper_on = 1: hyper_update after every
    // iteration, i.e. the steady state of the reference loop past hyper.update.n0
    // (R/bayesian.R:342), hyper[] is updated; 0: hyper-parameters held fixed.
    std::vector<cudaEvent_t> ev((size_t)iters * 4 + 2, nullptr);
    struct DestroyEvents {  // on every return
        std::vector<cudaEvent_t> &e;
        ~DestroyEvents() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); }
    } destroy_events{ev};
    for (auto &e : ev) CK(cudaEventCreate(&e));
    vbnmf_cfg cfg;
    cfg.itmax = iters; cfg.tol = -1.0; cfg.n0 = hyper_on ? 0 : 1 << 30; cfg.dn = 1;
    cfg.fudge = fudge;
    for (int q = 0; q < 4; q++) cfg.hyper_update[q] = hyper_on ? 1 : 0;
    double hy[4] = {hyper[0], hyper[1], hyper[2], hyper[3]}, lml = 0.0;
    int niter = 0, why = 0;
    const int64_t l0 = h->launches;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaEventRecord(ev[0], h->stream));
    rc = run_device_loop(h, &cfg, hy, nullptr, nullptr, &niter, &lml, &why, ev.data() + 2);
    if (rc) return rc;
    CK(cudaEventRecord(ev[1], h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (niter != iters) return fail(h, VBNMF_ERR_STATE, "bench loop stopped early (NaN bound)");
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, ev[0], ev[1]));
    ms[0] = t;
    ms[1] = ms[2] = 0.0;
    for (int it = 0; it < iters; it++) {
        CK(cudaEventElapsedTime(&t, ev[2 + it * 4 + 0], ev[2 + it * 4 + 1]));
        ms[1] += t;
        CK(cudaEventElapsedTime(&t, ev[2 + it * 4 + 2], ev[2 + it * 4 + 3]));
        ms[2] += t;
    }
    ms[3] = ms[0] - ms[1] - ms[2];
    for (int q = 0; q < 4; q++) hyper[q] = hy[q];
    if (launches) *launches = h->launches - l0;
    if (lkh_last) *lkh_last = h->h_ctl[vb::kCtlLkh];
    return 0;
}

int vbnmf_info(const vbnmf_handle *h, int64_t info[8]) {
    if (!h || !info) return VBNMF_ERR_ARG;
    info[0] = h->n; info[1] = h->m; info[2] = h->nnz; info[3] = h->r; info[4] = h->rs;
    info[5] = h->precision; info[6] = h->nranks; info[7] = h->m_global;
    return 0;
}

int vbnmf_layout_info(const vbnmf_handle *h, int64_t info[8]) {
    if (!h || !info) return VBNMF_ERR_ARG;
    if (!h->L) return VBNMF_ERR_STATE;
    const Layout *L = h->L;
    const int fmt = entry_format(h);
    const int64_t ebytes = fmt == vb::kEntP16 ? 4 : (fmt == vb::kEntF32 ? 8 : 12);
    const int64_t pbytes = fmt == vb::kEntP16 ? 4 : 8;
    info[0] = fmt; info[1] = L->T; info[2] = L->Sg; info[3] = L->Sc;
    info[4] = L->cols.nent; info[5] = L->rows.nent;
    info[6] = fmt == vb::kEntP16 ? L->npg : 0;
    info[7] = (L->cols.nent + L->rows.nent) * ebytes + (L->cols.E + L->rows.E + 2) * pbytes +
              (fmt == vb::kEntP16 ? (L->cols.E + L->rows.E) * 4 : 0);  // + owner of each position
    return 0;
}

int mlnmf_run(vbnmf_handle *h, int r, const double *w0, const double *h0, int itmax, double tol,
              double *w, double *h_out, double *lik_trace, int *niter) {
    return mlnmf_run2(h, r, w0, h0, itmax, tol, VBNMF_ML_LIKELIHOOD, 0, w, h_out, lik_trace, nullptr,
                      niter);
}

int mlnmf_run2(vbnmf_handle *h, int r, const double *w0, const double *h0, int itmax, double tol,
               int criterion, int ncnn_step, double *w, double *h_out, double *lik_trace,
               double *nchange_trace, int *niter) {
    if (!h || !w0 || !h0 || !niter || itmax < 1) return VBNMF_ERR_ARG;
    if (int rc = check_rank(h, r)) return rc;
    if (criterion != VBNMF_ML_LIKELIHOOD && criterion != VBNMF_ML_CONNECTIVITY)
        return fail(h, VBNMF_ERR_ARG, "Unknown stopping criterion.");   // R/factorize.R:212
    if (criterion == VBNMF_ML_CONNECTIVITY && ncnn_step < 1)
        return fail(h, VBNMF_ERR_ARG, "ncnn_step must be >= 1");
    CK(cudaSetDevice(h->device));
    int rc;
    if ((rc = alloc_panels(h, r))) return rc;  // (lw and lh only: the ML path has no alw, alh)
    CK(cudaMemsetAsync(h->d_lw, 0, (size_t)h->L->NG * h->rs * 8, h->stream));
    CK(cudaMemsetAsync(h->d_lh, 0, (size_t)h->L->NC * h->rs * 8, h->stream));
    if ((rc = upload_panel(h, h->d_lw, nullptr, w0, true, r))) return rc;
    if ((rc = upload_panel(h, h->d_lh, nullptr, h0, false, r))) return rc;
    if ((rc = refresh_mirrors(h))) return rc;
    h->stats_valid = false;
    h->has_posterior = false;
    const Layout *L = h->L;
    const double eps = 2.220446049250313e-16;  // .Machine$double.eps, R/factorize.R:15,24
    const int rs = h->rs, wd = rs + 8;
    double *tail = h->d_red + tail_off(h);
    // connectivity criterion: labels of the previous and the current h, their contingency table
    ScopedBufs B(h);
    int32_t *d_lab[2] = {nullptr, nullptr};
    double *d_cont = nullptr;
    std::vector<double> cont;
    if (criterion == VBNMF_ML_CONNECTIVITY) {
        CK(B.get(&d_lab[0], (size_t)L->NC * 4));
        CK(B.get(&d_lab[1], (size_t)L->NC * 4));
        CK(B.get(&d_cont, (size_t)r * r * 8));
        cont.resize((size_t)r * r);
    }
    auto colsum = [&](bool wside) -> int {
        vb::ColsumArgs a{wside ? L->NG : L->NC, wside ? h->d_lw : h->d_lh,
                         wside ? h->d_partW : h->d_partH, wside ? h->d_scal : tail,
                         h->d_counters + (wside ? 0 : 1), h->tsplit};
        h->tab->colsum(a, h->stream);
        h->launches += 1;
        return 0;
    };
    auto mlupd = [&](bool wside) -> int {
        vb::MlUpdateArgs a{wside ? L->NG : L->NC, L->T, wside ? L->Sg : L->Sc,
                           wside ? h->n : h->m, r, eps, wside ? tail : h->d_scal,
                           wside ? h->d_red : h->d_ShRaw, wside ? h->d_lw : h->d_lh,
                           wside ? h->d_partW : h->d_partH, wside ? h->d_scal : tail,
                           h->d_counters + (wside ? 0 : 1), wside ? h->d_lw32 : h->d_lh32,
                           h->tsplit, h->ctl};
        h->tab->ml_update(a, h->stream);
        h->launches += 1;
        return 0;
    };
    auto lik_now = [&](double *lik) -> int {
        // likelihood (R/factorize.R:40-49) of the current w, h; needs xlogp of a column sweep at
        // these factors, colSums(w) in d_scal and rowSums(h) in the tail
        if ((rc = fetch_scalars(h))) return rc;
        double swh = 0.0;
        for (int k = 0; k < r; k++) swh += h->h_scal[k] * h->h_scal[wd + k];
        *lik = (h->h_scal[wd + rs + 4] - swh + h->mlconst) / (double)h->n / (double)h->m_global;
        return 0;
    };
    // number of cell pairs whose co-clustering changed between labelings `prev` and `cur`
    // (sum(cnn != cnn0), R/factorize.R:197) from their contingency table
    auto nchange_of = [&](int prev, int cur, double *nchange) -> int {
        CK(cudaMemsetAsync(d_cont, 0, (size_t)r * r * 8, h->stream));
        vb::contingency_kernel<<<h->num_sms * 2, vb::kBlock, (size_t)r * r * 4, h->stream>>>(
            L->NC, r, d_lab[prev], d_lab[cur], d_cont);
        h->launches += 1;
        if ((rc = allreduce(h, d_cont, (int64_t)r * r))) return rc;
        CK(cudaMemcpyAsync(cont.data(), d_cont, (size_t)r * r * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        auto c2 = [](double x) { return x * (x - 1.0) * 0.5; };
        double both = 0.0, rows2 = 0.0, cols2 = 0.0;
        for (int a = 0; a < r; a++) {
            double ra = 0.0, ca = 0.0;
            for (int b2 = 0; b2 < r; b2++) {
                ra += cont[(size_t)a * r + b2];
                ca += cont[(size_t)b2 * r + a];
                both += c2(cont[(size_t)a * r + b2]);
            }
            rows2 += c2(ra);
            cols2 += c2(ca);
        }
        *nchange = rows2 + cols2 - 2.0 * both;
        return 0;
    };
    if ((rc = colsum(true))) return rc;   // colSums(w0)
    if ((rc = colsum(false))) return rc;  // rowSums(h0) (local)
    if ((rc = allreduce(h, tail, rs))) return rc;
    if (criterion == VBNMF_ML_LIKELIHOOD && !getenv("VBNMF_HOST_LOOP")) {
        // Device-controlled loop: the likelihood, the stopping rule (:207) and the iteration count
        // live in the control block; turns are enqueued in batches of 8 without a host round trip
        // and become no-ops once the run has ended (as in run_device_loop for the VB path).
        double *c = h->h_ctl;
        for (int i = 0; i < vb::kCtlLen; i++) c[i] = 0.0;
        c[vb::kCtlLk0] = -INFINITY;                                        // lkold, :190
        CK(cudaMemcpyAsync(h->d_ctl, c, vb::kCtlLen * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        ScopedBufs Bt(h);
        double *d_trace = nullptr;
        CK(Bt.get(&d_trace, (size_t)itmax * 8));
        DeviceControl dc(h);
        vb::MlControlArgs ca{h->d_ctl, h->d_scal, tail, d_trace, (double)h->n, (double)h->m_global,
                             h->mlconst, tol, r, rs, itmax};
        int turns = 0;
        bool fin = false;
        while (!fin && turns < itmax + 1) {
            const int nb = std::min(8, itmax + 1 - turns);
            for (int b = 0; b < nb; b++) {
                if ((rc = launch_sweep_cols(h))) return rc;      // ShRaw, xlogp at (w, h) of turn - 1
                if ((rc = allreduce(h, tail + rs + 3, 2))) return rc;
                vb::ml_control_kernel<<<1, 32, 0, h->stream>>>(ca);
                h->launches += 1;
                if (turns + b + 1 <= itmax) {
                    if ((rc = mlupd(false))) return rc;          // h update, :8-15
                    if ((rc = launch_sweep_rows(h))) return rc;  // SwRaw at (w, h_new), :17
                    if ((rc = allreduce(h, h->d_red, tail_off(h) + rs))) return rc;
                    if ((rc = mlupd(true))) return rc;           // w update, :17-24
                }
            }
            turns += nb;
            CK(cudaMemcpyAsync(c, h->d_ctl, vb::kCtlLen * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            CK(cudaGetLastError());
            fin = c[vb::kCtlDone] != 0.0;
        }
        const int done_it = (int)c[vb::kCtlIt] - 1;              // likelihoods evaluated = iterations
        if (lik_trace && done_it > 0)
            CK(copy_sync(h, lik_trace, d_trace, (size_t)done_it * 8, cudaMemcpyDeviceToHost));
        *niter = done_it;
        h->ctl = nullptr;
        if (w || h_out) {
            if ((rc = vbnmf_get_state(h, w, h_out, nullptr, nullptr, nullptr, nullptr))) return rc;
        }
        return 0;
    }
    double lkold = -INFINITY, lk0 = NAN;
    int it, done = 0, zstep = 0;
    bool stop_after = false;
    for (it = 1; it <= itmax; it++) {                                      // R/factorize.R:191
        if ((rc = launch_sweep_cols(h))) return rc;  // ShRaw and xlogp at (w, h) of iteration it-1
        if ((rc = allreduce(h, tail + rs + 3, 2))) return rc;
        if (it > 1) {
            if ((rc = lik_now(&lk0))) return rc;                           // :193
            if (lik_trace) lik_trace[it - 2] = lk0;
            if (stop_after) { done = it - 1; break; }                      // :203 (zstep == ncnn.step)
            if (criterion == VBNMF_ML_LIKELIHOOD) {
                if (fabs(lkold - lk0) < tol * fabs(lkold)) { done = it - 1; break; }  // :207
                lkold = lk0;
            }
        }
        if ((rc = mlupd(false))) return rc;          // h update, :8-15 -> rowSums(h_new) in tail
        if (criterion == VBNMF_ML_CONNECTIVITY) {                          // :194-204 on h of iteration it
            const int cur = it & 1, prev = cur ^ 1;
            vb::ml_labels_kernel<<<cdiv(L->NC, vb::kBlock), vb::kBlock, 0, h->stream>>>(
                L->NC, L->T, L->Sc, h->m, rs, r, h->tsplit, h->d_lh, d_lab[cur]);
            h->launches += 1;
            double nchange = (double)h->m_global * ((double)h->m_global - 1.0) * 0.5;  // it == 1: npair
            if (it > 1 && (rc = nchange_of(prev, cur, &nchange))) return rc;
            if (nchange_trace) nchange_trace[it - 1] = nchange;
            zstep = nchange == 0.0 ? zstep + 1 : 0;
            if (zstep == ncnn_step) stop_after = true;
        }
        if ((rc = launch_sweep_rows(h))) return rc;  // SwRaw at (w, h_new), :17
        if ((rc = allreduce(h, h->d_red, tail_off(h) + rs))) return rc;
        if ((rc = mlupd(true))) return rc;           // w update, :17-24 -> colSums(w_new) in d_scal
    }
    if (!done) {
        if ((rc = launch_sweep_cols(h))) return rc;
        if ((rc = allreduce(h, tail + rs + 3, 2))) return rc;
        if ((rc = lik_now(&lk0))) return rc;
        if (lik_trace) lik_trace[itmax - 1] = lk0;
        done = itmax;
    }
    CK(cudaGetLastError());
    *niter = done;
    if (w || h_out) {
        if ((rc = vbnmf_get_state(h, w, h_out, nullptr, nullptr, nullptr, nullptr))) return rc;
    }
    return 0;
}

}  // extern "C"
