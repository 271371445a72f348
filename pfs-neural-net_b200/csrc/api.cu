// api.cu -- extern "C" entry points of libpfs_b200.so (see include/pfs_b200.h).
// Host-side orchestration only: argument checks, workspace carving, kernel launches on the
// caller's stream.  No torch types, no synchronisation, no host allocation in the hot calls.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "edge_model.cuh"
#include "node_ops.cuh"
#include "source_model.cuh"
#include "source_node_mma.cuh"
#include "source_node_bwd_mma.cuh"
#include "target_model.cuh"

using namespace pfs;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define PFS_CUDA(expr)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (expr);                                                                   \
        if (e__ != cudaSuccess) return fail(PFS_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)
// ---- launch accounting / optional per-kernel timing ------------------------------------------
// Every kernel launch goes through PFS_LAUNCH_CHECK(name) with the launch stream `st` in scope.
// The launch counter is always on.  With profiling enabled (pfs_profile_enable(1), used by
// bench.py) an event is recorded on the launch stream after every kernel and at the start of
// every entry point; a kernel's duration is the gap between its event and the previous one on
// that stream, which for back-to-back launches on one stream is its execution time.
struct ProfMark {
    const char* name;   // nullptr = start-of-call marker
    cudaEvent_t ev;
};
std::atomic<long long> g_launches{0};
bool g_prof_on = false;
std::vector<ProfMark> g_marks;
std::vector<cudaEvent_t> g_event_pool;
size_t g_events_used = 0;

void prof_mark(const char* name, cudaStream_t st) {
    if (name) ++g_launches;
    if (!g_prof_on) return;
    if (g_events_used == g_event_pool.size()) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        g_event_pool.push_back(e);
    }
    cudaEvent_t e = g_event_pool[g_events_used++];
    if (cudaEventRecord(e, st) != cudaSuccess) return;
    g_marks.push_back({name, e});
}

#define PFS_LAUNCH_CHECK(name)                                                                       \
    do {                                                                                            \
        cudaError_t e__ = cudaGetLastError();                                                       \
        if (e__ != cudaSuccess) return fail(PFS_ERR_CUDA, "launch %s: %s", name, cudaGetErrorString(e__)); \
        prof_mark(name, st);                                                                        \
    } while (0)
#define PFS_REQUIRE(cond, msg)                                  \
    do {                                                        \
        if (!(cond)) return fail(PFS_ERR_ARG, "%s (%s)", msg, #cond); \
    } while (0)
#define PFS_TRY(expr)            \
    do {                         \
        int rc__ = (expr);       \
        if (rc__ != PFS_OK) return rc__; \
    } while (0)

// ---- single-stream contract (include/pfs_b200.h, "Conventions") --------------------------------------------
// The module-level entry points share one __constant__ weight bank and one caller-provided workspace per device, so
// consecutive calls on a device must be ordered.  Every such call records an event on its stream when it returns;
// a call arriving on a DIFFERENT stream first makes that stream wait for the previous call's event (device-side
// wait, no host synchronisation).  Streams under CUDA-graph capture are left alone (the capture orders them).
struct StreamOrder {
    static constexpr int kMaxDev = 16;
    cudaStream_t last[kMaxDev] = {};
    cudaEvent_t ev[kMaxDev] = {};
    bool valid[kMaxDev] = {};
};
StreamOrder g_order;

struct CallGuard {
    cudaStream_t st;
    int dev = -1;
    bool capturing = false;
    explicit CallGuard(void* stream) : st((cudaStream_t)stream) {
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= StreamOrder::kMaxDev) { dev = -1; return; }
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { (void)cudaGetLastError(); dev = -1; return; }
        capturing = cs != cudaStreamCaptureStatusNone;
        if (capturing) { g_order.valid[dev] = false; return; }
        if (g_order.valid[dev] && g_order.last[dev] != st) (void)cudaStreamWaitEvent(st, g_order.ev[dev], 0);
    }
    ~CallGuard() {
        if (dev < 0 || capturing) return;
        if (!g_order.ev[dev] && cudaEventCreateWithFlags(&g_order.ev[dev], cudaEventDisableTiming) != cudaSuccess) {
            g_order.ev[dev] = nullptr;
            return;
        }
        g_order.valid[dev] = cudaEventRecord(g_order.ev[dev], st) == cudaSuccess;
        g_order.last[dev] = st;
    }
};

constexpr int kMaxCtas = 1024;

int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return kNumSM;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = kNumSM;
    }
    return n;
}

// persistent grid: resident CTAs of this kernel on the whole device, capped by the work items
template <class Kern>
int persistent_grid(Kern kern, size_t smem, long long items, int threads = kThreads) {
    int per_sm = 0;
    const cudaError_t oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
    static const bool dbg = getenv("PFS_DEBUG_GRID") != nullptr;
    if (dbg) {
        cudaFuncAttributes fa{};
        (void)cudaFuncGetAttributes(&fa, kern);
        fprintf(stderr, "[pfs] occupancy: %d blocks/SM (threads %d, smem %zu, err %s; regs %d, static smem %zu, max dyn %d, local %zu)\n",
                per_sm, threads, smem, cudaGetErrorString(oe), fa.numRegs, fa.sharedSizeBytes, fa.maxDynamicSharedSizeBytes,
                fa.localSizeBytes);
    }
    if (oe != cudaSuccess || per_sm < 1) {
        (void)cudaGetLastError();
        per_sm = 1;
    }
    long long g = (long long)per_sm * num_sms();
    if (g > kMaxCtas) g = kMaxCtas;
    if (g > items) g = items;
    return (int)(g < 1 ? 1 : g);
}

template <class Kern>
int allow_smem(Kern kern, size_t smem) {
    if (smem > 8 * 1024) {   // static + dynamic may cross the 48 KB default even when dynamic alone does not
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(PFS_ERR_CUDA, "cudaFuncSetAttribute(%zu B): %s", smem, cudaGetErrorString(e));
    }
    return PFS_OK;
}

struct Bump {
    char* p;
    size_t left;
    bool ok = true;
    Bump(void* base, size_t bytes) : p((char*)base), left(bytes) {
        const size_t mis = (size_t)((uintptr_t)p & 255);
        if (mis) {
            const size_t adv = 256 - mis;
            if (adv > left) { ok = false; left = 0; } else { p += adv; left -= adv; }
        }
    }
    float* f(size_t n) {
        const size_t bytes = ((n * sizeof(float) + 255) / 256) * 256;
        if (!ok || bytes > left) { ok = false; return nullptr; }
        float* r = (float*)p;
        p += bytes;
        left -= bytes;
        return r;
    }
};

int dense_fpt(int T) { return T > 0 ? kTile / T : 0; }
int dense_ntiles(int S, int T) {
    const int fpt = dense_fpt(T);
    return fpt > 0 ? (S + fpt - 1) / fpt : 0;
}
// node-MLP route per Fdim: 4, 8 and 10 on the tensor-core kernels with W4 in the constant bank (source_node_mma.cuh,
// source_node_bwd_mma.cuh), 16 on the shared-memory kernels (source_model.cuh)
template <int F> constexpr bool node_route_mma(bool mma) {
    return SourceNodeConst<F>::fits == mma && SourceNodeMma<F>::fits == mma && SourceNodeBwdMma<F>::fits == mma;
}
static_assert(node_route_mma<4>(true) && node_route_mma<8>(true) && node_route_mma<10>(true) && node_route_mma<16>(false),
              "node-MLP kernel route per Fdim");
// node tiles: the tensor-core forward uses 128-fibre tiles, the shared-memory kernels node_rows<F>()
template <int F> constexpr int node_tile_rows() { return SourceNodeConst<F>::fits ? kNodeRowsC : node_rows<F>(); }
template <int F> int node_ntiles(int S) { return (S + node_tile_rows<F>() - 1) / node_tile_rows<F>(); }

int make_topo(const pfs_topology& t, Topo& o) {
    PFS_REQUIRE(t.G >= 1 && t.S >= 1 && t.T >= 1 && t.E >= 0 && t.F >= 2, "bad topology sizes");
    o.layout = t.layout; o.G = t.G; o.F = t.F; o.S = t.S; o.T = t.T; o.E = t.E;
    o.rowptr = t.csr_rowptr; o.eid = t.csr_eid; o.csrc = t.csr_src; o.ctgt = t.csr_tgt;
    o.tile_fibre = t.tile_fibre; o.colptr = t.csc_colptr; o.cscq = t.csc_q;
    o.tile_q = t.tile_q; o.tile_slot = t.tile_slot; o.split_fibre = t.split_fibre; o.split_ptr = t.split_ptr;
    o.nsplit = t.nsplit; o.nslots = t.nslots;
    if (t.nsplit != 0) {
        PFS_REQUIRE(t.layout == PFS_LAYOUT_CSR && t.nsplit > 0 && t.nslots >= 2 * t.nsplit && t.tile_q && t.tile_slot &&
                        t.split_fibre && t.split_ptr, "split tiles need the CSR layout and the arrays of pfs_build_split_tiles");
    }
    if (t.layout == PFS_LAYOUT_DENSE) {
        if ((long long)t.S * t.T != t.E) return fail(PFS_ERR_ARG, "dense layout needs E == S*T");
        o.fpt = dense_fpt(t.T);
        if (o.fpt < 1)
            return fail(PFS_ERR_UNSUPPORTED, "dense layout with T=%d > %d classes per fibre is not supported by this build",
                        t.T, kTile);
        o.ntiles = dense_ntiles(t.S, t.T);
    } else if (t.layout == PFS_LAYOUT_CSR) {
        PFS_REQUIRE(t.csr_rowptr && t.csr_src && t.csr_tgt && t.tile_fibre && t.csc_colptr && t.csc_q && t.ntiles >= 1,
                    "CSR layout needs the arrays of pfs_build_topology");
        o.fpt = 0;
        o.ntiles = t.ntiles;
    } else {
        return fail(PFS_ERR_ARG, "unknown layout %d", t.layout);
    }
    return PFS_OK;
}

// message-MLP weights of the SModel / TModel edge kernels (common.cuh: MsgEdgeConst) appended to a pack list
template <int F>
void add_msg_weights(PackList& pl, const float* w1, const float* w2, const float* b2) {
    using CW = MsgEdgeConst<F>;
    constexpr int M = 2 * F;
    int n = pl.n;
    pl.it[n++] = PackItem{w1, M, F, F, M, 1, CW::kW1t};       // W1[:, F:] input-major [F][M]
    pl.it[n++] = PackItem{w1, M, F, F, M, 0, CW::kW1o};       // W1[:, F:] as stored [M][F]
    if (w2) {
        pl.it[n++] = PackItem{w2, M, 0, M, M, 1, CW::kW2t};   // W2 input-major
        pl.it[n++] = PackItem{w2, M, 0, M, M, 0, CW::kW2o};   // W2 as stored
    }
    if (b2) pl.it[n++] = PackItem{b2, 1, 0, 1, M, 0, CW::kB2};
    pl.n = n;
}

// Prologue of a module call: node tables + weight packing in ONE launch (node_ops.cuh: k_prep), then ONE copy of the
// packed weights into the constant bank.  Either part may be empty.
template <int F, int J>
int run_prep(int G, const TableJob* jobs, int njobs, const float* W, int ldw, const float* u, const PackList& pl,
             int nfloats, float* wstage, cudaStream_t st) {
    if (nfloats > kConstFloats) return fail(PFS_ERR_UNSUPPORTED, "weights (%d floats) exceed the constant bank", nfloats);
    PrepParams p{};
    long long maxn = 0;
    for (int q = 0; q < njobs; ++q) {
        p.job[q] = jobs[q];
        const long long n = (long long)jobs[q].rows * G;
        maxn = n > maxn ? n : maxn;
    }
    p.njobs = njobs; p.G = G; p.W = W; p.ldw = ldw; p.u = u; p.pl = pl; p.stage = wstage;
    p.pack_blocks = pl.n > 0 ? 8 : 0;
    long long tb = njobs > 0 ? (maxn + kThreads - 1) / kThreads : 0;
    if (tb > 4LL * num_sms()) tb = 4LL * num_sms();
    if (njobs > 0 && tb < 1) tb = 1;
    const int grid = p.pack_blocks + (int)tb;
    if (grid == 0) return PFS_OK;
    k_prep<F, J><<<grid, kThreads, 0, st>>>(p);
    PFS_LAUNCH_CHECK("k_prep");
    if (pl.n > 0)
        PFS_CUDA(cudaMemcpyToSymbolAsync(c_w, wstage, sizeof(float) * (size_t)nfloats, 0, cudaMemcpyDeviceToDevice, st));
    return PFS_OK;
}

// staging geometry of the edge kernels (common.cuh: TileStage)
int max_fibres_per_tile(const Topo& tp) {
    const int m = tp.layout == PFS_LAYOUT_DENSE ? tp.fpt : kTile;
    return m < tp.S ? m : tp.S;
}
bool stage_class_table(const Topo& tp, int row_floats) {   // both buffers of the class table <= 32 KB
    return (size_t)tp.T * (row_floats + 4) * sizeof(float) * 2 <= 32 * 1024;
}

// staging depth that fits: 2 buffers when the kernel's shared memory stays under the per-CTA limit
constexpr size_t kSmemLimit = 220 * 1024;
template <class SizeFn>
int pick_nbuf(SizeFn bytes_for, size_t& smem) {
    for (int nbuf = 2; nbuf >= 1; --nbuf) {
        smem = bytes_for(nbuf);
        if (smem <= kSmemLimit) return nbuf;
    }
    return 0;
}

bool fdim_supported(int F) { return F == 4 || F == 8 || F == 10 || F == 16; }

#define PFS_DISPATCH_F(Fv, CALL)                                   \
    switch (Fv) {                                                  \
        case 4: { constexpr int kF = 4; CALL; } break;            \
        case 8: { constexpr int kF = 8; CALL; } break;            \
        case 10: { constexpr int kF = 10; CALL; } break;          \
        case 16: { constexpr int kF = 16; CALL; } break;          \
        default: return fail(PFS_ERR_UNSUPPORTED, "Fdim=%d has no compiled kernels (built: 4, 8, 10, 16)", Fv); \
    }

// ---- small launch helpers ---------------------------------------------------------------
template <int K, int J>
int node_linear(const float* x, int rows, int G, const float* W, int ldw, int koff, const float* bias,
                const float* addvec, float* out, cudaStream_t st) {
    const long long N = (long long)rows * G;
    if (N == 0) return PFS_OK;
    long long blocks = (N + kThreads - 1) / kThreads;
    if (blocks > 4 * num_sms()) blocks = 4 * num_sms();
    k_node_linear<K, J><<<(int)blocks, kThreads, 0, st>>>(x, rows, G, W, ldw, koff, bias, addvec, out);
    PFS_LAUNCH_CHECK("k_node_linear");
    return PFS_OK;
}
template <int K, int J>
int node_linear_bwd(const float* d, long long N, const float* W, int ldw, int koff, float* dx, cudaStream_t st) {
    if (N == 0) return PFS_OK;
    long long blocks = (N + kThreads - 1) / kThreads;
    if (blocks > 4 * num_sms()) blocks = 4 * num_sms();
    k_node_linear_bwd<K, J, false><<<(int)blocks, kThreads, 0, st>>>(d, N, W, ldw, koff, dx);
    PFS_LAUNCH_CHECK("k_node_linear_bwd");
    return PFS_OK;
}
// builder for k_reduce_multi: segments of any number of partial buffers, one launch
struct Reducer {
    ReduceList rl{};
    const float* cur = nullptr;
    int cur_ncta = 0, cur_pstride = 0;
    bool overflow = false;
    void source(const float* partial, int ncta, int pstride) { cur = partial; cur_ncta = ncta; cur_pstride = pstride; }
    void add(int poff, int n, int cols, float* out, int ldo, int coff) {
        if (!out || n <= 0) return;
        if (rl.nseg >= kMaxReduceSegs) { overflow = true; return; }
        rl.seg[rl.nseg++] = ReduceSeg{cur, cur_ncta, cur_pstride, poff, n, cols, ldo, coff, out};
        rl.total += n;
    }
    int run(cudaStream_t st) {
        if (overflow) return fail(PFS_ERR_UNSUPPORTED, "too many reduction segments in one call");
        if (rl.nseg == 0) return PFS_OK;
        k_reduce_multi<<<(rl.total + 31) / 32, 32 * kReduceSlices, 0, st>>>(rl);
        PFS_LAUNCH_CHECK("k_reduce_partials");
        rl = ReduceList{};
        return PFS_OK;
    }
    int run(const float* partial, int ncta, int pstride, cudaStream_t st) {   // single-buffer form
        for (int q = 0; q < rl.nseg; ++q) {
            rl.seg[q].partial = partial; rl.seg[q].ncta = ncta; rl.seg[q].pstride = pstride;
        }
        return run(st);
    }
};

int colsum_all(const float* x, long long N, int ld, int off, int J, float* out, cudaStream_t st) {
    k_colsum_all<<<(J + 31) / 32, dim3(32, 8), 0, st>>>(x, N, ld, off, J, out);
    PFS_LAUNCH_CHECK("k_colsum_all");
    return PFS_OK;
}
// two column blocks of one [N, ld] matrix in one launch: out0 = sum of x[:, off0 : off0 + J], out1 = of x[:, off1 : off1 + J]
int colsum_pair(const float* x, long long N, int ld, int off0, float* out0, int off1, float* out1, int J, cudaStream_t st) {
    k_colsum_pair<<<dim3((J + 31) / 32, 2), dim3(32, 8), 0, st>>>(x, N, ld, off0, out0, off1, out1, J);
    PFS_LAUNCH_CHECK("k_colsum_all");
    return PFS_OK;
}
int colsum_graph(const float* x, int rows, int J, int G, float* out, cudaStream_t st) {
    k_colsum_graph<<<dim3((J + 31) / 32, G), dim3(32, 8), 0, st>>>(x, rows, J, out);
    PFS_LAUNCH_CHECK("k_colsum_graph");
    return PFS_OK;
}
int outer_graphs(const float* a, const float* b, int G, int J, int K, float* out, int ldo, int koff, cudaStream_t st) {
    k_outer_graphs<<<(J * K + 31) / 32, 256, 0, st>>>(a, b, G, J, K, out, ldo, koff);
    PFS_LAUNCH_CHECK("k_outer_graphs");
    return PFS_OK;
}
// dW[:, coff:coff+K] = D^T X, (optionally) db = column sums of D and (optionally) dx = D . W[:, coff:coff+K], over N rows
// of a node table's gradient D, in ONE pass over D (the input gradient used to be a k_node_linear_bwd launch of its own)
// The fixed-order sums of the CTA partials are queued on the caller's Reducer (scratch_partial must stay untouched until
// the caller runs it).
template <int J, int K, int TJ, int TK>
int outer_rows(Reducer& rd, const float* D, const float* X, long long N, float* scratch_partial, float* dW, int ldo, int coff,
               float* db, cudaStream_t st, const float* W = nullptr, float* dx = nullptr) {
    constexpr size_t smem = outer_rows_smem<J, K, TJ, TK>();
    if (N == 0) return PFS_OK;
    auto kern = dx ? k_outer_rows<J, K, TJ, TK, true> : k_outer_rows<J, K, TJ, TK, false>;
    PFS_TRY(allow_smem(kern, smem));
    const long long tiles = (N + kTile - 1) / kTile;
    const int grid = persistent_grid(kern, smem, tiles);
    constexpr int pstride = J * K + J;
    kern<<<grid, kThreads, smem, st>>>(D, X, N, scratch_partial, pstride, W, ldo, coff, dx);
    PFS_LAUNCH_CHECK("k_outer_rows");
    rd.source(scratch_partial, grid, pstride);
    rd.add(0, J * K, K, dW, ldo, coff);
    if (db) rd.add(J * K, J, J, db, J, 0);
    return PFS_OK;
}
// class-side sums: dense -> second stage over per-tile partials; CSR -> class-sorted segment sums
// chunks per class segment of the CSC sums: enough blocks to fill the device when there are few classes
int csc_chunks(const Topo& tp) {
    const long long blocks = (long long)tp.T * tp.G;
    long long n = (4LL * num_sms() + blocks - 1) / blocks;
    const long long avg = tp.E / (tp.T > 0 ? tp.T : 1);
    if (n > avg / 64) n = avg / 64;
    if (n > 64) n = 64;
    return (int)(n < 1 ? 1 : n);
}
size_t csc_scratch_floats(const Topo& tp, int J) {
    return tp.layout == PFS_LAYOUT_DENSE ? 0 : (size_t)tp.G * csc_chunks(tp) * tp.T * J;
}
int class_sums(const Topo& tp, const float* part_or_rows, int J, float* out, float* scratch, cudaStream_t st) {
    if (tp.layout == PFS_LAYOUT_DENSE) {
        const int TJ = tp.T * J;
        k_class_reduce<<<dim3((TJ + 127) / 128, tp.G), 128, 0, st>>>(part_or_rows, tp.ntiles, TJ, out);
        PFS_LAUNCH_CHECK("k_class_reduce");
    } else {
        if (J > kCscThreads) return fail(PFS_ERR_UNSUPPORTED, "class sums of %d features per row", J);
        const int nchunk = csc_chunks(tp);
        k_csc_segment_sum<<<dim3(tp.T, nchunk, tp.G), kCscThreads, 0, st>>>(part_or_rows, tp.colptr, tp.cscq, tp.E, tp.T, J,
                                                                            nchunk, out, scratch);
        PFS_LAUNCH_CHECK("k_csc_segment_sum");
        if (nchunk > 1) {
            const int TJ = tp.T * J;
            k_csc_segment_final<<<dim3((TJ + 127) / 128, tp.G), 128, 0, st>>>(scratch, nchunk, TJ, out);
            PFS_LAUNCH_CHECK("k_csc_segment_final");
        }
    }
    return PFS_OK;
}
// fibre sums of the split fibres from the partial rows of their tiles (W floats per row)
int split_sums(const Topo& tp, int W, const float* part, float* out, cudaStream_t st) {
    const long long n = (long long)tp.G * tp.nsplit * W;
    k_split_sums<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(tp, W, part, out);
    PFS_LAUNCH_CHECK("k_split_sums");
    return PFS_OK;
}
size_t class_stage_floats(const Topo& tp, int J) {
    return tp.layout == PFS_LAYOUT_DENSE ? (size_t)tp.G * tp.ntiles * tp.T * J : (size_t)tp.G * tp.E * J;
}
int bn_forward_tail(int F, int G, long long rows, const float* partial, int ntiles, int twice, int training,
                    const float* gamma, const float* beta, float* rm, float* rv, long long* nbt, float eps,
                    float momentum, float* save, cudaStream_t st, int rec_ncta = 0, int rec_nrec = 0) {
    const int n = G * F;
    if (training) {
        if (rows <= 1) return fail(PFS_ERR_ARG, "Expected more than 1 value per channel when training");
        if (F > 32) return fail(PFS_ERR_UNSUPPORTED, "BatchNorm finalisation handles up to 32 features");
        BnFinalizeAll fa{partial, rec_ncta, rec_nrec, ntiles, bn_partial_stride(F), F, G, twice, gamma, beta, eps, momentum, rows,
                         save, rm, rv, nbt};
        k_bn_finalize_all<<<(n + 255) / 256, 256, 0, st>>>(fa);
        PFS_LAUNCH_CHECK("k_bn_finalize_all");
    } else {
        PFS_REQUIRE(rm && rv, "eval-mode BatchNorm needs running_mean / running_var");
        k_bn_eval_coeffs<<<(n + 127) / 128, 128, 0, st>>>(rm, rv, F, G, gamma, beta, eps, twice, save);
        PFS_LAUNCH_CHECK("k_bn_eval_coeffs");
    }
    return PFS_OK;
}
int affine_rows(const float* in, const float* save, int F, long long rows, int G, float* out, cudaStream_t st) {
    const long long per_graph = rows * F / 2;
    if (per_graph == 0) return PFS_OK;
    long long blocks = (per_graph + 255) / 256;
    const long long cap = (16LL * num_sms() + G - 1) / G;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    k_affine_rows<<<dim3((unsigned)blocks, G), 256, 0, st>>>(in, save, F, rows * F, G, out);
    PFS_LAUNCH_CHECK("k_affine_rows");
    return PFS_OK;
}

// ==========================================================================================
// EdgeModel
// ==========================================================================================
// node tables of the EdgeModel's first-layer split: P_s = x_s . W1_s^T, P_t = x_t . W1_t^T + W1_u . u + b1
template <int F>
void edge_table_jobs(const pfs_edge_args& a, const Topo& tp, float* Ps, float* Pt, TableJob (&jobs)[2]) {
    jobs[0] = TableJob{a.x_s, tp.S, 0, -1, nullptr, Ps};
    jobs[1] = TableJob{a.x_t, tp.T, F, 3 * F, a.b1, Pt};
}

template <int F>
int edge_fwd_impl(const pfs_edge_args& a, const Topo& tp) {
    constexpr int H = 4 * F;
    cudaStream_t st = (cudaStream_t)a.stream;
    prof_mark(nullptr, st);
    const int total = tp.ntiles * tp.G;
    const int max_fib = max_fibres_per_tile(tp);
    const bool sc = stage_class_table(tp, H);
    size_t smem = 0;
    const int nbuf = pick_nbuf([&](int nb) { return sizeof(float) * TileStage<F, 1, H, H>::floats(max_fib, tp.T, sc, nb); }, smem);
    if (!nbuf) return fail(PFS_ERR_UNSUPPORTED, "edge_fwd: tile staging does not fit shared memory");
    auto kern = tp.nsplit > 0 ? k_edge_fwd<F, true> : k_edge_fwd<F>;
    PFS_TRY(allow_smem(kern, smem));
    const int grid = persistent_grid(kern, smem, total);
    const int nrec = chunk_records(grid, total, tp.ntiles);
    Bump ws(a.workspace, a.workspace_bytes);
    float* uvec = ws.f((size_t)tp.G * H);
    PFS_REQUIRE((a.table_s == nullptr) == (a.table_t == nullptr), "table_s and table_t go together");
    float* Ps = a.table_s ? a.table_s : ws.f((size_t)tp.G * tp.S * H);
    float* Pt = a.table_t ? a.table_t : ws.f((size_t)tp.G * tp.T * H);
    float* part = ws.f((size_t)grid * nrec * bn_partial_stride(F));
    float* wstage = ws.f(kConstFloats);
    if (!ws.ok) return fail(PFS_ERR_WORKSPACE, "edge_fwd: workspace too small (%zu B)", a.workspace_bytes);
    (void)uvec;
    TableJob jobs[2];
    edge_table_jobs<F>(a, tp, Ps, Pt, jobs);
    PackList pl{};
    pl.it[0] = PackItem{a.w1, H, 2 * F, F, H, 1, 0};            // W1_e input-major [F][H]
    pl.it[1] = PackItem{a.w2, H, 0, H, F, 1, F * H};            // W2 input-major [H][F]
    pl.it[2] = PackItem{a.b2, 1, 0, 1, F, 0, 2 * F * H};        // b2
    pl.n = 3;
    PFS_TRY((run_prep<F, H>(tp.G, jobs, 2, a.w1, H, a.u, pl, 2 * F * H + F, wstage, st)));
    const bool stats = a.normed && a.training;
    EdgeFwdParams p{tp, a.x_e, Ps, Pt, a.w1, a.w2, a.b2, a.x_e_out, stats ? part : nullptr, max_fib, sc ? 1 : 0, nrec, nbuf};
    kern<<<grid, kThreads, smem, st>>>(p);
    PFS_LAUNCH_CHECK("k_edge_fwd");
    if (a.normed) {
        PFS_REQUIRE(a.gamma && a.beta && a.bn_save, "normed edge model needs gamma, beta, bn_save");
        PFS_TRY(bn_forward_tail(F, tp.G, tp.E, part, tp.ntiles, 1, a.training, a.gamma, a.beta, a.running_mean,
                                a.running_var, (long long*)a.num_batches_tracked, a.eps, a.momentum, a.bn_save, st,
                                grid, nrec));
        if (!a.defer_affine) PFS_TRY(affine_rows(a.x_e_out, a.bn_save, F, tp.E, tp.G, a.x_e_out, st));
    }
    return PFS_OK;
}

template <int F>
int edge_bwd_impl(const pfs_edge_args& a, const Topo& tp) {
    constexpr int H = 4 * F;
    cudaStream_t st = (cudaStream_t)a.stream;
    prof_mark(nullptr, st);
    const int total = tp.ntiles * tp.G;
    const int mode = !a.normed ? 0 : (a.training ? 1 : 2);
    using SM = EdgeBwdSmem<F>;
    // k_edge_bwd2 (two CTAs per SM: x_e staged only, hidden layer in two halves, shared accumulator registers) where
    // its tiles fit 113 KB, else the double-buffered one-CTA-per-SM k_edge_bwd (Fdim 16).
    // Measured at C3: 1.21 ms against 1.60 ms.
    constexpr bool lean = SM::lean_fits;
    const bool split = tp.nsplit > 0;
    auto kern = lean ? (split ? k_edge_bwd2<F, true> : k_edge_bwd2<F>) : (split ? k_edge_bwd<F, true> : k_edge_bwd<F>);
    const int max_fib = max_fibres_per_tile(tp);
    const bool sc = stage_class_table(tp, H);
    size_t smem_bwd = SM::bytes_lean;
    int nbuf = 1;
    if (!lean) {
        nbuf = pick_nbuf([&](int nb) { return SM::bytes(max_fib, tp.T, sc, nb); }, smem_bwd);
        if (!nbuf) return fail(PFS_ERR_UNSUPPORTED, "edge_bwd: tile staging does not fit shared memory");
    }
    PFS_TRY(allow_smem(kern, smem_bwd));
    const int grid = persistent_grid(kern, smem_bwd, total);
    constexpr int pstride = 2 * H * F + F;
    Bump ws(a.workspace, a.workspace_bytes);
    float* uvec = ws.f((size_t)tp.G * H);
    PFS_REQUIRE((a.table_s == nullptr) == (a.table_t == nullptr), "table_s and table_t go together");
    const bool cached = a.table_s != nullptr;              // node tables kept by the forward: not recomputed
    float* Ps = cached ? a.table_s : ws.f((size_t)tp.G * tp.S * H);
    float* Pt = cached ? a.table_t : ws.f((size_t)tp.G * tp.T * H);
    float* coef = ws.f((size_t)tp.G * 6 * F);
    float* statp = ws.f((size_t)total * 2 * F);
    float* dgb = ws.f((size_t)tp.G * 2 * F);
    float* dPs = ws.f((size_t)tp.G * tp.S * H);
    float* stage = ws.f(class_stage_floats(tp, H));
    float* cscs = ws.f(csc_scratch_floats(tp, H) + 1);
    double* statsum = (double*)ws.f((size_t)tp.G * 4 * F + 2);
    float* dPt = ws.f((size_t)tp.G * tp.T * H);
    float* tot = ws.f((size_t)tp.G * H);
    float* wpart = ws.f((size_t)grid * pstride);
    float* opart = ws.f((size_t)kMaxCtas * (H * F + H));
    float* opart2 = ws.f((size_t)((tp.G * tp.T + kTile - 1) / kTile + 1) * (H * F + H));     // class table: few row tiles
    float* wstage = ws.f(kConstFloats);
    float* dPs_split = split ? ws.f((size_t)tp.G * tp.nslots * H) : nullptr;
    if (!ws.ok) return fail(PFS_ERR_WORKSPACE, "edge_bwd: workspace too small (%zu B)", a.workspace_bytes);
    {
        (void)uvec;
        using CW = EdgeBwdConst<F>;
        TableJob jobs[2];
        edge_table_jobs<F>(a, tp, Ps, Pt, jobs);
        PackList pl{};
        pl.it[0] = PackItem{a.w1, H, 2 * F, F, H, 1, CW::kW1t};     // W1_e input-major [F][H]
        pl.it[1] = PackItem{a.w2, H, 0, H, F, 0, CW::kW2o};         // W2 as stored [F][H]
        pl.it[2] = PackItem{a.w1, H, 2 * F, F, H, 0, CW::kW1o};     // W1_e as stored [H][F]
        pl.n = 3;
        PFS_TRY((run_prep<F, H>(tp.G, jobs, cached ? 0 : 2, a.w1, H, a.u, pl, CW::kFloats, wstage, st)));
    }
    const int n = tp.G * F;
    k_edge_bn_bwd_coef<<<(n + 127) / 128, 128, 0, st>>>(0, mode, F, tp.G, tp.ntiles, tp.E, a.bn_save, a.gamma, a.beta,
                                                         a.running_mean, a.running_var, a.eps, statsum, coef, dgb);
    PFS_LAUNCH_CHECK("k_edge_bn_bwd_coef/0");
    if (mode != 0) {
        EdgeBnStatParams sp{tp, a.x_e_out, a.g_out, coef, statp};
        auto ks = split ? k_edge_bn_bwd_stats<F, true> : k_edge_bn_bwd_stats<F>;
        const int g2 = persistent_grid(ks, 0, total);
        ks<<<g2, kThreads, 0, st>>>(sp);
        PFS_LAUNCH_CHECK("k_edge_bn_bwd_stats");
        k_tile_partial_sums<<<tp.G, 256, 0, st>>>(statp, tp.ntiles, 2 * F, statsum);
        PFS_LAUNCH_CHECK("k_tile_partial_sums");
        k_edge_bn_bwd_coef<<<(n + 127) / 128, 128, 0, st>>>(1, mode, F, tp.G, tp.ntiles, tp.E, a.bn_save,
                                                             a.gamma, a.beta, a.running_mean, a.running_var, a.eps, statsum,
                                                             coef, dgb);
        PFS_LAUNCH_CHECK("k_edge_bn_bwd_coef/1");
        PFS_TRY(colsum_pair(dgb, tp.G, 2 * F, 0, a.g_gamma, F, a.g_beta, F, st));
    }
    const bool dense = tp.layout == PFS_LAYOUT_DENSE;
    EdgeBwdParams p{tp, a.x_e, a.x_e_out, a.g_out, Ps, Pt, coef, a.g_x_e, dPs,
                    dense ? stage : nullptr, dense ? nullptr : stage, wpart, pstride, max_fib, sc ? 1 : 0, nbuf, dPs_split};
    kern<<<grid, kThreads, smem_bwd, st>>>(p);
    if (lean) {
        PFS_LAUNCH_CHECK("k_edge_bwd2");
    } else {
        PFS_LAUNCH_CHECK("k_edge_bwd");
    }
    Reducer rd;                       // all the final sums of this call go out in one launch at its end
    rd.source(wpart, grid, pstride);
    rd.add(0, H * F, F, a.g_w1, H, 2 * F);
    rd.add(H * F, F * H, H, a.g_w2, H, 0);
    rd.add(2 * H * F, F, F, a.g_b2, F, 0);
    PFS_TRY(class_sums(tp, stage, H, dPt, cscs, st));
    if (split) PFS_TRY(split_sums(tp, H, dPs_split, dPs, st));
    // node-table backward, one pass per table: g_x_s = dPs . W1_s, dW1_s += dPs^T x_s (the same for the class table)
    PFS_TRY((outer_rows<H, F, 8, F / 2>(rd, dPs, a.x_s, (long long)tp.G * tp.S, opart, a.g_w1, H, 0, nullptr, st, a.w1, a.g_x_s)));
    PFS_TRY((outer_rows<H, F, 8, F / 2>(rd, dPt, a.x_t, (long long)tp.G * tp.T, opart2, a.g_w1, H, F, nullptr, st, a.w1, a.g_x_t)));
    PFS_TRY(rd.run(st));
    PFS_TRY(colsum_graph(dPt, tp.T, H, tp.G, tot, st));
    PFS_TRY(colsum_all(tot, tp.G, H, 0, H, a.g_b1, st));
    PFS_TRY(outer_graphs(tot, a.u, tp.G, H, F, a.g_w1, H, 3 * F, st));
    PFS_TRY((node_linear_bwd<F, H>(tot, tp.G, a.w1, H, 3 * F, a.g_u, st)));
    return PFS_OK;
}

// ==========================================================================================
// SModel
// ==========================================================================================
template <int F>
int source_fwd_impl(const pfs_source_args& a, const Topo& tp) {
    constexpr int M = 2 * F;
    cudaStream_t st = (cudaStream_t)a.stream;
    prof_mark(nullptr, st);
    const int total = tp.ntiles * tp.G;
    const int ntn = node_ntiles<F>(tp.S);
    Bump ws(a.workspace, a.workspace_bytes);
    float* Qt = ws.f((size_t)tp.G * tp.T * M);
    float* partn = ws.f((size_t)tp.G * ntn * bn_partial_stride(F));
    float* wstage = ws.f(kConstFloats);
    const bool split = tp.nsplit > 0;
    float* srec = split ? ws.f((size_t)tp.G * tp.nslots * moment_record_floats(M)) : nullptr;
    if (!ws.ok) return fail(PFS_ERR_WORKSPACE, "source_fwd: workspace too small (%zu B)", a.workspace_bytes);
    {
        // one prologue: the class table Q_t, the message-MLP weights and the node-MLP weights (disjoint regions of the
        // constant bank: MsgEdgeConst below SourceNodeConst::kBase), one upload
        TableJob jobs[2] = {TableJob{a.x_t, tp.T, 0, -1, a.b1, Qt}, TableJob{}};
        PackList pl{};
        add_msg_weights<F>(pl, a.w1, a.w2, a.b2);
        int nfloats = MsgEdgeConst<F>::kFloats;
        if constexpr (SourceNodeConst<F>::fits) {
            using CW = SourceNodeConst<F>;
            constexpr int J = 10 * F;
            pl.it[pl.n++] = PackItem{a.w4, J, 0, J, F, 1, CW::kW4t};       // W4 input-major [J][F]
            pl.it[pl.n++] = PackItem{a.b4, 1, 0, 1, F, 0, CW::kB4};
            nfloats = CW::kFwdMmaFloats;
        }
        PFS_TRY((run_prep<F, M>(tp.G, jobs, 1, a.w1, M, a.u, pl, nfloats, wstage, st)));
    }
    {
        if (a.x_e_affine) PFS_REQUIRE(a.x_e_norm_out, "x_e_affine needs x_e_norm_out");
        SourceEdgeFwdParams p{tp, a.x_e, Qt, a.w1, a.w2, a.b2, a.moments, a.x_e_affine, a.x_e_norm_out, srec};
        auto kern = split ? k_source_edge_fwd<F, true> : k_source_edge_fwd<F>;
        const int grid = persistent_grid(kern, 0, total);
        kern<<<grid, kThreads, 0, st>>>(p);
        PFS_LAUNCH_CHECK("k_source_edge_fwd");
        if (split) {
            const long long n = (long long)tp.G * tp.nsplit * M;
            k_split_moments<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(tp, M, srec, a.moments);
            PFS_LAUNCH_CHECK("k_split_moments");
        }
    }
    {
        const bool stats = a.normed && a.training;
        SourceNodeFwdParams p{tp.G, tp.S, a.x_s, a.u, a.moments, a.w3, a.b3, a.w4, a.b4, a.hidden, a.y_pre,
                              stats ? partn : nullptr, ntn};
        if constexpr (SourceNodeConst<F>::fits) {
            // first layer on tcgen05 (3xTF32), see source_node_mma.cuh
            auto kern = k_source_node_fwd_mma<F>;
            constexpr size_t smem = SourceNodeMma<F>::bytes;
            PFS_TRY(allow_smem(kern, smem));
            const int grid = persistent_grid(kern, smem, (long long)ntn * tp.G, kNodeThreadsC);
            kern<<<grid, kNodeThreadsC, smem, st>>>(p);
            PFS_LAUNCH_CHECK("k_source_node_fwd_mma");
        } else {
            using SM = SourceNodeFwdSmem<F>;
            auto kern = k_source_node_fwd<F>;
            PFS_TRY(allow_smem(kern, SM::bytes));
            const int grid = persistent_grid(kern, SM::bytes, (long long)ntn * tp.G);
            kern<<<grid, kThreads, SM::bytes, st>>>(p);
            PFS_LAUNCH_CHECK("k_source_node_fwd");
        }
    }
    if (a.normed) {
        PFS_REQUIRE(a.gamma && a.beta && a.bn_save, "normed source model needs gamma, beta, bn_save");
        PFS_TRY(bn_forward_tail(F, tp.G, tp.S, partn, ntn, 0, a.training, a.gamma, a.beta, a.running_mean,
                                a.running_var, (long long*)a.num_batches_tracked, a.eps, a.momentum, a.bn_save, st));
        PFS_TRY(affine_rows(a.y_pre, a.bn_save, F, tp.S, tp.G, a.x_s_out, st));
    } else {
        PFS_CUDA(cudaMemcpyAsync(a.x_s_out, a.y_pre, sizeof(float) * (size_t)tp.G * tp.S * F, cudaMemcpyDeviceToDevice, st));
    }
    return PFS_OK;
}

template <int F>
int source_bwd_impl(const pfs_source_args& a, const Topo& tp) {
    constexpr int M = 2 * F, J = 10 * F, K9 = 9 * F;
    cudaStream_t st = (cudaStream_t)a.stream;
    prof_mark(nullptr, st);
    const int total = tp.ntiles * tp.G;
    int ntn = node_ntiles<F>(tp.S);
    const int mode = !a.normed ? 0 : (a.training ? 1 : 2);
    constexpr size_t smem_e = SourceEdgeBwdSmem<F>::bytes;
    constexpr bool kNodeMma = SourceNodeBwdMma<F>::fits;
    auto ke = tp.nsplit > 0 ? k_source_edge_bwd<F, true> : k_source_edge_bwd<F>;
    PFS_TRY(allow_smem(ke, smem_e));
    int gridn = 0;
    if constexpr (kNodeMma) {
        ntn = (tp.S + kNodeRowsB - 1) / kNodeRowsB;        // 48-fibre tiles
        PFS_TRY(allow_smem(k_source_node_bwd_mma<F>, SourceNodeBwdMma<F>::bytes));
        gridn = persistent_grid(k_source_node_bwd_mma<F>, SourceNodeBwdMma<F>::bytes, (long long)ntn * tp.G, kNodeThreadsC);
    } else {
        PFS_TRY(allow_smem(k_source_node_bwd<F>, SourceNodeBwdSmem<F>::bytes));
        gridn = persistent_grid(k_source_node_bwd<F>, SourceNodeBwdSmem<F>::bytes, (long long)ntn * tp.G);
    }
    const int gride = persistent_grid(ke, smem_e, total);
    constexpr int pstride_n = J * K9 + F * J + F;
    constexpr int pstride_e = M * F + M * M + M;
    Bump ws(a.workspace, a.workspace_bytes);
    float* Qt = ws.f((size_t)tp.G * tp.T * M);
    float* bnstat = ws.f((size_t)tp.G * 2 * F);
    float* bnpart = ws.f((size_t)tp.G * 64 * 2 * F);
    float* coefA = ws.f((size_t)tp.G * tp.S * 4 * M);
    float* tot3p = ws.f((size_t)tp.G * ntn * J);
    float* tot3 = ws.f((size_t)tp.G * J);
    float* wpn = ws.f((size_t)gridn * pstride_n);
    float* stage = ws.f(class_stage_floats(tp, M));
    float* cscs = ws.f(csc_scratch_floats(tp, M) + 1);
    float* dQt = ws.f((size_t)tp.G * tp.T * M);
    float* wpe = ws.f((size_t)gride * pstride_e);
    float* opart = ws.f((size_t)kMaxCtas * (M * F + M));
    float* wstage = ws.f(kConstFloats);
    if (!ws.ok) return fail(PFS_ERR_WORKSPACE, "source_bwd: workspace too small (%zu B)", a.workspace_bytes);
    {
        // one prologue for the whole backward: Q_t, the node-MLP weights and the message-MLP weights (disjoint regions
        // of the constant bank), one upload
        TableJob jobs[2] = {TableJob{a.x_t, tp.T, 0, -1, a.b1, Qt}, TableJob{}};
        PackList pl{};
        add_msg_weights<F>(pl, a.w1, a.w2, a.b2);
        int nfloats = MsgEdgeConst<F>::kFloats;
        if constexpr (kNodeMma) {
            using CW = SourceNodeConst<F>;
            pl.it[pl.n++] = PackItem{a.w4, J, 0, J, F, 0, CW::kW4o};       // W4 as stored [F][J]
            nfloats = CW::kBwdMmaFloats;
        }
        PFS_TRY((run_prep<F, M>(tp.G, jobs, 1, a.w1, M, a.u, pl, nfloats, wstage, st)));
    }
    if (mode != 0) {
        int nchunk = (tp.S + 4095) / 4096;           // one CTA per 4096 fibres of a graph (1 for the C3 graphs)
        if (nchunk > 64) nchunk = 64;
        constexpr int kStatThreads = 1024;           // ~100 row lanes per CTA: few rows, many loads in flight per lane
        k_bn_bwd_stats_rows<<<dim3(nchunk, tp.G), kStatThreads, sizeof(float) * 2 * kStatThreads, st>>>(
            a.g_out, a.y_pre, a.bn_save, tp.S, F, a.eps, nchunk, nchunk > 1 ? bnpart : bnstat);
        PFS_LAUNCH_CHECK("k_bn_bwd_stats_rows");
        if (nchunk > 1) {
            k_bn_bwd_stats_final<<<(tp.G * 2 * F + 127) / 128, 128, 0, st>>>(bnpart, nchunk, 2 * F, tp.G, bnstat);
            PFS_LAUNCH_CHECK("k_bn_bwd_stats_final");
        }
        PFS_TRY(colsum_pair(bnstat, tp.G, 2 * F, F, a.g_gamma, 0, a.g_beta, F, st));
    }
    {
        SourceNodeBwdParams p{tp.G, tp.S, ntn, mode, a.eps, a.x_s, a.moments, a.hidden, a.y_pre, a.g_out, a.bn_save,
                              bnstat, a.w3, a.w4, a.g_x_s, coefA, tot3p, wpn, pstride_n};
        if constexpr (kNodeMma) {
            // both 9F x 10F contractions on tcgen05 (3xTF32), see source_node_bwd_mma.cuh
            k_source_node_bwd_mma<F><<<gridn, kNodeThreadsC, SourceNodeBwdMma<F>::bytes, st>>>(p);
            PFS_LAUNCH_CHECK("k_source_node_bwd_mma");
        } else {
            k_source_node_bwd<F><<<gridn, kThreads, SourceNodeBwdSmem<F>::bytes, st>>>(p);
            PFS_LAUNCH_CHECK("k_source_node_bwd");
        }
    }
    Reducer rd;                       // all the final sums of this call go out in one launch at its end
    rd.source(wpn, gridn, pstride_n);
    rd.add(0, J * K9, K9, a.g_w3, J, 0);
    rd.add(J * K9, F * J, J, a.g_w4, J, 0);
    rd.add(J * K9 + F * J, F, F, a.g_b4, F, 0);
    k_class_reduce<<<dim3((J + 127) / 128, tp.G), 128, 0, st>>>(tot3p, ntn, J, tot3);
    PFS_LAUNCH_CHECK("k_class_reduce(tot3)");
    PFS_TRY(colsum_all(tot3, tp.G, J, 0, J, a.g_b3, st));
    PFS_TRY(outer_graphs(tot3, a.u, tp.G, J, F, a.g_w3, J, K9, st));
    PFS_TRY((node_linear_bwd<F, J>(tot3, tp.G, a.w3, J, K9, a.g_u, st)));
    {
        const bool dense = tp.layout == PFS_LAYOUT_DENSE;
        SourceEdgeBwdParams p{tp, a.x_e, Qt, a.w1, a.w2, a.b2, a.moments, coefA, a.g_x_e, a.g_x_e_add,
                              dense ? stage : nullptr, dense ? nullptr : stage, wpe, pstride_e};
        ke<<<gride, kThreads, smem_e, st>>>(p);
        PFS_LAUNCH_CHECK("k_source_edge_bwd");
    }
    rd.source(wpe, gride, pstride_e);
    rd.add(0, M * F, F, a.g_w1, M, F);
    rd.add(M * F, M * M, M, a.g_w2, M, 0);
    rd.add(M * F + M * M, M, M, a.g_b2, M, 0);
    PFS_TRY(class_sums(tp, stage, M, dQt, cscs, st));
    PFS_TRY((outer_rows<M, F, 4, F / 2>(rd, dQt, a.x_t, (long long)tp.G * tp.T, opart, a.g_w1, M, 0, a.g_b1, st, a.w1, a.g_x_t)));
    PFS_TRY(rd.run(st));
    return PFS_OK;
}

// ==========================================================================================
// TModel
// ==========================================================================================
TargetTailParams make_tail(const pfs_target_args& a, const Topo& tp) {
    TargetTailParams p{};
    p.G = tp.G; p.T = tp.T; p.F = tp.F;
    p.mode = !a.normed ? 0 : (a.training ? 1 : 2);
    p.eps = a.eps;
    p.x_t = a.x_t; p.u = a.u; p.act_sum = a.act_sum;
    p.colptr = tp.layout == PFS_LAYOUT_DENSE ? nullptr : tp.colptr;
    p.dense_count = tp.S;
    p.w2 = a.w2; p.b2 = a.b2; p.w3 = a.w3; p.b3 = a.b3; p.w4 = a.w4; p.b4 = a.b4;
    p.gamma = a.gamma; p.beta = a.beta; p.rm = a.running_mean; p.rv = a.running_var;
    p.y_pre = a.y_pre; p.x_t_out = a.x_t_out; p.bn_save = a.bn_save;
    p.gout = a.g_out; p.g_x_t = a.g_x_t; p.g_u = a.g_u;
    return p;
}

template <int F>
int target_fwd_impl(const pfs_target_args& a, const Topo& tp) {
    constexpr int M = 2 * F;
    cudaStream_t st = (cudaStream_t)a.stream;
    prof_mark(nullptr, st);
    const int total = tp.ntiles * tp.G;
    Bump ws(a.workspace, a.workspace_bytes);
    float* Rs = a.table_s ? a.table_s : ws.f((size_t)tp.G * tp.S * M);
    float* stage = ws.f(class_stage_floats(tp, M));
    float* cscs = ws.f(csc_scratch_floats(tp, M) + 1);
    float* wstage = ws.f(kConstFloats);
    if (!ws.ok) return fail(PFS_ERR_WORKSPACE, "target_fwd: workspace too small (%zu B)", a.workspace_bytes);
    if (a.normed) PFS_REQUIRE(a.gamma && a.beta && a.bn_save, "normed target model needs gamma, beta, bn_save");
    if (a.normed && a.training && tp.T <= 1)
        return fail(PFS_ERR_ARG, "Expected more than 1 value per channel when training");
    if (a.normed && !a.training) PFS_REQUIRE(a.running_mean && a.running_var, "eval-mode BatchNorm needs running buffers");
    {
        TableJob jobs[2] = {TableJob{a.x_s, tp.S, 0, -1, a.b1, Rs}, TableJob{}};
        PackList pl{};
        add_msg_weights<F>(pl, a.w1, nullptr, nullptr);
        PFS_TRY((run_prep<F, M>(tp.G, jobs, 1, a.w1, M, a.u, pl, MsgEdgeConst<F>::kFloats, wstage, st)));
    }
    {
        const bool dense = tp.layout == PFS_LAYOUT_DENSE;
        TargetEdgeFwdParams p{tp, a.x_e, Rs, a.w1, dense ? stage : nullptr, dense ? nullptr : stage};
        auto kern = tp.nsplit > 0 ? k_target_edge_fwd<F, true> : k_target_edge_fwd<F>;
        const int grid = persistent_grid(kern, 0, total);
        kern<<<grid, kThreads, 0, st>>>(p);
        PFS_LAUNCH_CHECK("k_target_edge_fwd");
    }
    PFS_TRY(class_sums(tp, stage, M, a.act_sum, cscs, st));
    {
        TargetTailParams p = make_tail(a, tp);
        const size_t smem = sizeof(float) * ((size_t)tp.T * 8 * F + 4 * F);
        if (smem > 200 * 1024) return fail(PFS_ERR_UNSUPPORTED, "target tail: T*F too large for one CTA (%zu B)", smem);
        PFS_TRY(allow_smem(k_target_tail_fwd, smem));
        k_target_tail_fwd<<<tp.G, kThreads, smem, st>>>(p);
        PFS_LAUNCH_CHECK("k_target_tail_fwd");
    }
    if (a.normed && a.training && a.running_mean && a.running_var) {
        k_bn_running<<<F, 32, 0, st>>>(a.bn_save, F, tp.G, tp.T, a.gamma, a.beta, a.eps, a.momentum, 0, a.running_mean,
                                       a.running_var, (long long*)a.num_batches_tracked);
        PFS_LAUNCH_CHECK("k_bn_running");
    }
    return PFS_OK;
}

template <int F>
int target_bwd_impl(const pfs_target_args& a, const Topo& tp) {
    constexpr int M = 2 * F, H = 4 * F;
    cudaStream_t st = (cudaStream_t)a.stream;
    prof_mark(nullptr, st);
    const int total = tp.ntiles * tp.G;
    using SM = TargetEdgeBwdSmem<F>;
    const bool split = tp.nsplit > 0;
    auto ke = split ? k_target_edge_bwd<F, true> : k_target_edge_bwd<F>;
    PFS_TRY(allow_smem(ke, SM::bytes));
    const int gride = persistent_grid(ke, SM::bytes, total);
    constexpr int pstride_e = M * F;
    constexpr int ptail = tail_partial_floats(F);
    Bump ws(a.workspace, a.workspace_bytes);
    const bool cached = a.table_s != nullptr;              // R_s kept by the forward: not recomputed
    float* Rs = cached ? a.table_s : ws.f((size_t)tp.G * tp.S * M);
    float* dasum = ws.f((size_t)tp.G * tp.T * M);
    float* gpart = ws.f((size_t)tp.G * ptail);
    float* dRs = ws.f((size_t)tp.G * tp.S * M);
    float* wpe = ws.f((size_t)gride * pstride_e);
    float* opart = ws.f((size_t)kMaxCtas * (M * F + M));
    float* wstage = ws.f(kConstFloats);
    float* dRs_split = split ? ws.f((size_t)tp.G * tp.nslots * M) : nullptr;
    if (!ws.ok) return fail(PFS_ERR_WORKSPACE, "target_bwd: workspace too small (%zu B)", a.workspace_bytes);
    {
        TargetTailParams p = make_tail(a, tp);
        p.dasum = dasum;
        p.gpartial = gpart;
        const size_t smem = sizeof(float) * ((size_t)tp.T * 8 * F + 6 * F);
        if (smem > 200 * 1024) return fail(PFS_ERR_UNSUPPORTED, "target tail: T*F too large for one CTA (%zu B)", smem);
        PFS_TRY(allow_smem(k_target_tail_bwd, smem));
        k_target_tail_bwd<<<tp.G, kThreads, smem, st>>>(p);
        PFS_LAUNCH_CHECK("k_target_tail_bwd");
    }
    Reducer rd;                       // all the final sums of this call go out in one launch at its end
    {
        rd.source(gpart, tp.G, ptail);
        rd.add(tail_off_w2(F), M * M, M, a.g_w2, M, 0);
        rd.add(tail_off_b2(F), M, M, a.g_b2, M, 0);
        rd.add(tail_off_w3(F), H * H, H, a.g_w3, H, 0);
        rd.add(tail_off_b3(F), H, H, a.g_b3, H, 0);
        rd.add(tail_off_w4(F), F * H, H, a.g_w4, H, 0);
        rd.add(tail_off_b4(F), F, F, a.g_b4, F, 0);
        if (a.normed) {
            rd.add(tail_off_gamma(F), F, F, a.g_gamma, F, 0);
            rd.add(tail_off_beta(F), F, F, a.g_beta, F, 0);
        }
    }
    {
        TableJob jobs[2] = {TableJob{a.x_s, tp.S, 0, -1, a.b1, Rs}, TableJob{}};
        PackList pl{};
        add_msg_weights<F>(pl, a.w1, nullptr, nullptr);
        PFS_TRY((run_prep<F, M>(tp.G, jobs, cached ? 0 : 1, a.w1, M, a.u, pl, MsgEdgeConst<F>::kFloats, wstage, st)));
    }
    {
        TargetEdgeBwdParams p{tp, a.x_e, Rs, a.w1, dasum, a.g_x_e, a.g_x_e_add, dRs, wpe, pstride_e, dRs_split};
        ke<<<gride, kThreads, SM::bytes, st>>>(p);
        PFS_LAUNCH_CHECK("k_target_edge_bwd");
    }
    if (split) PFS_TRY(split_sums(tp, M, dRs_split, dRs, st));
    rd.source(wpe, gride, pstride_e);
    rd.add(0, M * F, F, a.g_w1, M, F);
    PFS_TRY((outer_rows<M, F, 4, F / 2>(rd, dRs, a.x_s, (long long)tp.G * tp.S, opart, a.g_w1, M, 0, a.g_b1, st, a.w1, a.g_x_s)));
    PFS_TRY(rd.run(st));
    return PFS_OK;
}

// ==========================================================================================
// time head
// ==========================================================================================
template <int F>
int head_impl(const pfs_head_args& a, const Topo& tp, bool backward) {
    cudaStream_t st = (cudaStream_t)a.stream;
    prof_mark(nullptr, st);
    const long long N = (long long)tp.G * tp.E;
    constexpr int pstride = F * F + 2 * F + 1;
    HeadParams p{tp, a.x_e, a.w1, a.b1, a.w2, a.b2, a.scale, a.class_hours, (const long long*)a.edge_tgt,
                 a.time, a.visits, a.time_int, a.g_time, a.g_x_e, nullptr, pstride};
    if (!backward) {
        if (tp.layout != PFS_LAYOUT_DENSE && a.class_hours) PFS_REQUIRE(a.edge_tgt, "CSR layout head needs edge_tgt");
        long long blocks = (N + kThreads - 1) / kThreads;
        if (blocks > 8 * num_sms()) blocks = 8 * num_sms();
        if (blocks < 1) blocks = 1;
        k_head_fwd<F><<<(int)blocks, kThreads, 0, st>>>(p);
        PFS_LAUNCH_CHECK("k_head_fwd");
        return PFS_OK;
    }
    const long long tiles = (N + kTile - 1) / kTile;
    const int grid = persistent_grid(k_head_bwd<F>, 0, tiles);
    Bump ws(a.workspace, a.workspace_bytes);
    float* wpart = ws.f((size_t)grid * pstride);
    if (!ws.ok) return fail(PFS_ERR_WORKSPACE, "head_bwd: workspace too small (%zu B)", a.workspace_bytes);
    p.wpartial = wpart;
    k_head_bwd<F><<<grid, kThreads, 0, st>>>(p);
    PFS_LAUNCH_CHECK("k_head_bwd");
    {
        Reducer rd;
        rd.add(0, F * F, F, a.g_w1, F, 0);
        rd.add(F * F, F, F, a.g_b1, F, 0);
        rd.add(F * F + F, F, F, a.g_w2, F, 0);
        rd.add(F * F + 2 * F, 1, 1, a.g_b2, 1, 0);
        PFS_TRY(rd.run(wpart, grid, pstride, st));
    }
    return PFS_OK;
}

// ==========================================================================================
// topology kernels
// ==========================================================================================
__global__ void k_set_flag(int* flag, int v) { *flag = v; }
__global__ void k_detect_dense(const long long* ei, long long E, int T, int* flag) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    if (ei[e] != e / T || ei[E + e] != e % T) *flag = 0;   // benign race: every writer stores 0
}
__global__ void k_split_edges(const long long* ei, long long E, int* src, int* eid) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    src[e] = (int)ei[e];
    eid[e] = (int)e;
}
__global__ void k_gather_tgt(const long long* ei, long long E, const int* eid, int* tgt, int* q) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= E) return;
    tgt[i] = (int)ei[E + eid[i]];
    q[i] = (int)i;
}
// ptr[s] = number of sorted keys < s  (lower bound), s in [0, n]
__global__ void k_lower_bounds(const int* keys, int E, int n, int* ptr) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s > n) return;
    int lo = 0, hi = E;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (keys[mid] < s) lo = mid + 1; else hi = mid;
    }
    ptr[s] = lo;
}
// greedy packing of whole fibres into tiles of <= kTile edges (sequential, one-time per topology)
__global__ void k_pack_tiles(const int* rowptr, int S, int* tile_fibre, int* ntiles, int* max_degree) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    int nt = 0, cur = 0, nf = 0, maxd = 0;   // a tile holds <= kTile edges AND <= kTile fibres
    tile_fibre[0] = 0;
    for (int f = 0; f < S; ++f) {
        const int d = rowptr[f + 1] - rowptr[f];
        maxd = d > maxd ? d : maxd;
        if ((cur + d > kTile && cur > 0) || nf >= kTile) {
            tile_fibre[++nt] = f;
            cur = 0;
            nf = 0;
        }
        cur += d;
        ++nf;
    }
    tile_fibre[++nt] = S;
    *ntiles = nt;
    *max_degree = maxd;
}

// Tile table with split fibres (sequential, one-time per topology): whole fibres packed as k_pack_tiles packs them, a
// fibre of d > kTile edges cut into ceil(d / kTile) consecutive tiles of its own whose sizes differ by at most one
// (257 -> 129 + 128: no chunk of a handful of edges)
__global__ void k_pack_split_tiles(const int* rowptr, int S, int* tile_fibre, int* tile_q, int* tile_slot, int* split_fibre,
                                   int* split_ptr, int* counts) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    int nt = 0, cur = 0, nf = 0, ns = 0, nslot = 0;
    bool open = false;                      // the last tile holds whole fibres and may take more
    for (int f = 0; f < S; ++f) {
        const int q = rowptr[f], d = rowptr[f + 1] - q;
        if (d > kTile) {
            const int k = (d + kTile - 1) / kTile, base = d / k, rem = d - base * k;
            split_fibre[ns] = f;
            split_ptr[ns++] = nslot;
            for (int c = 0, qc = q; c < k; ++c) {
                tile_fibre[nt] = f;
                tile_q[nt] = qc;
                tile_slot[nt++] = nslot++;
                qc += base + (c < rem ? 1 : 0);
            }
            open = false;
            continue;
        }
        if (!open || (cur + d > kTile && cur > 0) || nf >= kTile) {
            tile_fibre[nt] = f;
            tile_q[nt] = q;
            tile_slot[nt++] = -1;
            cur = 0;
            nf = 0;
            open = true;
        }
        cur += d;
        ++nf;
    }
    tile_fibre[nt] = S;
    tile_q[nt] = rowptr[S];
    split_ptr[ns] = nslot;
    counts[0] = nt;
    counts[1] = ns;
    counts[2] = nslot;
}

size_t sort_temp_bytes(long long E) {
    size_t bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const int*)nullptr, (int*)nullptr, (const int*)nullptr,
                                    (int*)nullptr, (int)E);
    return ((bytes + 255) / 256) * 256;
}

}  // namespace

// host-side services shared with the other translation units of the library (wide.cu)
namespace pfs_host {
int fail_msg(int code, const char* msg) { return fail(code, "%s", msg); }
void mark_launch(const char* name, cudaStream_t st) { prof_mark(name, st); }
int sm_count() { return num_sms(); }
}  // namespace pfs_host

// ==========================================================================================
// extern "C"
// ==========================================================================================
extern "C" {

int pfs_abi_version(void) { return PFS_ABI_VERSION; }
const char* pfs_last_error(void) { return g_err; }
int pfs_supports_fdim(int32_t F) { return fdim_supported(F) ? 1 : 0; }
size_t pfs_sizeof_topology(void) { return sizeof(pfs_topology); }
size_t pfs_sizeof_edge_args(void) { return sizeof(pfs_edge_args); }
size_t pfs_sizeof_source_args(void) { return sizeof(pfs_source_args); }
size_t pfs_sizeof_target_args(void) { return sizeof(pfs_target_args); }
size_t pfs_sizeof_global_args(void) { return sizeof(pfs_global_args); }
size_t pfs_sizeof_head_args(void) { return sizeof(pfs_head_args); }

long long pfs_launch_count(void) { return g_launches; }
int pfs_profile_enable(int on) {
    g_prof_on = on != 0;
    g_marks.clear();
    g_events_used = 0;
    return PFS_OK;
}
// Text report "name launches total_ms\n" per kernel, summed over everything recorded since
// pfs_profile_enable(1).  Waits for the recorded events (call it outside the timed region).
int pfs_profile_report(char* buf, size_t buflen) {
    if (!buf || buflen == 0) return fail(PFS_ERR_ARG, "null buffer");
    struct Row { const char* name; long long n; double ms; };
    std::vector<Row> rows;
    for (size_t i = 1; i < g_marks.size(); ++i) {
        if (!g_marks[i].name) continue;
        float ms = 0.f;
        if (cudaEventSynchronize(g_marks[i].ev) != cudaSuccess) continue;
        if (cudaEventElapsedTime(&ms, g_marks[i - 1].ev, g_marks[i].ev) != cudaSuccess) continue;
        bool found = false;
        for (auto& r : rows)
            if (strcmp(r.name, g_marks[i].name) == 0) { r.n++; r.ms += ms; found = true; break; }
        if (!found) rows.push_back({g_marks[i].name, 1, ms});
    }
    size_t off = 0;
    for (auto& r : rows) {
        int w = snprintf(buf + off, buflen - off, "%s %lld %.6f\n", r.name, r.n, r.ms);
        if (w < 0 || (size_t)w >= buflen - off) break;
        off += (size_t)w;
    }
    buf[off < buflen ? off : buflen - 1] = 0;
    g_marks.clear();
    g_events_used = 0;
    return (int)off;
}

size_t pfs_workspace_bytes(const pfs_topology* t) {
    if (!t) return 0;
    const size_t G = t->G, S = t->S, T = t->T, E = t->E, F = t->F;
    const size_t ntiles = t->layout == PFS_LAYOUT_DENSE ? (size_t)dense_ntiles(t->S, t->T) : (size_t)t->ntiles;
    const size_t ntn = ((size_t)t->S + 49) / 50;   // smallest node tile of any Fdim
    size_t fl = 0;
    fl += G * S * 16 * F;                               // node tables, fibre sums, moment coefficients
    fl += G * T * 16 * F;
    fl += G * ntiles * (T * 4 * F + 4 * F + 8);         // per-tile class partials and BatchNorm partials
    fl += G * ntn * (12 * F + 8);
    if (t->layout != PFS_LAYOUT_DENSE) fl += G * E * 4 * F + G * 64 * T * 4 * F;   // materialised rows + CSC chunk partials
    fl += (size_t)kMaxCtas * (100 * F * F + 32 * F + 64) * 2;   // per-CTA weight-gradient partials
    fl += 2 * kConstFloats;                                       // weight staging for the constant bank
    fl += G * (36 * F * F + 128 * F);
    fl += G * 64 * 2 * F + 64;                                   // chunk partials of the node BatchNorm backward sums
    if (t->nsplit > 0) fl += G * (size_t)t->nslots * (10 * F + 1) + 64;   // split tiles: chunk records / partial fibre sums
    fl += 4096;
    return fl * sizeof(float) + 64 * 256;
}

int pfs_detect_dense(const int64_t* edge_index, int64_t E, int32_t S, int32_t T, int32_t* flag_dev, void* stream) {
    PFS_REQUIRE(edge_index && flag_dev && S >= 1 && T >= 1, "bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const bool maybe = (long long)S * T == E && E > 0;
    k_set_flag<<<1, 1, 0, st>>>(flag_dev, maybe ? 1 : 0);
    PFS_LAUNCH_CHECK("k_set_flag");
    if (maybe) {
        k_detect_dense<<<(unsigned)((E + 255) / 256), 256, 0, st>>>((const long long*)edge_index, E, T, flag_dev);
        PFS_LAUNCH_CHECK("k_detect_dense");
    }
    return PFS_OK;
}

size_t pfs_build_topology_temp_bytes(int64_t E, int32_t S, int32_t T) {
    (void)S; (void)T;
    const size_t arr = (((size_t)E * sizeof(int) + 255) / 256) * 256;
    return 4 * arr + sort_temp_bytes(E) + 1024;
}

int pfs_build_topology(const int64_t* edge_index, int64_t E, int32_t S, int32_t T, int32_t* csr_rowptr,
                       int32_t* csr_eid, int32_t* csr_src, int32_t* csr_tgt, int32_t* csc_colptr, int32_t* csc_q,
                       int32_t* tile_fibre, int32_t* ntiles_dev, int32_t* max_degree_dev, void* temp,
                       size_t temp_bytes, void* stream) {
    PFS_REQUIRE(edge_index && csr_rowptr && csr_eid && csr_src && csr_tgt && csc_colptr && csc_q && tile_fibre &&
                    ntiles_dev && max_degree_dev && temp, "null pointer");
    PFS_REQUIRE(E >= 1 && E < (1ll << 31) && S >= 1 && T >= 1, "bad sizes");
    if (temp_bytes < pfs_build_topology_temp_bytes(E, S, T)) return fail(PFS_ERR_WORKSPACE, "topology temp too small");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t arr = (((size_t)E * sizeof(int) + 255) / 256) * 256;
    char* base = (char*)temp;
    int* k_in = (int*)base;
    int* v_in = (int*)(base + arr);
    int* k_tmp = (int*)(base + 2 * arr);
    int* v_tmp = (int*)(base + 3 * arr);
    void* cub_tmp = base + 4 * arr;
    size_t cub_bytes = sort_temp_bytes(E);
    const unsigned blocks = (unsigned)((E + 255) / 256);
    const long long* ei = (const long long*)edge_index;
    // fibre-sorted (CSR) order: stable LSD radix sort of (src, edge id)
    k_split_edges<<<blocks, 256, 0, st>>>(ei, E, k_in, v_in);
    PFS_LAUNCH_CHECK("k_split_edges");
    PFS_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, k_in, csr_src, v_in, csr_eid, (int)E, 0, 32, st));
    k_gather_tgt<<<blocks, 256, 0, st>>>(ei, E, csr_eid, csr_tgt, v_tmp);
    PFS_LAUNCH_CHECK("k_gather_tgt");
    k_lower_bounds<<<(S + 1 + 255) / 256, 256, 0, st>>>(csr_src, (int)E, S, csr_rowptr);
    PFS_LAUNCH_CHECK("k_lower_bounds(src)");
    // class-sorted (CSC) order of the CSR positions
    PFS_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, csr_tgt, k_tmp, v_tmp, csc_q, (int)E, 0, 32, st));
    k_lower_bounds<<<(T + 1 + 255) / 256, 256, 0, st>>>(k_tmp, (int)E, T, csc_colptr);
    PFS_LAUNCH_CHECK("k_lower_bounds(tgt)");
    k_pack_tiles<<<1, 1, 0, st>>>(csr_rowptr, S, tile_fibre, ntiles_dev, max_degree_dev);
    PFS_LAUNCH_CHECK("k_pack_tiles");
    return PFS_OK;
}

int pfs_build_split_tiles(const int32_t* csr_rowptr, int32_t S, int32_t* tile_fibre, int32_t* tile_q, int32_t* tile_slot,
                          int32_t* split_fibre, int32_t* split_ptr, int32_t* counts_dev, void* stream) {
    PFS_REQUIRE(csr_rowptr && tile_fibre && tile_q && tile_slot && split_fibre && split_ptr && counts_dev, "null pointer");
    PFS_REQUIRE(S >= 1, "bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    k_pack_split_tiles<<<1, 1, 0, st>>>(csr_rowptr, S, tile_fibre, tile_q, tile_slot, split_fibre, split_ptr, counts_dev);
    PFS_LAUNCH_CHECK("k_pack_split_tiles");
    return PFS_OK;
}

int pfs_edge_fwd(const pfs_edge_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    PFS_REQUIRE(a && a->x_s && a->x_t && a->x_e && a->u && a->w1 && a->b1 && a->w2 && a->b2 && a->x_e_out && a->workspace,
                "null pointer");
    Topo tp;
    PFS_TRY(make_topo(a->topo, tp));
    PFS_DISPATCH_F(tp.F, return edge_fwd_impl<kF>(*a, tp));
    return PFS_OK;
}
int pfs_edge_bwd(const pfs_edge_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    PFS_REQUIRE(a && a->x_s && a->x_t && a->x_e && a->u && a->w1 && a->b1 && a->w2 && a->x_e_out && a->g_out &&
                    a->g_x_s && a->g_x_t && a->g_x_e && a->g_u && a->g_w1 && a->g_b1 && a->g_w2 && a->g_b2 && a->workspace,
                "null pointer");
    if (a->normed) PFS_REQUIRE(a->gamma && a->beta && a->bn_save && a->g_gamma && a->g_beta, "normed backward needs norm tensors");
    Topo tp;
    PFS_TRY(make_topo(a->topo, tp));
    PFS_DISPATCH_F(tp.F, return edge_bwd_impl<kF>(*a, tp));
    return PFS_OK;
}
int pfs_source_fwd(const pfs_source_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    PFS_REQUIRE(a && a->x_s && a->x_t && a->x_e && a->u && a->w1 && a->b1 && a->w2 && a->b2 && a->w3 && a->b3 && a->w4 &&
                    a->b4 && a->x_s_out && a->moments && a->hidden && a->y_pre && a->workspace, "null pointer");
    Topo tp;
    PFS_TRY(make_topo(a->topo, tp));
    PFS_DISPATCH_F(tp.F, return source_fwd_impl<kF>(*a, tp));
    return PFS_OK;
}
int pfs_source_bwd(const pfs_source_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    PFS_REQUIRE(a && a->x_s && a->x_t && a->x_e && a->u && a->w1 && a->b1 && a->w2 && a->b2 && a->w3 && a->w4 &&
                    a->moments && a->hidden && a->y_pre && a->g_out && a->g_x_s && a->g_x_t && a->g_x_e && a->g_u &&
                    a->g_w1 && a->g_b1 && a->g_w2 && a->g_b2 && a->g_w3 && a->g_b3 && a->g_w4 && a->g_b4 && a->workspace,
                "null pointer");
    if (a->normed) PFS_REQUIRE(a->gamma && a->bn_save && a->g_gamma && a->g_beta, "normed backward needs norm tensors");
    Topo tp;
    PFS_TRY(make_topo(a->topo, tp));
    PFS_DISPATCH_F(tp.F, return source_bwd_impl<kF>(*a, tp));
    return PFS_OK;
}
int pfs_target_fwd(const pfs_target_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    PFS_REQUIRE(a && a->x_s && a->x_t && a->x_e && a->u && a->w1 && a->b1 && a->w2 && a->b2 && a->w3 && a->b3 && a->w4 &&
                    a->b4 && a->x_t_out && a->act_sum && a->y_pre && a->workspace, "null pointer");
    Topo tp;
    PFS_TRY(make_topo(a->topo, tp));
    PFS_DISPATCH_F(tp.F, return target_fwd_impl<kF>(*a, tp));
    return PFS_OK;
}
int pfs_target_bwd(const pfs_target_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    PFS_REQUIRE(a && a->x_s && a->x_t && a->x_e && a->u && a->w1 && a->b1 && a->w2 && a->b2 && a->w3 && a->b3 && a->w4 &&
                    a->act_sum && a->y_pre && a->g_out && a->g_x_s && a->g_x_t && a->g_x_e && a->g_u && a->g_w1 &&
                    a->g_b1 && a->g_w2 && a->g_b2 && a->g_w3 && a->g_b3 && a->g_w4 && a->g_b4 && a->workspace,
                "null pointer");
    if (a->normed) PFS_REQUIRE(a->gamma && a->bn_save && a->g_gamma && a->g_beta, "normed backward needs norm tensors");
    Topo tp;
    PFS_TRY(make_topo(a->topo, tp));
    PFS_DISPATCH_F(tp.F, return target_bwd_impl<kF>(*a, tp));
    return PFS_OK;
}

static int global_common(const pfs_global_args* a, GlobalParams& p) {
    PFS_REQUIRE(a && a->x_s && a->x_t && a->u && a->w1 && a->b1 && a->w2 && a->b2, "null pointer");
    PFS_REQUIRE(a->G >= 1 && a->F >= 2 && a->S >= 1 && a->T >= 1 && 3 * a->F <= kThreads, "bad sizes");
    if (a->normed) PFS_REQUIRE(a->rms_weight, "normed global model needs norm.weight");
    p = GlobalParams{};
    p.G = a->G; p.F = a->F; p.S = a->S; p.T = a->T; p.normed = a->normed; p.rms_eps = a->rms_eps;
    p.x_s = a->x_s; p.x_t = a->x_t; p.u = a->u;
    p.w1 = a->w1; p.b1 = a->b1; p.w2 = a->w2; p.b2 = a->b2; p.rms_w = a->rms_weight;
    p.u_out = a->u_out; p.gout = a->g_out; p.g_x_s = a->g_x_s; p.g_x_t = a->g_x_t; p.g_u = a->g_u;
    return PFS_OK;
}
int pfs_global_fwd(const pfs_global_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    GlobalParams p;
    PFS_TRY(global_common(a, p));
    PFS_REQUIRE(a->u_out, "null pointer");
    cudaStream_t st = (cudaStream_t)a->stream;
    prof_mark(nullptr, st);
    const size_t smem = sizeof(float) * (kThreads + 14 * (size_t)a->F + 2);
    k_global_fwd<<<a->G, kThreads, smem, st>>>(p);
    PFS_LAUNCH_CHECK("k_global_fwd");
    return PFS_OK;
}
int pfs_global_bwd(const pfs_global_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    GlobalParams p;
    PFS_TRY(global_common(a, p));
    PFS_REQUIRE(a->g_out && a->g_x_s && a->g_x_t && a->g_u && a->g_w1 && a->g_b1 && a->g_w2 && a->g_b2 && a->workspace,
                "null pointer");
    cudaStream_t st = (cudaStream_t)a->stream;
    prof_mark(nullptr, st);
    const int F = a->F, K = 3 * F, pg = global_partial_floats(F);
    Bump ws(a->workspace, a->workspace_bytes);
    float* gpart = ws.f((size_t)a->G * pg);
    if (!ws.ok) return fail(PFS_ERR_WORKSPACE, "global_bwd: workspace too small");
    p.gpartial = gpart;
    const size_t smem = sizeof(float) * (kThreads + 14 * (size_t)F + 2);
    k_global_bwd<<<a->G, kThreads, smem, st>>>(p);
    PFS_LAUNCH_CHECK("k_global_bwd");
    {
        if (a->normed) PFS_REQUIRE(a->g_rms_weight, "null pointer");
        Reducer rd;
        rd.add(glob_off_w1(F), K * K, K, a->g_w1, K, 0);
        rd.add(glob_off_b1(F), K, K, a->g_b1, K, 0);
        rd.add(glob_off_w2(F), F * K, K, a->g_w2, K, 0);
        rd.add(glob_off_b2(F), F, F, a->g_b2, F, 0);
        if (a->normed) rd.add(glob_off_rms(F), F, F, a->g_rms_weight, F, 0);
        PFS_TRY(rd.run(gpart, a->G, pg, st));
    }
    return PFS_OK;
}

int pfs_time_head_fwd(const pfs_head_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    PFS_REQUIRE(a && a->x_e && a->w1 && a->b1 && a->w2 && a->b2 && a->time, "null pointer");
    Topo tp;
    PFS_TRY(make_topo(a->topo, tp));
    PFS_DISPATCH_F(tp.F, return head_impl<kF>(*a, tp, false));
    return PFS_OK;
}
int pfs_time_head_bwd(const pfs_head_args* a) {
    CallGuard guard(a ? a->stream : nullptr);
    PFS_REQUIRE(a && a->x_e && a->w1 && a->b1 && a->w2 && a->b2 && a->g_time && a->g_x_e && a->g_w1 && a->g_b1 &&
                    a->g_w2 && a->g_b2 && a->workspace, "null pointer");
    Topo tp;
    PFS_TRY(make_topo(a->topo, tp));
    PFS_DISPATCH_F(tp.F, return head_impl<kF>(*a, tp, true));
    return PFS_OK;
}

}  // extern "C"
