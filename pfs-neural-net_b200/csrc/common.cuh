// common.cuh -- device-side building blocks shared by every kernel of libpfs_b200.so (sm_100a).
//
// Thread mapping used throughout (DESIGN.md section 4): a CTA of kThreads threads owns one tile of
// at most kTile fibre-sorted edges made of WHOLE fibres.  Per-edge work (the small MLPs) is
// thread-per-edge with the whole row in registers and the weights broadcast from shared memory;
// per-fibre work (moments, fibre sums) and per-class work (class sums) switch to
// thread-per-(segment, feature) over a shared-memory staging of the tile, so every reduction has
// a fixed order: no atomics anywhere, results are bit-reproducible.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pfs_b200.h"

namespace pfs {

constexpr int kTile = PFS_TILE_EDGES;
constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr float kSlope = 0.1f;      // LeakyReLU(0.1) of every MLP (reference src/gnn.py:69)
constexpr float kSlopeVar = 0.01f;  // F.leaky_relu default on the variance (reference src/gnn.py:141)
constexpr float kStdEps = 1e-6f;    // reference src/gnn.py:142,149
constexpr int kNumSM = 148;

__device__ __forceinline__ float lrelu(float x) { return fmaxf(x, kSlope * x); }   // slope < 1
__device__ __forceinline__ float dlrelu(float x) { return x > 0.f ? 1.f : kSlope; }

// ------------------------------------------------------------------------------------------
// topology
// ------------------------------------------------------------------------------------------
struct Topo {
    int layout, G, F, S, T, E;
    const int *rowptr, *eid, *csrc, *ctgt, *tile_fibre;
    int ntiles;  // tiles per graph
    const int *colptr, *cscq;
    int fpt;     // fibres per tile (dense layout)
    // split tiles (CSR layout, a fibre of more than kTile edges): see pfs_topology in include/pfs_b200.h
    const int *tile_q, *tile_slot, *split_fibre, *split_ptr;
    int nsplit, nslots;
};

struct Tile {
    int g, lt, fibre0, nfib, q0, ne;
    int slot;    // partial-record slot of a split tile (one chunk of one fibre), else -1
};

// SPLIT: the topology has split tiles (Topo::nsplit > 0).  The kernels that run on such a topology are separate
// instantiations, so the ones for whole-fibre tables compile exactly as without the split handling.
template <bool SPLIT = false>
__device__ __forceinline__ Tile get_tile(const Topo& tp, int tile) {
    Tile t;
    t.g = tile / tp.ntiles;
    t.lt = tile - t.g * tp.ntiles;
    t.slot = -1;
    if (tp.layout == PFS_LAYOUT_DENSE) {
        t.fibre0 = t.lt * tp.fpt;
        t.nfib = min(tp.fpt, tp.S - t.fibre0);
        t.q0 = t.fibre0 * tp.T;
        t.ne = t.nfib * tp.T;
    } else if constexpr (SPLIT) {
        t.fibre0 = tp.tile_fibre[t.lt];
        t.q0 = tp.tile_q[t.lt];
        t.ne = tp.tile_q[t.lt + 1] - t.q0;
        t.slot = tp.tile_slot[t.lt];
        t.nfib = t.slot >= 0 ? 1 : tp.tile_fibre[t.lt + 1] - t.fibre0;
    } else {
        t.fibre0 = tp.tile_fibre[t.lt];
        const int f1 = tp.tile_fibre[t.lt + 1];
        t.nfib = f1 - t.fibre0;
        t.q0 = tp.rowptr[t.fibre0];
        t.ne = tp.rowptr[f1] - t.q0;
    }
    return t;
}

struct EdgeRef {
    int e, src, tgt;  // row of x_e, fibre, class (all per graph)
};

__device__ __forceinline__ EdgeRef get_edge(const Topo& tp, const Tile& t, int tid) {
    EdgeRef r;
    const int q = t.q0 + tid;
    if (tp.layout == PFS_LAYOUT_DENSE) {
        const int lf = tid / tp.T;
        r.src = t.fibre0 + lf;
        r.tgt = tid - lf * tp.T;
        r.e = q;
    } else {
        r.src = tp.csrc[q];
        r.tgt = tp.ctgt[q];
        r.e = tp.eid ? tp.eid[q] : q;
    }
    return r;
}

// edges of local fibre lf inside the tile: [e0, e0 + n) (SPLIT: clipped to the tile, a split tile holds a chunk)
template <bool SPLIT = false>
__device__ __forceinline__ void fibre_range(const Topo& tp, const Tile& t, int lf, int& e0, int& n) {
    if (tp.layout == PFS_LAYOUT_DENSE) {
        e0 = lf * tp.T;
        n = tp.T;
    } else if constexpr (SPLIT) {
        const int a = max(tp.rowptr[t.fibre0 + lf], t.q0);
        const int b = min(tp.rowptr[t.fibre0 + lf + 1], t.q0 + t.ne);
        e0 = a - t.q0;
        n = b - a;
    } else {
        const int a = tp.rowptr[t.fibre0 + lf];
        e0 = a - t.q0;
        n = tp.rowptr[t.fibre0 + lf + 1] - a;
    }
}

// ------------------------------------------------------------------------------------------
// row loads / stores (rows of F, 2F, 4F floats; F is even so rows are at least 8-byte aligned)
// ------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void load_row(const float* __restrict__ p, float (&x)[N]) {
    if constexpr (N % 4 == 0) {
        const float4* q = reinterpret_cast<const float4*>(p);
#pragma unroll
        for (int i = 0; i < N / 4; ++i) {
            const float4 v = __ldg(q + i);
            x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
        }
    } else {
        const float2* q = reinterpret_cast<const float2*>(p);
#pragma unroll
        for (int i = 0; i < N / 2; ++i) {
            const float2 v = __ldg(q + i);
            x[2 * i] = v.x; x[2 * i + 1] = v.y;
        }
    }
}

template <int N>
__device__ __forceinline__ void add_row(const float* __restrict__ p, float (&x)[N]) {
    if constexpr (N % 4 == 0) {
        const float4* q = reinterpret_cast<const float4*>(p);
#pragma unroll
        for (int i = 0; i < N / 4; ++i) {
            const float4 v = __ldg(q + i);
            x[4 * i] += v.x; x[4 * i + 1] += v.y; x[4 * i + 2] += v.z; x[4 * i + 3] += v.w;
        }
    } else {
        const float2* q = reinterpret_cast<const float2*>(p);
#pragma unroll
        for (int i = 0; i < N / 2; ++i) {
            const float2 v = __ldg(q + i);
            x[2 * i] += v.x; x[2 * i + 1] += v.y;
        }
    }
}

template <int N>
__device__ __forceinline__ void store_row(float* __restrict__ p, const float (&x)[N]) {
    if constexpr (N % 4 == 0) {
        float4* q = reinterpret_cast<float4*>(p);
#pragma unroll
        for (int i = 0; i < N / 4; ++i) q[i] = make_float4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
    } else {
        float2* q = reinterpret_cast<float2*>(p);
#pragma unroll
        for (int i = 0; i < N / 2; ++i) q[i] = make_float2(x[2 * i], x[2 * i + 1]);
    }
}

// shared-memory row store with an arbitrary (even) leading dimension
template <int N>
__device__ __forceinline__ void store_row_smem(float* p, const float (&x)[N]) {
    float2* q = reinterpret_cast<float2*>(p);
#pragma unroll
    for (int i = 0; i < N / 2; ++i) q[i] = make_float2(x[2 * i], x[2 * i + 1]);
}

// ------------------------------------------------------------------------------------------
// weights: global (torch Linear layout W[j][k], leading dimension ld) -> shared memory
// ------------------------------------------------------------------------------------------
// dst[k * J + j] = W[j * ld + koff + k]      ("input-major": forward layers, y_j += W_jk x_k)
template <int K, int J>
__device__ __forceinline__ void load_w_inmajor(float* dst, const float* __restrict__ W, int ld, int koff) {
    for (int i = threadIdx.x; i < J * K; i += blockDim.x) {
        const int j = i / K, k = i - j * K;
        dst[k * J + j] = __ldg(W + (size_t)j * ld + koff + k);
    }
}
// dst[j * K + k] = W[j * ld + koff + k]      ("output-major": backward layers, dx_k += W_jk dy_j)
template <int K, int J>
__device__ __forceinline__ void load_w_outmajor(float* dst, const float* __restrict__ W, int ld, int koff) {
    for (int i = threadIdx.x; i < J * K; i += blockDim.x) {
        const int j = i / K, k = i - j * K;
        dst[j * K + k] = __ldg(W + (size_t)j * ld + koff + k);
    }
}
template <int N>
__device__ __forceinline__ void load_vec(float* dst, const float* __restrict__ v) {
    for (int i = threadIdx.x; i < N; i += blockDim.x) dst[i] = __ldg(v + i);
}

// y[j] += sum_k Wt[k * J + j] * x[k]; Wt in shared memory (every lane reads the same address:
// one broadcast wavefront per LDS.128), x and y in registers.  The multiply-adds are issued as
// packed FFMA2 (fma.rn.f32x2, sm_100+): two output features per instruction, x[k] broadcast.
template <int K, int J>
__device__ __forceinline__ void dense_acc(const float* Wt, const float (&x)[K], float (&y)[J]) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const float2 xx = make_float2(x[k], x[k]);
        if constexpr (J % 4 == 0) {
            const float4* w = reinterpret_cast<const float4*>(Wt + k * J);
#pragma unroll
            for (int j = 0; j < J / 4; ++j) {
                const float4 v = w[j];
                const float2 a = __ffma2_rn(make_float2(v.x, v.y), xx, make_float2(y[4 * j], y[4 * j + 1]));
                const float2 b = __ffma2_rn(make_float2(v.z, v.w), xx, make_float2(y[4 * j + 2], y[4 * j + 3]));
                y[4 * j] = a.x; y[4 * j + 1] = a.y; y[4 * j + 2] = b.x; y[4 * j + 3] = b.y;
            }
        } else {
            const float2* w = reinterpret_cast<const float2*>(Wt + k * J);
#pragma unroll
            for (int j = 0; j < J / 2; ++j) {
                const float2 a = __ffma2_rn(w[j], xx, make_float2(y[2 * j], y[2 * j + 1]));
                y[2 * j] = a.x; y[2 * j + 1] = a.y;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// asynchronous staging of a tile's inputs (global -> shared, double-buffered): the loads of tile
// i+1 are in flight while tile i is computed, so DRAM/L2 latency never sits in front of the FMAs.
// cp.async (LDGSTS) in 8-byte chunks handles every alignment the rows can have (F is even) and
// row gathers; contiguous 16-byte aligned slabs use 16-byte chunks.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async8(float* smem, const float* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async16(float* smem, const float* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// flat copy of `nfloats` floats (even count; both pointers 8-byte aligned)
__device__ __forceinline__ void stage_flat(float* dst, const float* __restrict__ src, int nfloats) {
    const bool a16 = ((((uintptr_t)src) | ((uintptr_t)dst)) & 15) == 0;
    if (a16) {
        const int n4 = nfloats >> 2;
        for (int i = threadIdx.x; i < n4; i += kThreads) cp_async16(dst + 4 * i, src + 4 * i);
        for (int i = (n4 << 2) + 2 * threadIdx.x; i < nfloats; i += 2 * kThreads) cp_async8(dst + i, src + i);
    } else {
        const int n2 = nfloats >> 1;
        for (int i = threadIdx.x; i < n2; i += kThreads) cp_async8(dst + 2 * i, src + 2 * i);
    }
}
// rows of ROW floats: dst[r * LD + c] = src[rowidx(r) * ROW + c]  (gather by an index array, or
// consecutive rows starting at row0 when idx == nullptr)
template <int ROW, int LD, int SRC_LD = ROW>
__device__ __forceinline__ void stage_rows(float* dst, const float* __restrict__ src, long long row0,
                                           const int* __restrict__ idx, int nrows) {
    if (idx == nullptr && LD == ROW && SRC_LD == ROW) {
        stage_flat(dst, src + row0 * ROW, nrows * ROW);
        return;
    }
    constexpr int C = ROW / 2;
    for (int i = threadIdx.x; i < nrows * C; i += kThreads) {
        const int r = i / C, c = i - r * C;
        const long long row = idx ? (row0 + idx[r]) : (row0 + r);
        cp_async8(dst + r * LD + 2 * c, src + row * SRC_LD + 2 * c);
    }
}

// Double-buffered inputs of one tile: NE per-edge tensors (rows of F floats, in CSR order), one
// per-fibre table (rows of PF floats, the tile's fibres are consecutive) and one per-class table
// (rows of PC floats, padded to PC + 4 in shared memory against bank conflicts; staged only
// when it is small enough, else read through L1).  All threads of the CTA call issue().
// TMA bulk copy (cp.async.bulk, 1-D): one elected thread moves a whole contiguous slab global -> shared and the
// bytes land on an mbarrier; addresses and size must be multiples of 16 bytes
__device__ __forceinline__ void bulk_g2s(float* smem, const float* gmem, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     (unsigned)__cvta_generic_to_shared(smem)),
                 "l"(gmem), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar))
                 : "memory");
}
// L2 prefetch of a contiguous slab (no completion, no correctness impact): turns the DRAM latency of the per-thread
// row loads of the NEXT tile into an L2 hit.  Skipped unless address and size are multiples of 16 bytes.
__device__ __forceinline__ void bulk_prefetch_l2(const float* gmem, size_t bytes) {
    if (gmem == nullptr || bytes == 0 || ((((uintptr_t)gmem) | bytes) & 15)) return;
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gmem), "r"((unsigned)bytes) : "memory");
}
__device__ __forceinline__ void stage_bar_init(uint64_t* bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)));
}
__device__ __forceinline__ void stage_bar_expect(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void stage_bar_wait(uint64_t* bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}

template <int F, int NE, int PF, int PC>
struct TileStage {
    static constexpr int PCP = PC + 4;
    float* base;
    uint64_t* bars;          // one mbarrier per buffer (bulk-copied tiles)
    unsigned phase;          // bit b = parity of buffer b's mbarrier
    int per, max_fib;
    bool with_class, dbl;
    // nbuf = 2: double-buffered (tile i+1 in flight while tile i is computed); 1: load-then-compute
    __host__ __device__ static size_t floats(int max_fib, int T, bool with_class, int nbuf = 2) {
        return nbuf * ((size_t)NE * kTile * F + (size_t)max_fib * PF + (with_class ? (size_t)T * PCP : 0)) + 4;   // + 2 mbarriers
    }
    // all threads of the CTA call init(); ends with a __syncthreads()
    __device__ __forceinline__ void init(float* dyn, int max_fib_, int T, bool with_class_, int nbuf = 2) {
        base = dyn;
        max_fib = max_fib_;
        with_class = with_class_;
        dbl = nbuf == 2;
        per = NE * kTile * F + max_fib * PF + (with_class ? T * PCP : 0);
        bars = reinterpret_cast<uint64_t*>(base + (size_t)nbuf * per + ((nbuf * per) & 1));
        phase = 0u;
        if (threadIdx.x == 0) {
            stage_bar_init(bars);
            stage_bar_init(bars + 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
    }
    // A tile of the dense layout is a few contiguous slabs: when every slab is 16-byte aligned and a multiple of
    // 16 bytes it is fetched by TMA bulk copies issued by ONE thread (no per-thread address arithmetic, completion
    // on an mbarrier); otherwise (general edge lists: row gathers; odd sizes) every thread issues cp.async chunks.
    __device__ __forceinline__ bool bulk_ok(const Topo& tp, const Tile& t, const float* const* esrc, const float* fsrc,
                                            const float* csrc) const {
        if (tp.layout != PFS_LAYOUT_DENSE) return false;
        uintptr_t bits = (uintptr_t)base | (uintptr_t)((size_t)per * sizeof(float)) | (uintptr_t)((size_t)t.ne * F * sizeof(float));
#pragma unroll
        for (int i = 0; i < NE; ++i) bits |= (uintptr_t)(esrc[i] + ((size_t)t.g * tp.E + t.q0) * F);
        if constexpr (PF > 0) bits |= (uintptr_t)(fsrc + ((size_t)t.g * tp.S + t.fibre0) * PF) | (uintptr_t)(PF * sizeof(float)) |
                                      (uintptr_t)((size_t)max_fib * PF * sizeof(float));
        if constexpr (PC > 0) {
            if (with_class) bits |= (uintptr_t)(csrc + (size_t)t.g * tp.T * PC) | (uintptr_t)(PC * sizeof(float));
        }
        return (bits & 15) == 0;
    }
    // pipeline step at the top of the loop body for `tile` (buffer parity b): returns the buffer
    // holding this tile once the following __syncthreads() has passed
    template <class GetTile>
    __device__ __forceinline__ int step(const Topo& tp, int tile, int t_end, int b, const float* const* esrc,
                                        const float* fsrc, const float* csrc, GetTile get) {
        if (dbl) {
            if (tile + 1 < t_end) issue(tp, get(tile + 1), b ^ 1, esrc, fsrc, csrc);
            cp_async_commit();
            cp_async_wait<1>();
            wait_bulk(tp, get(tile), b, esrc, fsrc, csrc);
            return b;
        }
        issue(tp, get(tile), 0, esrc, fsrc, csrc);
        cp_async_commit();
        cp_async_wait<0>();
        wait_bulk(tp, get(tile), 0, esrc, fsrc, csrc);
        return 0;
    }
    __device__ __forceinline__ void wait_bulk(const Topo& tp, const Tile& t, int b, const float* const* esrc,
                                              const float* fsrc, const float* csrc) {
        if (bulk_ok(tp, t, esrc, fsrc, csrc)) {
            stage_bar_wait(bars + b, (phase >> b) & 1u);
            phase ^= 1u << b;
        }
    }
    // before the loop: first tile of a double-buffered pipeline
    template <class GetTile>
    __device__ __forceinline__ void prologue(const Topo& tp, int t_begin, int t_end, const float* const* esrc,
                                             const float* fsrc, const float* csrc, GetTile get) const {
        if (dbl) {
            if (t_begin < t_end) issue(tp, get(t_begin), 0, esrc, fsrc, csrc);
            cp_async_commit();
        }
    }
    __device__ __forceinline__ float* edge(int b, int i) const { return base + b * per + i * kTile * F; }
    __device__ __forceinline__ float* fib(int b) const { return base + b * per + NE * kTile * F; }
    __device__ __forceinline__ float* cls(int b) const { return fib(b) + max_fib * PF; }
    // enqueue the copies of tile t into buffer b (no commit: the caller may add more, then commits)
    __device__ __forceinline__ void issue(const Topo& tp, const Tile& t, int b, const float* const* esrc,
                                          const float* fsrc, const float* csrc) const {
        if (bulk_ok(tp, t, esrc, fsrc, csrc)) {
            if (threadIdx.x == 0) {
                const unsigned eb = (unsigned)(t.ne * F * sizeof(float)), fb = (unsigned)(t.nfib * PF * sizeof(float));
                const unsigned cb = (PC > 0 && with_class) ? (unsigned)(tp.T * PC * sizeof(float)) : 0u;
                stage_bar_expect(bars + b, NE * eb + fb + cb);
#pragma unroll
                for (int i = 0; i < NE; ++i) bulk_g2s(edge(b, i), esrc[i] + ((size_t)t.g * tp.E + t.q0) * F, eb, bars + b);
                if constexpr (PF > 0) bulk_g2s(fib(b), fsrc + ((size_t)t.g * tp.S + t.fibre0) * PF, fb, bars + b);
                if constexpr (PC > 0) {
                    if (with_class)      // rows are padded to PCP floats in shared memory: one copy per class row
                        for (int c = 0; c < tp.T; ++c)
                            bulk_g2s(cls(b) + c * PCP, csrc + ((size_t)t.g * tp.T + c) * PC, (unsigned)(PC * sizeof(float)), bars + b);
                }
            }
            return;
        }
        const int* idx = (tp.layout != PFS_LAYOUT_DENSE && tp.eid) ? tp.eid + t.q0 : nullptr;
        const long long row0 = idx ? 0 : t.q0;
#pragma unroll
        for (int i = 0; i < NE; ++i)
            stage_rows<F, F>(edge(b, i), esrc[i] + (size_t)t.g * tp.E * F, row0, idx, t.ne);
        if constexpr (PF > 0) stage_rows<PF, PF>(fib(b), fsrc + (size_t)t.g * tp.S * PF, t.fibre0, nullptr, t.nfib);
        if constexpr (PC > 0) {
            if (with_class) stage_rows<PC, PCP>(cls(b), csrc + (size_t)t.g * tp.T * PC, 0, nullptr, tp.T);
        }
    }
};

// rows out of shared memory (same vector widths as load_row, no read-only-cache hint)
template <int N>
__device__ __forceinline__ void lds_row(const float* p, float (&x)[N]) {
    if constexpr (N % 4 == 0) {
        const float4* q = reinterpret_cast<const float4*>(p);
#pragma unroll
        for (int i = 0; i < N / 4; ++i) {
            const float4 v = q[i];
            x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
        }
    } else {
        const float2* q = reinterpret_cast<const float2*>(p);
#pragma unroll
        for (int i = 0; i < N / 2; ++i) {
            const float2 v = q[i];
            x[2 * i] = v.x; x[2 * i + 1] = v.y;
        }
    }
}
template <int N>
__device__ __forceinline__ void lds_add_row(const float* p, float (&x)[N]) {
    if constexpr (N % 4 == 0) {
        const float4* q = reinterpret_cast<const float4*>(p);
#pragma unroll
        for (int i = 0; i < N / 4; ++i) {
            const float4 v = q[i];
            x[4 * i] += v.x; x[4 * i + 1] += v.y; x[4 * i + 2] += v.z; x[4 * i + 3] += v.w;
        }
    } else {
        const float2* q = reinterpret_cast<const float2*>(p);
#pragma unroll
        for (int i = 0; i < N / 2; ++i) {
            const float2 v = q[i];
            x[2 * i] += v.x; x[2 * i + 1] += v.y;
        }
    }
}

// ------------------------------------------------------------------------------------------
// weights through the uniform datapath: the small MLP weights are warp-uniform operands, so they
// live in __constant__ memory (packed input-major by k_pack_weights, copied with
// cudaMemcpyToSymbolAsync on the launch stream) and reach the FMAs as LDCU.128 -> uniform
// registers -> FFMA R, R, UR, R.  Nothing is replicated per lane, so the shared-memory return
// path (128 B/clk/SM, 4 clk per broadcast LDS.128) no longer caps the FMA pipe at ~25 %.
// ------------------------------------------------------------------------------------------
constexpr int kConstFloats = 15360;   // 60 KB of the 64 KB constant bank
__constant__ __align__(16) float c_w[kConstFloats];

// y[j] += sum_k c_w[OFF + k * J + j] * x[k]   (J even; packed FFMA2 R, R.F32, UR.F32x2, R)
// (LDW = row stride of the packed matrix: a column block of a wider matrix is OFF + first column, LDW = its width)
template <int K, int J, int OFF, int LDW = J>
__device__ __forceinline__ void dense_acc_c(const float (&x)[K], float (&y)[J]) {
    static_assert(J % 2 == 0 && OFF % 2 == 0 && LDW % 2 == 0, "pairs of outputs");
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const float2 xx = make_float2(x[k], x[k]);
#pragma unroll
        for (int j = 0; j < J; j += 2) {
            const float2 a = __ffma2_rn(make_float2(c_w[OFF + k * LDW + j], c_w[OFF + k * LDW + j + 1]), xx,
                                        make_float2(y[j], y[j + 1]));
            y[j] = a.x;
            y[j + 1] = a.y;
        }
    }
}

// constant-bank layout of the SModel / TModel edge kernels (floats; common.cuh: c_w).  The message-MLP weights are
// warp-uniform operands: read as LDCU -> uniform registers -> FFMA2 they do not touch the shared-memory return
// path, whose 128 B/clk/SM capped the broadcast-LDS version of these kernels at ~25 % of the FMA pipe.
//   W1t [F][M] input-major (h_j += W1[j][F+k] x_k), W2t [M][M] input-major, W2o [M][M] as stored
//   (da_k += W2[j][k] dm_j), W1o [M][F] as stored (dx_k += W1[j][F+k] dh_j), b2 [M]
template <int F>
struct MsgEdgeConst {
    static constexpr int M = 2 * F;
    static constexpr int kW1t = 0, kW2t = F * M, kW2o = F * M + M * M, kW1o = F * M + 2 * M * M,
                         kB2 = 2 * F * M + 2 * M * M, kFloats = 2 * F * M + 2 * M * M + M;
};

// packs dst[k * J + j] = W[j * ld + koff + k] (input-major) or dst[j * K + k] (output-major)
struct PackItem {
    const float* W;
    int ld, koff, K, J, transpose, dst_off;   // K inputs, J outputs
};
constexpr int kMaxPack = 8;
struct PackList {
    PackItem it[kMaxPack];
    int n;
};
__global__ void k_pack_weights(const PackList pl, float* __restrict__ dst) {
    for (int q = 0; q < pl.n; ++q) {
        const PackItem& it = pl.it[q];
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < it.J * it.K; i += gridDim.x * blockDim.x) {
            const int j = i / it.K, k = i - j * it.K;
            const float v = __ldg(it.W + (size_t)j * it.ld + it.koff + k);
            dst[it.dst_off + (it.transpose ? k * it.J + j : j * it.K + k)] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------
// warp / block reductions (fixed shuffle tree => deterministic)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// BatchNorm tile statistics, two-pass inside the tile (robust against |mean| >> std):
// every thread holds one row z[N] (inactive threads contribute nothing); writes
// out[0..N) = tile mean, out[N..2N) = sum of squared deviations, out[2N] = count.
// `red` is shared scratch of (kWarps + 1) * N floats.
template <int N>
__device__ __forceinline__ void tile_bn_partial(const float (&z)[N], bool active, int count, float* red,
                                                float* __restrict__ out) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float* mean_s = red + kWarps * N;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const float v = warp_sum(active ? z[j] : 0.f);
        if (lane == 0) red[w * N + j] = v;
    }
    __syncthreads();
    if (threadIdx.x < N) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < kWarps; ++i) s += red[i * N + threadIdx.x];
        mean_s[threadIdx.x] = count > 0 ? s / (float)count : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const float d = active ? z[j] - mean_s[j] : 0.f;
        const float v = warp_sum(d * d);
        if (lane == 0) red[w * N + j] = v;
    }
    __syncthreads();
    if (threadIdx.x < N) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < kWarps; ++i) s += red[i * N + threadIdx.x];
        out[threadIdx.x] = mean_s[threadIdx.x];
        out[N + threadIdx.x] = s;
        if (threadIdx.x == 0) out[2 * N] = (float)count;
    }
    __syncthreads();
}
__host__ __device__ constexpr int bn_partial_stride(int N) { return 2 * N + 2; }

// ------------------------------------------------------------------------------------------
// contiguous tile ranges: CTA c of n owns tiles [c * total / n, (c + 1) * total / n).  A CTA then
// crosses only a few graph boundaries, so per-graph statistics can ride in registers and be
// reduced once per graph segment instead of once per tile.
// ------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ int chunk_begin(int cta, int ncta, int total) {
    return (int)((long long)cta * total / ncta);
}
// records a CTA can emit: graph segments its chunk can touch
__host__ __device__ __forceinline__ int chunk_records(int ncta, int total, int tiles_per_graph) {
    const int chunk = (total + ncta - 1) / ncta;
    return (chunk + tiles_per_graph - 1) / tiles_per_graph + 1;
}

// Running BatchNorm statistics of the rows a thread has seen (shifted by its first row, so the
// single-pass sums do not cancel), flushed once per graph segment into a record
// {mean[N], M2[N], count, graph}: Chan-combined over the warp by a fixed shuffle tree, then
// over the warps in order.  `red` is shared scratch of kWarps * (2N + 1) floats.
template <int N>
struct RunningStats {
    float z0[N], s1[N], s2[N];
    int n;
    __device__ __forceinline__ void reset() {
        n = 0;
#pragma unroll
        for (int j = 0; j < N; ++j) z0[j] = s1[j] = s2[j] = 0.f;
    }
    __device__ __forceinline__ void add(const float (&z)[N]) {
        if (n == 0) {
#pragma unroll
            for (int j = 0; j < N; ++j) z0[j] = z[j];
        }
#pragma unroll
        for (int j = 0; j < N; ++j) {
            const float d = z[j] - z0[j];
            s1[j] += d;
            s2[j] = fmaf(d, d, s2[j]);
        }
        ++n;
    }
    // all threads of the CTA call flush(); writes one record and resets
    __device__ __forceinline__ void flush(float* red, float* __restrict__ rec, int graph) {
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        float cnt = (float)n;
#pragma unroll
        for (int j = 0; j < N; ++j) {
            float c = cnt;
            float mean = n > 0 ? z0[j] + s1[j] / cnt : 0.f;
            float m2 = n > 0 ? fmaxf(s2[j] - s1[j] * s1[j] / cnt, 0.f) : 0.f;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float cb = __shfl_xor_sync(0xffffffffu, c, o);
                const float mb = __shfl_xor_sync(0xffffffffu, mean, o);
                const float qb = __shfl_xor_sync(0xffffffffu, m2, o);
                const float tot = c + cb;
                if (tot > 0.f) {
                    const float delta = mb - mean, fb = cb / tot;
                    mean = fmaf(delta, fb, mean);
                    m2 = m2 + qb + delta * delta * c * fb;
                }
                c = tot;
            }
            if (lane == 0) {
                red[w * (2 * N + 1) + j] = mean;
                red[w * (2 * N + 1) + N + j] = m2;
                if (j == 0) red[w * (2 * N + 1) + 2 * N] = c;
            }
        }
        __syncthreads();
        if (threadIdx.x < N) {
            const int j = threadIdx.x;
            float c = 0.f, mean = 0.f, m2 = 0.f;
#pragma unroll
            for (int i = 0; i < kWarps; ++i) {
                const float cb = red[i * (2 * N + 1) + 2 * N];
                const float tot = c + cb;
                if (cb > 0.f) {
                    const float delta = red[i * (2 * N + 1) + j] - mean, fb = cb / tot;
                    mean = fmaf(delta, fb, mean);
                    m2 = m2 + red[i * (2 * N + 1) + N + j] + delta * delta * c * fb;
                }
                c = tot;
            }
            rec[j] = mean;
            rec[N + j] = m2;
            if (j == 0) {
                rec[2 * N] = c;
                rec[2 * N + 1] = (float)graph;
            }
        }
        __syncthreads();
        reset();
    }
};

// ------------------------------------------------------------------------------------------
// in-tile segment sums over a shared-memory tile X[edge][LD] (W features, 4 per thread, 16-byte loads;
// the edges of a segment are added in their order, so the result does not depend on the mapping)
// ------------------------------------------------------------------------------------------
// out[lf * W + k] = sum over the edges of local fibre lf; `out` points at the row of the tile's first fibre.
// Threads [T0, T0 + NT) of the CTA take part (whole warps).  Two running sums per thread (even / odd edges, added at
// the end) halve the dependent FADD chain and keep 8 loads in flight: these sums are latency-bound, not
// bandwidth-bound (ncu source view of k_edge_bwd2: 16 % of the stall samples sat on their FADDs).
template <int W, int LD, int T0 = 0, int NT = kThreads, bool SPLIT = false>
__device__ __forceinline__ void tile_fibre_sums(const Topo& tp, const Tile& t, const float* X, float* __restrict__ out) {
    static_assert(W % 4 == 0 && LD % 4 == 0 && T0 % 32 == 0 && NT % 32 == 0, "16-byte rows, whole warps");
    constexpr int W4 = W / 4;
    const int tt = (int)threadIdx.x - T0;
    if (tt < 0 || tt >= NT) return;
    for (int i = tt; i < t.nfib * W4; i += NT) {
        const int lf = i / W4, k = (i - lf * W4) * 4;
        int e0, n;
        fibre_range<SPLIT>(tp, t, lf, e0, n);
        const float4* x = reinterpret_cast<const float4*>(X + e0 * LD + k);
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s;
        int e = 0;
#pragma unroll 4
        for (; e + 1 < n; e += 2) {
            const float4 v = x[e * (LD / 4)], v1 = x[(e + 1) * (LD / 4)];
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            s1.x += v1.x; s1.y += v1.y; s1.z += v1.z; s1.w += v1.w;
        }
        if (e < n) {
            const float4 v = x[e * (LD / 4)];
            s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
        s.x += s1.x; s.y += s1.y; s.z += s1.z; s.w += s1.w;
        *reinterpret_cast<float4*>(out + (size_t)lf * W + k) = s;
    }
}
// dense layout (edge lf * T + c belongs to class c): cp[c * W + k] = sum over the tile's fibres.  A lane pair shares
// one (class, 4 features) item: even lane = even fibres, odd lane = odd fibres, one shuffle adds them -- twice the
// threads busy on half the chain (T * W / 4 items alone leave most of the CTA idle when there are few classes).
template <int W, int LD, int T0 = 0, int NT = kThreads>
__device__ __forceinline__ void tile_class_sums(const Topo& tp, const Tile& t, const float* X, float* __restrict__ cp) {
    static_assert(W % 4 == 0 && LD % 4 == 0 && T0 % 32 == 0 && NT % 32 == 0, "16-byte rows, whole warps");
    constexpr int W4 = W / 4;
    const int tt = (int)threadIdx.x - T0;
    if (tt < 0 || tt >= NT) return;
    const int stride = tp.T * (LD / 4);
    const int items = tp.T * W4 * 2;
    for (int base = 0; base < items; base += NT) {      // uniform trip count per warp: the shuffle below is warp-wide
        const int i = base + tt;
        const bool on = i < items;
        const int half = i & 1, ci = on ? (i >> 1) : 0;
        const int c = ci / W4, k = (ci - c * W4) * 4;
        const float4* x = reinterpret_cast<const float4*>(X + c * LD + k);
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        if (on) {
#pragma unroll 4
            for (int lf = half; lf < t.nfib; lf += 2) {
                const float4 v = x[lf * stride];
                s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            }
        }
        s.x += __shfl_xor_sync(0xffffffffu, s.x, 1);
        s.y += __shfl_xor_sync(0xffffffffu, s.y, 1);
        s.z += __shfl_xor_sync(0xffffffffu, s.z, 1);
        s.w += __shfl_xor_sync(0xffffffffu, s.w, 1);
        if (on && half == 0) *reinterpret_cast<float4*>(cp + c * W + k) = s;
    }
}

// Row of the fibre sums of tile t: the fibre table's row of its first fibre, or the tile's partial-record row when the
// tile is one chunk of a split fibre (W floats per row, nslots rows per graph; combined by k_split_sums)
template <bool SPLIT>
__device__ __forceinline__ float* fibre_sum_row(const Topo& tp, const Tile& t, float* table, float* split_part, int W) {
    if constexpr (SPLIT) {
        if (t.slot >= 0) return split_part + ((size_t)t.g * tp.nslots + t.slot) * W;
    }
    return table + ((size_t)t.g * tp.S + t.fibre0) * W;
}

// out[(g, split_fibre[i])][k] = sum of the partial rows of split fibre i, in slot order (W floats per row)
__global__ void k_split_sums(const Topo tp, int W, const float* __restrict__ part, float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)tp.G * tp.nsplit * W) return;
    const int k = (int)(i % W);
    const long long gs = i / W;
    const int g = (int)(gs / tp.nsplit), sf = (int)(gs - (long long)g * tp.nsplit);
    float s = 0.f;
    for (int q = tp.split_ptr[sf]; q < tp.split_ptr[sf + 1]; ++q) s += part[((size_t)g * tp.nslots + q) * W + k];
    out[((size_t)g * tp.S + tp.split_fibre[sf]) * W + k] = s;
}

// ------------------------------------------------------------------------------------------
// outer-product accumulation  dW[J][K] += sum_r D[r][0..J) (x) X[r][0..K)
// D and X are shared-memory tiles with leading dimensions ldD / ldX.  The J x K result is
// register-blocked TJ x TK per thread; rows are split over `groups` thread groups and the
// groups are summed in a fixed order by flush().
// ------------------------------------------------------------------------------------------
template <int J, int K, int TJ, int TK, int T0 = 0, int NT = kThreads>
struct OuterAcc {
    // threads [T0, T0 + NT) of the CTA take part; the others hold no accumulators in use
    static_assert(J % TJ == 0 && K % TK == 0, "block must divide the matrix");
    static constexpr int NB = (J / TJ) * (K / TK);
    static_assert(NB <= NT, "too many blocks for the thread range");
    static constexpr int GROUPS = NT / NB;
    static constexpr int kScratchFloats = GROUPS * J * K;
    float acc[TJ][TK];
    int grp, j0, k0;
    bool live;

    __device__ __forceinline__ void init() {
        const int t = (int)threadIdx.x - T0;
        grp = t >= 0 ? t / NB : GROUPS;
        live = t >= 0 && grp < GROUPS;
        const int b = t >= 0 ? t - grp * NB : 0;
        j0 = (b / (K / TK)) * TJ;
        k0 = (b % (K / TK)) * TK;
#pragma unroll
        for (int a = 0; a < TJ; ++a)
#pragma unroll
            for (int c = 0; c < TK; ++c) acc[a][c] = 0.f;
    }
    __device__ __forceinline__ void fma_row(const float (&d)[TJ], const float (&x)[TK]) {
        if constexpr (TJ % 2 == 0) {
            // packed FFMA2 over row pairs (a, a+1), x[c] broadcast
#pragma unroll
            for (int a = 0; a < TJ; a += 2)
#pragma unroll
                for (int c = 0; c < TK; ++c) {
                    const float2 v = __ffma2_rn(make_float2(d[a], d[a + 1]), make_float2(x[c], x[c]),
                                                make_float2(acc[a][c], acc[a + 1][c]));
                    acc[a][c] = v.x;
                    acc[a + 1][c] = v.y;
                }
        } else {
#pragma unroll
            for (int a = 0; a < TJ; ++a)
#pragma unroll
                for (int c = 0; c < TK; ++c) acc[a][c] = fmaf(d[a], x[c], acc[a][c]);
        }
    }
    // A = alignment of p in floats the CALLER guarantees (4: 16 bytes, 2: 8 bytes, 1: none), 0 = test the address at
    // run time.  The run-time test costs two S2R (shared window of the generic address), two branches and a
    // duplicated load sequence per row in the hot loop (profiles/r02_outer_align.txt): the edge kernels pass A.
    template <int N, int A = 0>
    static __device__ __forceinline__ void load_vec_smem(const float* p, float (&v)[N]) {
        if constexpr (A == 4 && N % 4 == 0) {
#pragma unroll
            for (int i = 0; i < N / 4; ++i) {
                const float4 t = reinterpret_cast<const float4*>(p)[i];
                v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
            }
        } else if constexpr ((A == 2 || A == 4) && N % 2 == 0) {
#pragma unroll
            for (int i = 0; i < N / 2; ++i) {
                const float2 t = reinterpret_cast<const float2*>(p)[i];
                v[2 * i] = t.x; v[2 * i + 1] = t.y;
            }
        } else if constexpr (A != 0) {
#pragma unroll
            for (int i = 0; i < N; ++i) v[i] = p[i];
        } else {
        // widest aligned loads the address allows (p's alignment is uniform over the loop)
        if ((N % 4 == 0) && ((((uintptr_t)p) & 15) == 0)) {
#pragma unroll
            for (int i = 0; i < N / 4; ++i) {
                const float4 t = reinterpret_cast<const float4*>(p)[i];
                v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
            }
        } else if ((N % 2 == 0) && ((((uintptr_t)p) & 7) == 0)) {
#pragma unroll
            for (int i = 0; i < N / 2; ++i) {
                const float2 t = reinterpret_cast<const float2*>(p)[i];
                v[2 * i] = t.x; v[2 * i + 1] = t.y;
            }
        } else {
#pragma unroll
            for (int i = 0; i < N; ++i) v[i] = p[i];
        }
        }
    }
    // two rows per iteration: both rows' loads are in flight before the first FMA needs them
    // AD / AX: alignment (floats) of D + r * ldD + j0 and X + r * ldX + k0 guaranteed by the caller for every row and
    // block (0 = run-time test, see load_vec_smem)
    template <int AD = 0, int AX = 0>
    __device__ __forceinline__ void accumulate(const float* D, int ldD, const float* X, int ldX, int rows) {
        if (!live) return;
        int r = grp;
        for (; r + GROUPS < rows; r += 2 * GROUPS) {
            float d0[TJ], x0[TK], d1[TJ], x1[TK];
            load_vec_smem<TJ, AD>(D + r * ldD + j0, d0);
            load_vec_smem<TK, AX>(X + r * ldX + k0, x0);
            load_vec_smem<TJ, AD>(D + (r + GROUPS) * ldD + j0, d1);
            load_vec_smem<TK, AX>(X + (r + GROUPS) * ldX + k0, x1);
            fma_row(d0, x0);
            fma_row(d1, x1);
        }
        if (r < rows) {
            float d0[TJ], x0[TK];
            load_vec_smem<TJ, AD>(D + r * ldD + j0, d0);
            load_vec_smem<TK, AX>(X + r * ldX + k0, x0);
            fma_row(d0, x0);
        }
    }
    // Sums the groups through `scratch` (kScratchFloats floats of shared memory, may alias the
    // tiles) and writes the CTA's partial to out[j * ldo + ko + k].  Call with ALL threads of the CTA.
    __device__ __forceinline__ void flush(float* scratch, float* __restrict__ out, int ldo, int ko) {
        __syncthreads();
        if (live) {
#pragma unroll
            for (int a = 0; a < TJ; ++a)
#pragma unroll
                for (int c = 0; c < TK; ++c) scratch[grp * (J * K) + (j0 + a) * K + k0 + c] = acc[a][c];
        }
        __syncthreads();
        for (int i = threadIdx.x; i < J * K; i += kThreads) {
            float s = 0.f;
            for (int g = 0; g < GROUPS; ++g) s += scratch[g * (J * K) + i];
            const int j = i / K, k = i - j * K;
            out[j * ldo + ko + k] = s;
        }
        __syncthreads();
    }
};

// OuterAcc with the accumulators passed in by the caller: two accumulations that run on disjoint thread ranges
// of a CTA (each thread is live in exactly one) can share ONE register array instead of holding one each.
template <int J, int K, int TJ, int TK, int T0 = 0, int NT = kThreads>
struct OuterAccX {
    static_assert(J % TJ == 0 && K % TK == 0 && TJ % 2 == 0, "block must divide the matrix, row pairs");
    static constexpr int NB = (J / TJ) * (K / TK);
    static_assert(NB <= NT, "too many blocks for the thread range");
    static constexpr int GROUPS = NT / NB;
    static constexpr int kScratchFloats = GROUPS * J * K;
    static constexpr int kAcc = TJ * TK;
    int grp, j0, k0;
    bool live;
    // the FFMA2 operand pair (rows a, a+1 of column c) sits in two ADJACENT slots whatever the block shape, so two
    // accumulations of different shapes can share the register array without repacking moves
    static __device__ __forceinline__ constexpr int slot(int a, int c) { return ((a >> 1) * TK + c) * 2 + (a & 1); }
    __device__ __forceinline__ void init() {
        const int t = (int)threadIdx.x - T0;
        grp = t >= 0 ? t / NB : GROUPS;
        live = t >= 0 && grp < GROUPS;
        const int b = t >= 0 ? t - grp * NB : 0;
        j0 = (b / (K / TK)) * TJ;
        k0 = (b % (K / TK)) * TK;
    }
    template <int NA>
    __device__ __forceinline__ void fma_row(float (&A)[NA], const float (&d)[TJ], const float (&x)[TK]) const {
        static_assert(NA >= kAcc, "accumulator array too small");
#pragma unroll
        for (int a = 0; a < TJ; a += 2)
#pragma unroll
            for (int c = 0; c < TK; ++c) {
                const float2 v = __ffma2_rn(make_float2(d[a], d[a + 1]), make_float2(x[c], x[c]),
                                            make_float2(A[slot(a, c)], A[slot(a + 1, c)]));
                A[slot(a, c)] = v.x;
                A[slot(a + 1, c)] = v.y;
            }
    }
    template <int AD = 0, int AX = 0, int NA>
    __device__ __forceinline__ void accumulate(float (&A)[NA], const float* D, int ldD, const float* X, int ldX, int rows) const {
        if (!live) return;
        using Base = OuterAcc<J, K, TJ, TK, T0, NT>;
        int r = grp;
        for (; r + GROUPS < rows; r += 2 * GROUPS) {
            float d0[TJ], x0[TK], d1[TJ], x1[TK];
            Base::template load_vec_smem<TJ, AD>(D + r * ldD + j0, d0);
            Base::template load_vec_smem<TK, AX>(X + r * ldX + k0, x0);
            Base::template load_vec_smem<TJ, AD>(D + (r + GROUPS) * ldD + j0, d1);
            Base::template load_vec_smem<TK, AX>(X + (r + GROUPS) * ldX + k0, x1);
            fma_row(A, d0, x0);
            fma_row(A, d1, x1);
        }
        if (r < rows) {
            float d0[TJ], x0[TK];
            Base::template load_vec_smem<TJ, AD>(D + r * ldD + j0, d0);
            Base::template load_vec_smem<TK, AX>(X + r * ldX + k0, x0);
            fma_row(A, d0, x0);
        }
    }
    // call with ALL threads of the CTA
    template <int NA>
    __device__ __forceinline__ void flush(const float (&A)[NA], float* scratch, float* __restrict__ out, int ldo, int ko) const {
        __syncthreads();
        if (live) {
#pragma unroll
            for (int a = 0; a < TJ; ++a)
#pragma unroll
                for (int c = 0; c < TK; ++c) scratch[grp * (J * K) + (j0 + a) * K + k0 + c] = A[slot(a, c)];
        }
        __syncthreads();
        for (int i = threadIdx.x; i < J * K; i += kThreads) {
            float s = 0.f;
            for (int g = 0; g < GROUPS; ++g) s += scratch[g * (J * K) + i];
            const int j = i / K, k = i - j * K;
            out[j * ldo + ko + k] = s;
        }
        __syncthreads();
    }
};

}  // namespace pfs
