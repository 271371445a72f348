// edge_model.cuh -- EdgeModel kernels (reference src/gnn.py:73-101).
//
// forward : z = W2 . lrelu(P_s[src] + P_t[tgt] + W1_e . x_e) + b2 per edge (thread-per-edge), with the
//           BatchNorm tile statistics of z; the double BatchNorm is then one per-feature affine.
// backward: recompute the hidden layer, closed-form double-BatchNorm backward, input gradients in
//           registers, weight gradients as a CTA-wide outer-product accumulation over the tile,
//           fibre sums / class sums of dh for the node tables.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace pfs {

struct EdgeFwdParams {
    Topo tp;
    const float* x_e;   // [G,E,F]
    const float* Ps;    // [G,S,4F]
    const float* Pt;    // [G,T,4F]  (includes W1_u.u + b1)
    const float* w1;    // [4F,4F]
    const float* w2;    // [F,4F]
    const float* b2;    // [F]
    float* z_out;       // [G,E,F]
    float* bn_partial;  // [ncta,nrec,2F+2] statistics records, or null
    int max_fib;        // most fibres a tile can hold (sizes the staging buffers)
    int stage_class;    // 1: the class table P_t is staged in shared memory too
    int nrec;           // statistics records per CTA (chunk_records)
    int nbuf;           // staging buffers (2 = prefetch the next tile)
};

template <int F, bool SPLIT = false>
__global__ void __launch_bounds__(kThreads, 2) k_edge_fwd(const EdgeFwdParams p) {
    constexpr int H = 4 * F;
    using Stage = TileStage<F, 1, H, H>;
    // constant-memory layout written by edge_fwd_impl: W1_e input-major [F][H], W2 input-major [H][F], b2 [F]
    constexpr int kW1 = 0, kW2 = F * H, kB2 = 2 * F * H;
    __shared__ float red[kWarps * (2 * F + 1)];
    extern __shared__ __align__(16) float dyn[];
    const Topo& tp = p.tp;
    Stage stg;
    stg.init(dyn, p.max_fib, tp.T, p.stage_class != 0, p.nbuf);
    const float* esrc[1] = {p.x_e};
    auto tile_of = [&](int i) { return get_tile<SPLIT>(tp, i); };
    const int total = tp.ntiles * tp.G;
    const int t_begin = chunk_begin(blockIdx.x, gridDim.x, total), t_end = chunk_begin(blockIdx.x + 1, gridDim.x, total);
    RunningStats<F> rs;
    rs.reset();
    float* rec = p.bn_partial ? p.bn_partial + (size_t)blockIdx.x * p.nrec * bn_partial_stride(F) : nullptr;
    int slot = 0, cur_graph = -1, par = 0;
    stg.prologue(tp, t_begin, t_end, esrc, p.Ps, p.Pt, tile_of);
    for (int tile = t_begin; tile < t_end; ++tile, par ^= 1) {
        const Tile t = get_tile<SPLIT>(tp, tile);
        const int b = stg.step(tp, tile, t_end, par, esrc, p.Ps, p.Pt, tile_of);   // this tile's copies have landed
        if (rec && t.g != cur_graph) {   // graph boundary: emit the finished graph's statistics
            if (cur_graph >= 0) rs.flush(red, rec + (size_t)(slot++) * bn_partial_stride(F), cur_graph);
            cur_graph = t.g;
        }
        __syncthreads();
        if (threadIdx.x < t.ne) {
            const EdgeRef er = get_edge(tp, t, threadIdx.x);
            float x[F], h[H], z[F];
            lds_row<F>(stg.edge(b, 0) + threadIdx.x * F, x);
            lds_row<H>(stg.fib(b) + (er.src - t.fibre0) * H, h);
            if (p.stage_class) lds_add_row<H>(stg.cls(b) + er.tgt * Stage::PCP, h);
            else add_row<H>(p.Pt + ((size_t)t.g * tp.T + er.tgt) * H, h);
            dense_acc_c<F, H, kW1>(x, h);
#pragma unroll
            for (int j = 0; j < H; ++j) h[j] = lrelu(h[j]);
#pragma unroll
            for (int j = 0; j < F; ++j) z[j] = c_w[kB2 + j];
            dense_acc_c<H, F, kW2>(h, z);
            store_row<F>(p.z_out + ((size_t)t.g * tp.E + er.e) * F, z);
            if (rec) rs.add(z);
        }
        __syncthreads();     // the staging buffer is refilled two iterations later
    }
    if (rec) {
        if (cur_graph >= 0) rs.flush(red, rec + (size_t)(slot++) * bn_partial_stride(F), cur_graph);
        for (; slot < p.nrec; ++slot)      // unused records: count 0
            if (threadIdx.x == 0) rec[(size_t)slot * bn_partial_stride(F) + 2 * F] = 0.f;
    }
}

// ------------------------------------------------------------------------------------------
// backward statistics of the (double) BatchNorm over the edges of each graph:
// partial[tile][0..F) = sum g, partial[tile][F..2F) = sum g * xhat1, xhat1 = (x_e_out - beta) * inv
// ------------------------------------------------------------------------------------------
struct EdgeBnStatParams {
    Topo tp;
    const float* xe2;    // [G,E,F] forward output
    const float* gout;   // [G,E,F]
    const float* coef;   // [G,6,F]: A, c1, c2, inv, beta, (unused)   -- only inv and beta are read here
    float* partial;      // [G*ntiles][2F]
};

// A CTA owns a contiguous range of tiles; the rows' contributions are summed per thread over a whole graph segment
// of that range and reduced over the CTA ONCE per segment (not once per tile: the 2F warp-shuffle trees per tile
// made this streaming kernel instruction-bound at half the HBM rate).  The segment's sums go to the slot of its
// first tile, the other tiles of the segment get zeros, so the per-graph consumer (k_tile_partial_sums) is unchanged.
template <int F, bool SPLIT = false>
__global__ void __launch_bounds__(kThreads) k_edge_bn_bwd_stats(const EdgeBnStatParams p) {
    __shared__ float red[kWarps * 2 * F];
    const Topo& tp = p.tp;
    const int total = tp.ntiles * tp.G;
    const int t_begin = chunk_begin(blockIdx.x, gridDim.x, total), t_end = chunk_begin(blockIdx.x + 1, gridDim.x, total);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float sg[F], sx[F];
#pragma unroll
    for (int j = 0; j < F; ++j) sg[j] = sx[j] = 0.f;
    int seg_first = t_begin;
    for (int tile = t_begin; tile < t_end; ++tile) {
        const Tile t = get_tile<SPLIT>(tp, tile);
        if (threadIdx.x < t.ne) {
            const EdgeRef er = get_edge(tp, t, threadIdx.x);
            const size_t row = ((size_t)t.g * tp.E + er.e) * F;
            float g[F], xh[F];
            load_row<F>(p.gout + row, g);
            load_row<F>(p.xe2 + row, xh);
            const float* c = p.coef + (size_t)t.g * 6 * F;
#pragma unroll
            for (int j = 0; j < F; ++j) {
                const float v = (xh[j] - __ldg(c + 4 * F + j)) * __ldg(c + 3 * F + j);
                sg[j] += g[j];
                sx[j] = fmaf(g[j], v, sx[j]);
            }
        }
        const bool last = (tile + 1 == t_end) || ((tile + 1) / tp.ntiles != t.g);
        if (tile != seg_first && threadIdx.x < 2 * F) p.partial[(size_t)tile * 2 * F + threadIdx.x] = 0.f;
        if (last) {
#pragma unroll
            for (int j = 0; j < F; ++j) {
                const float a = warp_sum(sg[j]);
                const float b = warp_sum(sx[j]);
                if (lane == 0) {
                    red[w * 2 * F + j] = a;
                    red[w * 2 * F + F + j] = b;
                }
                sg[j] = sx[j] = 0.f;
            }
            __syncthreads();
            if (threadIdx.x < 2 * F) {
                float s = 0.f;
#pragma unroll
                for (int i = 0; i < kWarps; ++i) s += red[i * 2 * F + threadIdx.x];
                p.partial[(size_t)seg_first * 2 * F + threadIdx.x] = s;
            }
            __syncthreads();
            seg_first = tile + 1;
        }
    }
}

// Per-graph coefficient vectors of the closed-form backward (tests/kernel_model.py: edge_bwd).
//   stage 0 (before the statistics pass): coef[g] = {A, 0, 0, inv, beta}
//   stage 1 (after it): fills c1 = mean g, c2 = mean(g xhat1) * kappa and the per-graph
//            gamma / beta gradients dgb[g][0..F) , dgb[g][F..2F)
// mode: 0 = not normed, 1 = train, 2 = eval
__global__ void k_edge_bn_bwd_coef(int stage, int mode, int F, int G, int ntiles, long long n_rows,
                                   const float* __restrict__ save, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, const float* __restrict__ rm,
                                   const float* __restrict__ rv, float eps, const double* __restrict__ sums,
                                   float* __restrict__ coef, float* __restrict__ dgb) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G * F) return;
    const int g = i / F, f = i - g * F;
    float* c = coef + (size_t)g * 6 * F;
    if (mode == 0) {
        c[f] = 1.f; c[F + f] = 0.f; c[2 * F + f] = 0.f; c[3 * F + f] = 0.f; c[4 * F + f] = 0.f;
        return;
    }
    const double gm = gamma[f], bt = beta[f];
    const float* s = save + (size_t)g * 4 * F;
    if (mode == 2) {
        // eval: y1 = a (z - m) + bt, y2 = a (y1 - m) + bt, dz = a^2 g
        const double cc = 1.0 / sqrt((double)rv[f] + (double)eps), a = gm * cc, m = rm[f];
        if (stage == 0) {
            c[f] = (float)(a * a); c[F + f] = 0.f; c[2 * F + f] = 0.f;
            // xhat slot is reused to recover z: z = (xe2 - shift) / A
            c[3 * F + f] = (a != 0.0) ? (float)(1.0 / (a * a)) : 0.f;
            c[4 * F + f] = s[3 * F + f];
        } else {
            // sum g and sum g * z come from the statistics pass (xhat == z here)
            const double sg = sums[(size_t)g * 2 * F + f], sgz = sums[(size_t)g * 2 * F + F + f];
            // dgamma = sum g c [(y1 - m) + a (z - m)] = c [ 2a (sgz - m sg) + (bt - m) sg ]
            dgb[(size_t)g * 2 * F + f] = (float)(cc * (2.0 * a * (sgz - m * sg) + (bt - m) * sg));
            dgb[(size_t)g * 2 * F + F + f] = (float)((a + 1.0) * sg);
        }
        return;
    }
    const double var = s[F + f];
    const double r1 = 1.0 / sqrt(var + (double)eps);
    const double var2 = gm * gm * var * r1 * r1;
    const double r2 = 1.0 / sqrt(var2 + (double)eps);
    if (stage == 0) {
        c[f] = (float)(gm * gm * r1 * r2);
        c[F + f] = 0.f;
        c[2 * F + f] = 0.f;
        c[3 * F + f] = (gm != 0.0) ? (float)(1.0 / (gm * gm * r2)) : 0.f;
        c[4 * F + f] = (float)bt;
        return;
    }
    const double sg = sums[(size_t)g * 2 * F + f];
    const double sgx = sums[(size_t)g * 2 * F + F + f];
    const double n = (double)n_rows;
    const double gbar = sg / n, mgx = sgx / n;
    const double sc = gm * r2, q = var * r1 * r1;
    const double kappa = sc * sc + 1.0 - sc * sc * q;
    c[F + f] = (float)gbar;
    c[2 * F + f] = (float)(mgx * kappa);
    dgb[(size_t)g * 2 * F + f] = (float)(n * mgx * sc * (2.0 - sc * sc * q));
    dgb[(size_t)g * 2 * F + F + f] = (float)(n * gbar);
}

struct EdgeBwdParams {
    Topo tp;
    const float *x_e, *xe2, *gout;   // [G,E,F]
    const float *Ps, *Pt;            // [G,S,4F], [G,T,4F]
    const float* coef;               // [G,6,F]
    float* g_x_e;                    // [G,E,F]
    float* dPs;                      // [G,S,4F] fibre sums of dh
    float* class_part;               // dense: [G,ntiles,T,4F]
    float* dh_rows;                  // general: [G,E(q),4F]
    float* wpartial;                 // [ncta][pstride]: dW1_e [4F*F], dW2 [F*4F], db2 [F]
    int pstride;
    int max_fib, stage_class, nbuf;
    float* dPs_split;                // split tiles: [G,nslots,4F] partial fibre sums of dh (k_split_sums -> dPs)
};

// constant-bank layout of the edge backward (floats): W1_e input-major [F][H] (recompute h),
// W2 as stored [F][H] (da_k += W2[j][k] dz_j), W1_e as stored [H][F] (dx_k += W1[j][2F+k] dh_j)
template <int F>
struct EdgeBwdConst {
    static constexpr int H = 4 * F;
    static constexpr int kW1t = 0, kW2o = F * H, kW1o = 2 * F * H, kFloats = 3 * F * H;
};

template <int F>
struct EdgeBwdSmem {
    static constexpr int H = 4 * F;
    static constexpr int LDH = H + 4;   // 16-byte aligned rows, bank-staggered
    static constexpr int LDF = F + 2;
    using Stage = TileStage<F, 3, H, H>;
    using AccW1 = OuterAcc<H, F, 8, F / 2, 0, kThreads / 2>;              // dW1_e[j][k] = sum dh_j x_k
    using AccW2 = OuterAcc<F, H, 2, 2 * F, kThreads / 2, kThreads / 2>;   // dW2[j][k]   = sum dz_j a1_k
    static constexpr int kTiles = kTile * (2 * LDH + LDF);
    static size_t bytes(int max_fib, int T, bool with_class, int nbuf) {
        return sizeof(float) * ((size_t)kTiles + Stage::floats(max_fib, T, with_class, nbuf));
    }
    // lean variant (two CTAs per SM): only x_e is staged (single buffer, it is needed in shared memory for dW1_e);
    // the other per-edge rows and the node tables are read straight from global / L1, the second resident CTA
    // hides their latency
    using StageLean = TileStage<F, 1, 0, 0>;
    static constexpr size_t bytes_lean = sizeof(float) * ((size_t)kTiles + (size_t)kTile * F + 4);   // + one x_e buffer, 2 mbarriers
    static constexpr bool lean_fits = bytes_lean <= 113 * 1024;
};

template <int F, bool SPLIT = false>
__global__ void __launch_bounds__(kThreads) k_edge_bwd(const EdgeBwdParams p) {
    constexpr int H = 4 * F;
    using SM = EdgeBwdSmem<F>;
    using CW = EdgeBwdConst<F>;
    using Stage = typename SM::Stage;
    constexpr int LDH = SM::LDH, LDF = SM::LDF;
    extern __shared__ __align__(16) float sm[];
    float* DH = sm;                  // [kTile][LDH]
    float* A1 = DH + kTile * LDH;    // [kTile][LDH]
    float* DZ = A1 + kTile * LDH;    // [kTile][LDF]
    const Topo& tp = p.tp;
    Stage stg;
    stg.init(DZ + kTile * LDF, p.max_fib, tp.T, p.stage_class != 0, p.nbuf);
    auto tile_of = [&](int i) { return get_tile<SPLIT>(tp, i); };
    // the two weight-gradient accumulations run side by side on the two halves of the CTA
    typename SM::AccW1 accw1;
    typename SM::AccW2 accw2;
    accw1.init();
    accw2.init();
    float dzsum[F];
#pragma unroll
    for (int j = 0; j < F; ++j) dzsum[j] = 0.f;
    const float* esrc[3] = {p.x_e, p.xe2, p.gout};
    const int total = tp.ntiles * tp.G;
    const int t_begin = chunk_begin(blockIdx.x, gridDim.x, total), t_end = chunk_begin(blockIdx.x + 1, gridDim.x, total);
    int par = 0;
    stg.prologue(tp, t_begin, t_end, esrc, p.Ps, p.Pt, tile_of);
    for (int tile = t_begin; tile < t_end; ++tile, par ^= 1) {
        const Tile t = get_tile<SPLIT>(tp, tile);
        const int b = stg.step(tp, tile, t_end, par, esrc, p.Ps, p.Pt, tile_of);
        __syncthreads();
        const float* XE = stg.edge(b, 0);
        if (threadIdx.x < t.ne) {
            const EdgeRef er = get_edge(tp, t, threadIdx.x);
            float x[F], h[H], dz[F];
            lds_row<F>(XE + threadIdx.x * F, x);
            lds_row<H>(stg.fib(b) + (er.src - t.fibre0) * H, h);
            if (p.stage_class) lds_add_row<H>(stg.cls(b) + er.tgt * Stage::PCP, h);
            else add_row<H>(p.Pt + ((size_t)t.g * tp.T + er.tgt) * H, h);
            dense_acc_c<F, H, CW::kW1t>(x, h);
            {
                float gr[F], xo[F];
                lds_row<F>(stg.edge(b, 2) + threadIdx.x * F, gr);
                lds_row<F>(stg.edge(b, 1) + threadIdx.x * F, xo);
                const float* c = p.coef + (size_t)t.g * 6 * F;
#pragma unroll
                for (int j = 0; j < F; ++j) {
                    const float xh = (xo[j] - __ldg(c + 4 * F + j)) * __ldg(c + 3 * F + j);
                    dz[j] = __ldg(c + j) * (gr[j] - __ldg(c + F + j) - xh * __ldg(c + 2 * F + j));
                    dzsum[j] += dz[j];
                }
            }
            float da[H];
#pragma unroll
            for (int k = 0; k < H; ++k) da[k] = 0.f;
            dense_acc_c<F, H, CW::kW2o>(dz, da);
            store_row_smem<F>(DZ + threadIdx.x * LDF, dz);
#pragma unroll
            for (int k = 0; k < H; ++k) {
                da[k] *= dlrelu(h[k]);      // dh
                h[k] = lrelu(h[k]);         // a1
            }
            store_row_smem<H>(A1 + threadIdx.x * LDH, h);
            store_row_smem<H>(DH + threadIdx.x * LDH, da);
            float dx[F];
#pragma unroll
            for (int k = 0; k < F; ++k) dx[k] = 0.f;
            dense_acc_c<H, F, CW::kW1o>(da, dx);
            store_row<F>(p.g_x_e + ((size_t)t.g * tp.E + er.e) * F, dx);
            if (p.dh_rows) store_row<H>(p.dh_rows + ((size_t)t.g * tp.E + t.q0 + threadIdx.x) * H, da);
        }
        __syncthreads();
        accw1.accumulate(DH, LDH, XE, F, t.ne);
        accw2.accumulate(DZ, LDF, A1, LDH, t.ne);
        // fibre sums of dh -> dPs, class sums of dh (dense layout: edge lf*T + c belongs to class c)
        tile_fibre_sums<H, LDH, 0, kThreads, SPLIT>(tp, t, DH, fibre_sum_row<SPLIT>(tp, t, p.dPs, p.dPs_split, H));
        if (p.class_part) tile_class_sums<H, LDH>(tp, t, DH, p.class_part + (size_t)tile * tp.T * H);
        __syncthreads();
    }
    cp_async_wait<0>();
    float* out = p.wpartial + (size_t)blockIdx.x * p.pstride;
    accw1.flush(DH, out, F, 0);
    accw2.flush(DH, out + H * F, H, 0);
    // db2 = sum dz: block reduction of the per-thread sums
    {
        float* red = DH;
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
        for (int j = 0; j < F; ++j) {
            const float v = warp_sum(dzsum[j]);
            if (lane == 0) red[w * F + j] = v;
        }
        __syncthreads();
        if (threadIdx.x < F) {
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < kWarps; ++i) s += red[i * F + threadIdx.x];
            out[2 * H * F + threadIdx.x] = s;
        }
    }
}

// ------------------------------------------------------------------------------------------
// k_edge_bwd2: the same backward shaped for TWO CTAs per SM (<= 128 registers, 113 KB of shared memory; at Fdim 16,
// where its 170 KB allow one CTA per SM, it runs where k_edge_bwd's staged tiles do not fit and has all registers):
//   * only x_e is staged (single buffer: it has to be in shared memory for dW1_e); the other per-edge rows and
//     the node tables come straight from global / L1, the second resident CTA hides their latency;
//   * the hidden layer is processed in two halves of 2F units (h, dh: 2F live registers each instead of 4F);
//   * the two weight-gradient accumulations run on the two halves of the CTA and SHARE one register array;
//   * db2 = sum dz is taken from the staged dz rows instead of a per-thread running sum.
// ------------------------------------------------------------------------------------------
template <int F, int HALF>
__device__ __forceinline__ void edge_bwd_half(const EdgeBwdParams& p, const float* __restrict__ ps, const float* __restrict__ pt,
                                              const float (&x)[F], const float (&dz)[F], float (&dx)[F], float* A1row,
                                              float* DHrow, float* dh_row_out) {
    constexpr int H = 4 * F, HH = 2 * F;
    using CW = EdgeBwdConst<F>;
    float hh[HH], da[HH];
    load_row<HH>(ps + HALF * HH, hh);
    add_row<HH>(pt + HALF * HH, hh);
    dense_acc_c<F, HH, CW::kW1t + HALF * HH, H>(x, hh);
#pragma unroll
    for (int k = 0; k < HH; ++k) da[k] = 0.f;
    dense_acc_c<F, HH, CW::kW2o + HALF * HH, H>(dz, da);
#pragma unroll
    for (int k = 0; k < HH; ++k) {
        da[k] *= dlrelu(hh[k]);      // dh
        hh[k] = lrelu(hh[k]);        // a1
    }
    store_row_smem<HH>(A1row + HALF * HH, hh);
    store_row_smem<HH>(DHrow + HALF * HH, da);
    dense_acc_c<HH, F, CW::kW1o + HALF * HH * F, F>(da, dx);
    if (dh_row_out) store_row<HH>(dh_row_out + HALF * HH, da);
}

template <int F, bool SPLIT = false>
__global__ void __launch_bounds__(kThreads, EdgeBwdSmem<F>::lean_fits ? 2 : 1) k_edge_bwd2(const EdgeBwdParams p) {
    constexpr int H = 4 * F;
    using SM = EdgeBwdSmem<F>;
    using Stage = typename SM::StageLean;
    constexpr int LDH = SM::LDH, LDF = SM::LDF;
    extern __shared__ __align__(16) float sm[];
    float* DH = sm;                  // [kTile][LDH]
    float* A1 = DH + kTile * LDH;    // [kTile][LDH]
    float* DZ = A1 + kTile * LDH;    // [kTile][LDF]
    const Topo& tp = p.tp;
    Stage stg;
    stg.init(DZ + kTile * LDF, 0, tp.T, false, 1);
    auto tile_of = [&](int i) { return get_tile<SPLIT>(tp, i); };
    using AccW1 = OuterAccX<H, F, 8, F / 2, 0, kThreads / 2>;              // dW1_e[j][k] = sum dh_j x_k
    using AccW2 = OuterAccX<F, H, 2, 2 * F, kThreads / 2, kThreads / 2>;   // dW2[j][k]   = sum dz_j a1_k
    constexpr int kAcc = AccW1::kAcc > AccW2::kAcc ? AccW1::kAcc : AccW2::kAcc;
    float acc[kAcc];
#pragma unroll
    for (int i = 0; i < kAcc; ++i) acc[i] = 0.f;
    AccW1 accw1;
    AccW2 accw2;
    accw1.init();
    accw2.init();
    constexpr int kDzParts = kThreads / F;   // db2 partial of thread (row part = tid / F < kDzParts, column tid % F)
    float dzs = 0.f;
    const int dz_col = threadIdx.x % F, dz_part = threadIdx.x / F;
    const float* esrc[1] = {p.x_e};
    const int total = tp.ntiles * tp.G;
    const int t_begin = chunk_begin(blockIdx.x, gridDim.x, total), t_end = chunk_begin(blockIdx.x + 1, gridDim.x, total);
    for (int tile = t_begin; tile < t_end; ++tile) {
        const Tile t = get_tile<SPLIT>(tp, tile);
        const int b = stg.step(tp, tile, t_end, 0, esrc, nullptr, nullptr, tile_of);
        if (threadIdx.x == 0 && tile + 1 < t_end && tp.layout == PFS_LAYOUT_DENSE) {   // next tile's slabs -> L2
            const Tile tn = get_tile<SPLIT>(tp, tile + 1);
            const size_t off = ((size_t)tn.g * tp.E + tn.q0) * F, bytes = (size_t)tn.ne * F * sizeof(float);
            bulk_prefetch_l2(p.x_e + off, bytes);
            bulk_prefetch_l2(p.xe2 + off, bytes);
            bulk_prefetch_l2(p.gout + off, bytes);
        }
        __syncthreads();
        const float* XE = stg.edge(b, 0);
        if (threadIdx.x < t.ne) {
            const EdgeRef er = get_edge(tp, t, threadIdx.x);
            const size_t row = ((size_t)t.g * tp.E + er.e) * F;
            float x[F], dz[F], dx[F];
            lds_row<F>(XE + threadIdx.x * F, x);
            {
                float gr[F], xo[F];
                load_row<F>(p.gout + row, gr);
                load_row<F>(p.xe2 + row, xo);
                const float* c = p.coef + (size_t)t.g * 6 * F;
#pragma unroll
                for (int j = 0; j < F; ++j) {
                    const float xh = (xo[j] - __ldg(c + 4 * F + j)) * __ldg(c + 3 * F + j);
                    dz[j] = __ldg(c + j) * (gr[j] - __ldg(c + F + j) - xh * __ldg(c + 2 * F + j));
                }
            }
            store_row_smem<F>(DZ + threadIdx.x * LDF, dz);
#pragma unroll
            for (int k = 0; k < F; ++k) dx[k] = 0.f;
            const float* ps = p.Ps + ((size_t)t.g * tp.S + er.src) * H;
            const float* pt = p.Pt + ((size_t)t.g * tp.T + er.tgt) * H;
            float* dho = p.dh_rows ? p.dh_rows + ((size_t)t.g * tp.E + t.q0 + threadIdx.x) * H : nullptr;
            edge_bwd_half<F, 0>(p, ps, pt, x, dz, dx, A1 + threadIdx.x * LDH, DH + threadIdx.x * LDH, dho);
            edge_bwd_half<F, 1>(p, ps, pt, x, dz, dx, A1 + threadIdx.x * LDH, DH + threadIdx.x * LDH, dho);
            store_row<F>(p.g_x_e + row, dx);
        }
        __syncthreads();
        // The two halves of the CTA run the FFMA2-bound outer products and the latency-bound segment sums in OPPOSITE
        // order, so every scheduler always holds a warp of each kind (warp w and warp w + 4 share a scheduler).
        if (threadIdx.x < kThreads / 2) {
            accw1.template accumulate<4, 1>(acc, DH, LDH, XE, F, t.ne);       // DH rows, j0: 16-byte aligned; x_e rows: 40 B
            tile_fibre_sums<H, LDH, 0, kThreads / 2, SPLIT>(tp, t, DH, fibre_sum_row<SPLIT>(tp, t, p.dPs, p.dPs_split, H));
        } else {
            if (p.class_part) tile_class_sums<H, LDH, kThreads / 2, kThreads / 2>(tp, t, DH, p.class_part + (size_t)tile * tp.T * H);
            accw2.template accumulate<2, 4>(acc, DZ, LDF, A1, LDH, t.ne);      // dz pairs: 8 bytes; a1 rows, k0: 16 bytes
        }
        if (dz_part < kDzParts)
            for (int r = dz_part; r < t.ne; r += kDzParts) dzs += DZ[r * LDF + dz_col];
        __syncthreads();
    }
    float* out = p.wpartial + (size_t)blockIdx.x * p.pstride;
    accw1.flush(acc, DH, out, F, 0);
    accw2.flush(acc, DH, out + H * F, H, 0);
    {   // db2 = sum dz: the row parts of each column, fixed order
        float* red = DH;
        if (dz_part < kDzParts) red[threadIdx.x] = dzs;
        __syncthreads();
        if (threadIdx.x < F) {
            float s = 0.f;
#pragma unroll
            for (int q = 0; q < kDzParts; ++q) s += red[q * F + threadIdx.x];
            out[2 * H * F + threadIdx.x] = s;
        }
    }
}

}  // namespace pfs
