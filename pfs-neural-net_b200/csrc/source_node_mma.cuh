// source_node_mma.cuh -- SModel node MLP, first layer on the 5th-generation tensor cores.
//
// The fibre MLP (reference src/gnn.py:153: node_mlp_2 = MLP(10F, 10F, F)) is the one contraction of
// the layer that is a real dense GEMM even at Fdim 10: [fibres x 9F] . [9F x 10F] over hundreds of
// thousands of fibres (the u columns are folded into the bias).  It runs as tcgen05.mma
// kind::tf32 with the 3xTF32 split (a = a_hi + a_lo, b = b_hi + b_lo; a.b ~ a_hi b_hi + a_lo b_hi
// + a_hi b_lo, error ~2^-21) so the fp32 parity tolerance holds:
//   * a CTA owns 128-fibre tiles (UMMA M = 128, one fibre per TMEM lane);
//   * operands live in shared memory in the canonical K-major no-swizzle core-matrix layout
//     (8 rows x 16 bytes per core matrix), written by the threads themselves (the A operand is
//     computed on the fly from the raw moments, so there is nothing for TMA to fetch);
//   * one elected thread issues the K/8 x 3 MMAs into a [128 x N] fp32 accumulator in TMEM and
//     commits to an mbarrier; warps 0-3 read their 32 lanes back with tcgen05.ld and run the
//     epilogue (bias, LeakyReLU, hidden store, second layer, BatchNorm tile statistics).
#pragma once
#include <cfloat>
#include "source_model.cuh"
#include "tc_ptx.cuh"

namespace pfs {

constexpr int kNodeThreadsC = 320;   // 10 warps
constexpr int kNodeRowsC = 128;      // fibres per node tile of the forward

// Constant-bank layout of the node kernels (floats; common.cuh: c_w).  The node-MLP constants sit ABOVE the
// message-MLP constants (MsgEdgeConst, at most 2 * 16 * 32 + 2 * 32 * 32 + 32 floats at Fdim 16) so that one upload
// per module call serves the edge kernel and the node kernel.  W3 itself goes to shared memory as the MMA operand.
template <int F>
struct SourceNodeConst {
    static constexpr int K9 = 9 * F, J = 10 * F;
    static constexpr int kBase = 4096;
    // forward: W4 input-major [J][F] (y_f += W4[f][j] a_j), b4 [F]
    static constexpr int kW4t = kBase, kB4 = kBase + J * F, kFwdMmaFloats = kBase + J * F + F;
    // backward: W4 as stored [F][J] (dh3_j += W4[f][j] dy_f)
    static constexpr int kW4o = kBase, kBwdMmaFloats = kBase + F * J;
    // The tensor-core node kernels serve the widths at which the whole node MLP, W3 [J][9F] included, fits the bank
    // above kBase: Fdim 4, 8 and 10.  Fdim 16 runs the shared-memory kernels of source_model.cuh.  This predicate also
    // picks the node tile size and the workspace carve (api.cu: node_tile_rows).
    static constexpr bool fits = kBase + J * F + F + K9 * J <= kConstFloats;
};

__device__ __forceinline__ int warp_index_uniform() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

template <int F>
struct SourceNodeMma {
    static constexpr int K9 = 9 * F, J = 10 * F;
    static constexpr int KP = (K9 + 7) / 8 * 8;          // K padded to the MMA K (8 tf32)
    static constexpr int NP = (J + 15) / 16 * 16;        // N padded (M = 128 needs N % 16 == 0)
    static constexpr int KC = KP / 4;                    // 16-byte K chunks
    static constexpr int LBO_A = 16 * 128;               // 128 rows = 16 core matrices of 128 B per K chunk
    static constexpr int LBO_B = (NP / 8) * 128;
    static constexpr int A_FLOATS = KC * LBO_A / 4;      // one of (hi, lo)
    static constexpr int B_FLOATS = KC * LBO_B / 4;
    static constexpr int TMEM_COLS = NP <= 32 ? 32 : NP <= 64 ? 64 : NP <= 128 ? 128 : 256;
    static constexpr int LDA = J + 1;
    // shared memory (floats): A hi/lo, B hi/lo, bias [J], YS [128][F], A3 [128][LDA] aliases the A operand
    static constexpr int kRed = (J > 17 * F ? J : 17 * F);   // bias vector, reused by the statistics reduction
    static constexpr int kFloats = 2 * A_FLOATS + 2 * B_FLOATS + kRed + 2 * 128 * F + J * F + 16;
    static constexpr size_t bytes = sizeof(float) * kFloats;
    static constexpr bool fits = bytes <= 200 * 1024 && 2 * A_FLOATS >= 128 * LDA && NP <= 256 &&
                                 SourceNodeConst<F>::fits;
};

// epilogue of columns [C0, C1) of the first-layer accumulator of one fibre (TMEM lane): bias, LeakyReLU, hidden
// activation into the staging row, and this column range's share of the second layer y += a_j * W4[:, j]
template <int F, int C0, int C1>
__device__ __forceinline__ void node_fwd_epilogue_cols(uint32_t taddr, const float* b3e, float* a3row, float (&y)[F]) {
    using CW = SourceNodeConst<F>;
    constexpr int J = 10 * F;
#pragma unroll
    for (int c0 = C0; c0 < C1; c0 += 16) {
        if (c0 >= J) break;
        float v[16];
        tmem_ld16(taddr + c0, v);
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int j = c0 + q;
            if (j < J) {
                const float a = lrelu(v[q] + b3e[j]);
                a3row[j] = a;
                const float2 aa = make_float2(a, a);
#pragma unroll
                for (int f = 0; f < F; f += 2) {
                    const float2 e = __ffma2_rn(make_float2(c_w[CW::kW4t + j * F + f], c_w[CW::kW4t + j * F + f + 1]), aa,
                                                make_float2(y[f], y[f + 1]));
                    y[f] = e.x; y[f + 1] = e.y;
                }
            }
        }
    }
}

template <int F>
__global__ void __launch_bounds__(kNodeThreadsC) k_source_node_fwd_mma(const SourceNodeFwdParams p) {
    using MM = SourceNodeMma<F>;
    using CW = SourceNodeConst<F>;
    constexpr int K9 = MM::K9, J = MM::J, KP = MM::KP, NP = MM::NP, KC = MM::KC, LDA = MM::LDA, M2 = 2 * F;
    extern __shared__ __align__(1024) float smm[];
    float* sm = smm;
    float* Ahi = sm;
    float* Alo = Ahi + MM::A_FLOATS;
    float* Bhi = Alo + MM::A_FLOATS;
    float* Blo = Bhi + MM::B_FLOATS;
    float* b3e = Blo + MM::B_FLOATS;        // [J]
    float* YS = b3e + MM::kRed;             // [2][128][F] second-layer partials of the two column halves
    float* W4s = YS + 2 * 128 * F;          // [J][F] input-major second-layer weights
    uint64_t* bar = reinterpret_cast<uint64_t*>(W4s + J * F);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
    float* A3 = sm;                         // [128][LDA], aliases the A operand once the MMAs are done
    const int warp = warp_index_uniform(), lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        fence_barrier_init();
    }
    __syncwarp();
    if (warp == 0) tmem_alloc(tmem_slot, MM::TMEM_COLS);
    // B operand: W3[j][k], j < 10F (N), k < 9F (K), split hi/lo, zero padded, core-matrix layout
    for (int i = threadIdx.x; i < NP * KC; i += blockDim.x) {
        const int j = i / KC, kc = i - j * KC;
        float hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int k = 4 * kc + q;
            const float w = (j < J && k < K9) ? __ldg(p.w3 + (size_t)j * J + k) : 0.f;
            hi[q] = to_tf32(w);
            lo[q] = to_tf32(w - hi[q]);
        }
        const int o = (kc * MM::LBO_B + (j >> 3) * 128 + (j & 7) * 16) >> 2;
        *reinterpret_cast<float4*>(Bhi + o) = make_float4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<float4*>(Blo + o) = make_float4(lo[0], lo[1], lo[2], lo[3]);
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t idesc = umma_idesc_tf32(128, NP);
    uint32_t parity = 0;

    const int total = p.ntiles * p.G;
    // Tile-invariant work items of the operand build.  Moment items (fibre r, message feature j) and x_s items
    // (r, c) are numbered with the feature's low two bits fastest, then the fibre: a warp's 4-byte operand stores
    // fill whole 16-byte core-matrix rows (no bank conflicts) and its global reads are 16 contiguous bytes per
    // fibre.  Their inputs are fetched ONE TILE AHEAD into registers: with one CTA of 10 warps per SM nothing
    // else hides the DRAM latency in front of the MMAs.
    constexpr int NI = (kNodeRowsC * M2 + kNodeThreadsC - 1) / kNodeThreadsC;
    constexpr int XG = (F + 3) / 4;                                          // 4-column groups of x_s
    constexpr int NX = (kNodeRowsC * 4 * XG + kNodeThreadsC - 1) / kNodeThreadsC;
    auto item_r = [](int i) { return (i >> 2) & (kNodeRowsC - 1); };
    auto item_c = [](int i) { return ((i >> 9) << 2) | (i & 3); };           // feature index (j or c)
    float pf_mo[NI][4], pf_xs[NX];
#pragma unroll
    for (int n = 0; n < NI; ++n)
#pragma unroll
        for (int q = 0; q < 4; ++q) pf_mo[n][q] = 0.f;
#pragma unroll
    for (int n = 0; n < NX; ++n) pf_xs[n] = 0.f;
    auto prefetch = [&](int tile2) {
        if (tile2 >= total) return;
        const int g2 = tile2 / p.ntiles, f2 = (tile2 - g2 * p.ntiles) * kNodeRowsC;
        const int rows2 = min(kNodeRowsC, p.S - f2);
        const size_t row2 = (size_t)g2 * p.S + f2;
#pragma unroll
        for (int n = 0; n < NI; ++n) {
            const int i = threadIdx.x + n * kNodeThreadsC, r = item_r(i), j = item_c(i);
            if (i < kNodeRowsC * M2 && r < rows2) {
                const float* mo = p.moments + (row2 + r) * 5 * M2 + j;
                pf_mo[n][0] = __ldg(mo); pf_mo[n][1] = __ldg(mo + M2); pf_mo[n][2] = __ldg(mo + 3 * M2); pf_mo[n][3] = __ldg(mo + 4 * M2);
            }
        }
#pragma unroll
        for (int n = 0; n < NX; ++n) {
            const int i = threadIdx.x + n * kNodeThreadsC, r = item_r(i), c = item_c(i);
            if (i < kNodeRowsC * 4 * XG && c < F && r < rows2) pf_xs[n] = __ldg(p.x_s + (row2 + r) * F + c);
        }
    };
    prefetch(blockIdx.x);
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int g = tile / p.ntiles, lt = tile - g * p.ntiles;
        const int f0 = lt * kNodeRowsC;
        const int rows = min(kNodeRowsC, p.S - f0);
        const size_t row0 = (size_t)g * p.S + f0;
        // ---- A operand: hcat = [x_s | mean | std | skew | kurt] per fibre, split hi/lo ----------------
        // element (r, k) -> byte (k / 4) * LBO_A + r * 16 + (k % 4) * 4
        auto put = [&](int r, int k, float v) {
            const float hi = to_tf32(v);
            const int o = ((k >> 2) * MM::LBO_A + r * 16 + (k & 3) * 4) >> 2;
            Ahi[o] = hi;
            Alo[o] = to_tf32(v - hi);
        };
        for (int i = threadIdx.x; i < 128 * (KP - K9); i += blockDim.x)            // zero padding of K (A3 overwrote it)
            put(i & 127, K9 + (i >> 7), 0.f);
#pragma unroll
        for (int n = 0; n < NX; ++n) {
            const int i = threadIdx.x + n * kNodeThreadsC, r = item_r(i), c = item_c(i);
            if (i < kNodeRowsC * 4 * XG && c < F) put(r, c, r < rows ? pf_xs[n] : 0.f);
        }
#pragma unroll
        for (int n = 0; n < NI; ++n) {
            const int i = threadIdx.x + n * kNodeThreadsC, r = item_r(i), j = item_c(i);
            if (i >= kNodeRowsC * M2) continue;
            float mean_o = 0.f, std_o = 0.f, skew_o = 0.f, kurt_o = 0.f;
            if (r < rows) {
                const float mean = pf_mo[n][0], ex2 = pf_mo[n][1], c3 = pf_mo[n][2], c4 = pf_mo[n][3];
                const float vr = ex2 - mean * mean;
                const float var = vr > 0.f ? vr : kSlopeVar * vr;
                const float i1 = rsqrtf(var + kStdEps);          // 1 / std (NaN for var + eps < 0, like the sqrt)
                const float i2 = i1 * i1;
                const float skew = c3 * (i2 * i1), kurt = c4 * (i2 * i2);
                mean_o = mean; std_o = (var + kStdEps) * i1; skew_o = skew; kurt_o = kurt;
                // |x| <= FLT_MAX is false for NaN and +-inf: one compare per statistic on the common path
                if (!(fabsf(mean) <= FLT_MAX && fabsf(var) <= FLT_MAX && fabsf(skew) <= FLT_MAX && fabsf(kurt) <= FLT_MAX)) {
                    mean_o = nan_to_num(mean);                   // rare: torch.nan_to_num semantics
                    skew_o = nan_to_num(skew);
                    kurt_o = nan_to_num(kurt);
                    if (!(fabsf(var) <= FLT_MAX)) std_o = sqrtf(nan_to_num(var) + kStdEps);
                }
            }
            put(r, F + j, mean_o);
            put(r, F + M2 + j, std_o);
            put(r, F + 2 * M2 + j, skew_o);
            put(r, F + 3 * M2 + j, kurt_o);
        }
        prefetch(tile + gridDim.x);       // next tile's inputs: in flight under the MMAs and the epilogue
        for (int j = threadIdx.x; j < J; j += blockDim.x) {
            float s = __ldg(p.b3 + j);
            for (int k = 0; k < F; ++k) s = fmaf(__ldg(p.w3 + (size_t)j * J + K9 + k), __ldg(p.u + (size_t)g * F + k), s);
            b3e[j] = s;
        }
        fence_proxy_async();      // generic-proxy writes of the operands -> visible to the tensor core (async proxy)
        tc_fence_before();
        __syncthreads();
        // ---- MMAs: one thread issues KP/8 k-steps x 3 products --------------------------------------
        if (threadIdx.x == 0) {
            tc_fence_after();
            const uint32_t a_hi = smem_u32(Ahi), a_lo = smem_u32(Alo), b_hi = smem_u32(Bhi), b_lo = smem_u32(Blo);
#pragma unroll 1
            for (int ks = 0; ks < KP / 8; ++ks) {
                const uint32_t ao = ks * 2 * MM::LBO_A, bo = ks * 2 * MM::LBO_B;
                const uint64_t dah = umma_desc(a_hi + ao, MM::LBO_A), dal = umma_desc(a_lo + ao, MM::LBO_A);
                const uint64_t dbh = umma_desc(b_hi + bo, MM::LBO_B), dbl = umma_desc(b_lo + bo, MM::LBO_B);
                umma_tf32(tmem, dal, dbh, idesc, ks > 0 ? 1u : 0u);   // small terms first
                umma_tf32(tmem, dah, dbl, idesc, 1u);
                umma_tf32(tmem, dah, dbh, idesc, 1u);
            }
            umma_commit(bar);     // implies tcgen05.fence::before_thread_sync
        }
        // ---- epilogue: warps 0-3 own TMEM lanes 32w .. 32w+31 = fibres of the tile ------------------
        mbar_wait(bar, parity);
        parity ^= 1;
        tc_fence_after();
        if (warp < 8) {
            // warp w reads TMEM lanes 32 * (w % 4) .. + 31 (hardware rule) and the column half w / 4
            const int quarter = warp & 3, half = warp >> 2;
            const int r = quarter * 32 + lane;
            constexpr int NH = (NP / 16 + 1) / 2 * 16;       // columns of the first half (multiple of 16)
            float y[F];
#pragma unroll
            for (int f = 0; f < F; ++f) y[f] = half ? 0.f : c_w[CW::kB4 + f];
            // one fully unrolled copy of the column loop per half: the column index is then a compile-time
            // constant and the second-layer weights are constant-bank immediates of the FFMA2s (no shared-memory
            // weight reads)
            if (half == 0) node_fwd_epilogue_cols<F, 0, NH>(tmem + ((uint32_t)(quarter * 32) << 16), b3e, A3 + r * LDA, y);
            else node_fwd_epilogue_cols<F, NH, NP>(tmem + ((uint32_t)(quarter * 32) << 16), b3e, A3 + r * LDA, y);
#pragma unroll
            for (int f = 0; f < F; ++f) YS[(half * 128 + r) * F + f] = y[f];
        }
        tc_fence_before();
        __syncthreads();
        for (int i = threadIdx.x; i < rows * F; i += blockDim.x) {      // y = both column halves
            const float v = YS[i] + YS[128 * F + i];
            YS[i] = v;
            p.y_pre[row0 * F + i] = v;
        }
        tc_fence_before();
        __syncthreads();
        // hidden activations to global (coalesced), BatchNorm tile statistics
        static_assert(J % 4 == 0, "16-byte stores of the hidden rows");
        for (int i = threadIdx.x; i < rows * (J / 4); i += blockDim.x) {
            const int r = i / (J / 4), c = (i - r * (J / 4)) * 4;
            const float* a = A3 + r * LDA + c;
            *reinterpret_cast<float4*>(p.hidden + (row0 + r) * J + c) = make_float4(a[0], a[1], a[2], a[3]);
        }
        __syncthreads();
        if (p.bn_partial) {
            // two-pass tile statistics, kParts row slices per feature reduced in a fixed order
            constexpr int kParts = 16;
            float* red = b3e;     // the bias vector is dead: kParts * F + F floats of scratch
            const int f = threadIdx.x % F, part = threadIdx.x / F;
            float s = 0.f;
            if (part < kParts)
                for (int r = part; r < rows; r += kParts) s += YS[r * F + f];
            if (part < kParts) red[part * F + f] = s;
            __syncthreads();
            if (threadIdx.x < F) {
                float t = 0.f;
                for (int q = 0; q < kParts; ++q) t += red[q * F + threadIdx.x];
                red[kParts * F + threadIdx.x] = t / (float)rows;
            }
            __syncthreads();
            const float mean = red[kParts * F + f];
            float m2 = 0.f;
            if (part < kParts)
                for (int r = part; r < rows; r += kParts) {
                    const float d = YS[r * F + f] - mean;
                    m2 = fmaf(d, d, m2);
                }
            __syncthreads();
            if (part < kParts) red[part * F + f] = m2;
            __syncthreads();
            if (threadIdx.x < F) {
                float t = 0.f;
                for (int q = 0; q < kParts; ++q) t += red[q * F + threadIdx.x];
                float* o = p.bn_partial + (size_t)tile * bn_partial_stride(F);
                o[threadIdx.x] = red[kParts * F + threadIdx.x];
                o[F + threadIdx.x] = t;
                if (threadIdx.x == 0) o[2 * F] = (float)rows;
            }
        }
        __syncthreads();
        tc_fence_after();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, MM::TMEM_COLS);
}

}  // namespace pfs
