// source_node_bwd_mma.cuh -- backward of the SModel node MLP on the 5th-generation tensor cores.
//
// Per fibre the backward of node_mlp_2 = MLP(10F, 10F, F) (reference src/gnn.py:153) is two real
// dense contractions, both 9F x 10F wide:
//   dhcat [rows, 9F]  = dh3 [rows, 10F] . W3[:, :9F]           (input gradient, contraction over 10F)
//   dW3   [10F, 9F]  += dh3^T [10F, rows] . hcat [rows, 9F]    (weight gradient, contraction over rows)
// 18 k of the 20 k MACs per fibre.  Both run as tcgen05.mma kind::tf32 with the 3xTF32 split
// (x = hi + lo; a.b ~ a_lo b_hi + a_hi b_lo + a_hi b_hi), like the forward (source_node_mma.cuh).
//
//   * a CTA owns 48-fibre tiles.  Every operand is K-major in the no-swizzle core-matrix layout of
//     tc_ptx.cuh, split hi/lo, written by the threads that compute it.  dh3 is contracted over the
//     hidden units in the first product and over the fibres in the second, so it is written in both
//     arrangements (measured on B200: kind::tf32 reads an MN-major no-swizzle operand as zeros -- for
//     tf32 the only transposing layout is SWIZZLE_128B_BASE32B, which no K-major product can share);
//     that second copy is what limits the tile to 48 fibres (220 KB of shared memory);
//   * GEMM1 is computed transposed, D1[k, r] = sum_j W3[j, k] dh3[r, j] (UMMA M = 128 holds the 9F
//     hcat features, N = 48 fibres), because a 48-row accumulator would not fill the TMEM lanes;
//   * GEMM2 D2[j, k] accumulates in TMEM over ALL tiles of the CTA and is read back once at the end:
//     the 90 x 100 outer-product accumulators leave the register file entirely;
//   * the small pieces stay on the FMA pipe: dh3 = (dy . W4) * lrelu'(h3) (weights from the constant
//     bank), dW4 / db4 (outer-product accumulators on five warps, running under the MMAs), the
//     BatchNorm backward of the upstream gradient and the moment-polynomial coefficients.
#pragma once
#include <cfloat>
#include "source_node_mma.cuh"
#include "tc_ptx.cuh"

namespace pfs {

constexpr int kNodeRowsB = 48;   // fibres per tile of the tensor-core backward

template <int F>
struct SourceNodeBwdMma {
    static constexpr int K9 = 9 * F, J = 10 * F, R = kNodeRowsB;
    static constexpr int JP = (J + 7) / 8 * 8;            // K of GEMM1 (multiple of the tf32 MMA K)
    static constexpr int KN = (K9 + 15) / 16 * 16;        // N of GEMM2 (M = 128 needs N % 16 == 0)
    static constexpr int RW = (K9 + 7) / 8 * 8;           // rows of the W3 operand that exist in memory
    // chunk (16-byte K group) strides in bytes; the +16 keeps the threads' 4-byte stores and the column
    // sums free of bank conflicts
    static constexpr int CS_W = RW * 16;                  // W3   : rows k, chunks over j   (A of GEMM1)
    static constexpr int CS_D1 = R * 16 + 16;             // dh3  : rows r, chunks over j   (B of GEMM1)
    static constexpr int CS_D2 = JP * 16 + 16;            // dh3  : rows j, chunks over r   (A of GEMM2)
    static constexpr int CS_H = KN * 16 + 16;             // hcat : rows k, chunks over r   (B of GEMM2)
    static constexpr int W_FLOATS = (JP / 4) * CS_W / 4;  // one of (hi, lo)
    static constexpr int D1_FLOATS = (JP / 4) * CS_D1 / 4;
    static constexpr int D2_FLOATS = (R / 4) * CS_D2 / 4;
    static constexpr int H_FLOATS = (R / 4) * CS_H / 4;
    static constexpr int LDA = J, LDY = F + 1, LDC = K9 + 1;
    static constexpr int A3_FLOATS = (R * LDA > R * LDC ? R * LDA : R * LDC) + 8;   // hidden rows, later dhcat
    static constexpr int TMEM_COLS = 256;                 // D2 at column 0 (KN <= 128), D1 at column 128 (R)
    // dW4 accumulators on warps 5..9
    using AccW4 = OuterAcc<F, J, 2, 2 * F, 160, 160>;
    // order: W3, dh3 (GEMM1 form), dh3 (GEMM2 form), hcat, then the plain fp32 tiles.  The M = 128 operands
    // (W3: RW rows, dh3 GEMM2 form: JP rows per chunk) are read 128 rows deep, i.e. a little past their last
    // chunk into the next buffer; those accumulator lanes are never read back.
    static constexpr int kFloats = 2 * W_FLOATS + 2 * D1_FLOATS + 2 * D2_FLOATS + 2 * H_FLOATS + A3_FLOATS + R * LDY + 16;
    static constexpr size_t bytes = sizeof(float) * kFloats;
    static constexpr bool fits = bytes <= 227 * 1024 && K9 <= 128 && J <= 128 && KN <= 128 && R % 16 == 0 &&
                                 AccW4::kScratchFloats <= 2 * D1_FLOATS + 2 * D2_FLOATS && SourceNodeConst<F>::fits;
};

// dh3 accumulation of one warp-uniform chunk: d[c] += dy[f] * W4[f][CH * 2F + c], weights read as
// constant-bank operands of the FFMA2s (the offset is a compile-time constant per chunk)
template <int F, int CH>
__device__ __forceinline__ void dh3_chunk(const float* y, float (&d)[2 * F]) {
    using CW = SourceNodeConst<F>;
    constexpr int C = 2 * F, J = 10 * F, OFF = CW::kW4o + CH * C;
#pragma unroll
    for (int f = 0; f < F; ++f) {
        const float2 v = make_float2(y[f], y[f]);
#pragma unroll
        for (int c = 0; c < C; c += 2) {
            const float2 w = make_float2(c_w[OFF + f * J + c], c_w[OFF + f * J + c + 1]);
            const float2 e = __ffma2_rn(w, v, make_float2(d[c], d[c + 1]));
            d[c] = e.x; d[c + 1] = e.y;
        }
    }
}

template <int F>
__global__ void __launch_bounds__(kNodeThreadsC) k_source_node_bwd_mma(const SourceNodeBwdParams p) {
    using MM = SourceNodeBwdMma<F>;
    using CW = SourceNodeConst<F>;
    constexpr int K9 = MM::K9, J = MM::J, R = MM::R, JP = MM::JP, KN = MM::KN, RW = MM::RW, C = 2 * F, M = 2 * F;
    constexpr int LDA = MM::LDA, LDY = MM::LDY, LDC = MM::LDC;
    extern __shared__ __align__(1024) float smm[];
    float* Whi = smm;
    float* Wlo = Whi + MM::W_FLOATS;
    float* Dhi = Wlo + MM::W_FLOATS;         // dh3, rows = fibres   (GEMM1)
    float* Dlo = Dhi + MM::D1_FLOATS;
    float* Ehi = Dlo + MM::D1_FLOATS;        // dh3, rows = hidden units (GEMM2)
    float* Elo = Ehi + MM::D2_FLOATS;
    float* Hhi = Elo + MM::D2_FLOATS;
    float* Hlo = Hhi + MM::H_FLOATS;
    float* A3 = Hlo + MM::H_FLOATS;          // [R][LDA] hidden activations; after the MMAs [R][LDC] dhcat
    float* DY = A3 + MM::A3_FLOATS;          // [R][LDY]
    uint64_t* bar = reinterpret_cast<uint64_t*>(DY + R * LDY + ((R * LDY) & 1));
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
    const int warp = warp_index_uniform(), lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        fence_barrier_init();
    }
    __syncwarp();
    if (warp == 0) tmem_alloc(tmem_slot, MM::TMEM_COLS);
    // W3 operand: element (row k, column j) = W3[j][k], split hi/lo, zero padded
    for (int i = threadIdx.x; i < RW * (JP / 4); i += blockDim.x) {
        const int jc = i / RW, k = i - jc * RW;
        float hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = 4 * jc + q;
            const float w = (j < J && k < K9) ? __ldg(p.w3 + (size_t)j * J + k) : 0.f;
            hi[q] = to_tf32(w);
            lo[q] = to_tf32(w - hi[q]);
        }
        const int o = (jc * MM::CS_W + k * 16) >> 2;
        *reinterpret_cast<float4*>(Whi + o) = make_float4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<float4*>(Wlo + o) = make_float4(lo[0], lo[1], lo[2], lo[3]);
    }
    // padding of the per-tile operands (columns j >= J of dh3, k >= K9 of hcat) is written once
    for (int i = threadIdx.x; i < 2 * MM::D1_FLOATS + 2 * MM::D2_FLOATS + 2 * MM::H_FLOATS; i += blockDim.x) Dhi[i] = 0.f;
    typename MM::AccW4 accw4;
    accw4.init();
    float db4 = 0.f;        // threads 32 .. 32 + F
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tmem_d2 = tmem, tmem_d1 = tmem + 128;
    constexpr uint32_t idesc1 = umma_idesc_tf32_mn(128, R, 0, 0);
    constexpr uint32_t idesc2 = umma_idesc_tf32_mn(128, KN, 0, 0);
    uint32_t parity = 0;
    bool first = true;

    // dh3 mapping: warp = (row set, chunk of 2F hidden units), lane = fibre; rows >= R of the second row set idle
    const int chunk = warp % 5, r = (warp / 5) * 32 + lane;
    const int off = chunk * C;
    // Tile-invariant work items of the scalar phases.  Moment items (fibre rr, message feature j) and x_s items
    // (rr, c) are numbered so that consecutive lanes take rr % 4 fastest, then the feature: the 4-byte operand
    // stores of a warp then fill whole 16-byte core-matrix rows (no bank conflicts) and the global reads touch
    // 4 rows x 32 contiguous bytes.  What the forward pass of an item computes (1 / std, the nan_to_num masks)
    // stays in registers for its backward half after the MMAs.
    constexpr int NI = (R * M + kNodeThreadsC - 1) / kNodeThreadsC;      // moment items per thread
    constexpr int NX = (R * F + kNodeThreadsC - 1) / kNodeThreadsC;      // x_s / dy items per thread
    // every offset an item needs (operand slot, global rows relative to the tile, dhcat slot) is computed once here
    auto hslot = [](int rr, int k) { return ((rr >> 2) * MM::CS_H + k * 16 + (rr & 3) * 4) >> 2; };
    int it_rr[NI], it_po[NI], it_go[NI], it_co[NI], it_do[NI];
#pragma unroll
    for (int n = 0; n < NI; ++n) {
        const int i = threadIdx.x + n * kNodeThreadsC;
        const int q = i / (4 * M), rem = i - q * (4 * M);
        const int rr = i < R * M ? 4 * q + (rem & 3) : R, j = rem >> 2;   // R = no item
        it_rr[n] = rr;
        it_po[n] = hslot(rr < R ? rr : 0, F + j);        // operand slot of the mean; std / skew / kurt follow at + s * 4M floats
        it_go[n] = rr * 5 * M + j;                       // moments, relative to the tile's first row
        it_co[n] = rr * 4 * M + j;                       // coefA, relative to the tile's first row
        it_do[n] = rr * LDC + F + j;                     // dhcat staging
    }
    int ix_rr[NX], ix_po[NX], ix_go[NX], iy_rr[NX], iy_f[NX], iy_so[NX], iy_go[NX];
#pragma unroll
    for (int n = 0; n < NX; ++n) {
        const int i = threadIdx.x + n * kNodeThreadsC;
        const int q = i / (4 * F), rem = i - q * (4 * F);
        const int rr = i < R * F ? 4 * q + (rem & 3) : R, c = rem >> 2;
        ix_rr[n] = rr;
        ix_po[n] = hslot(rr < R ? rr : 0, c);
        ix_go[n] = rr * F + c;
        iy_rr[n] = i < R * F ? i / F : R;
        iy_f[n] = i % F;
        iy_so[n] = iy_rr[n] * LDY + iy_f[n];
        iy_go[n] = iy_rr[n] * F + iy_f[n];
    }
    auto put = [&](int o, float v) {
        const float hi = to_tf32(v);
        Hhi[o] = hi;
        Hlo[o] = to_tf32(v - hi);
    };
    const int total = p.ntiles * p.G;
    // Inputs of the scalar phase are fetched one tile ahead into registers: with one CTA of 10 warps per SM
    // nothing else hides their DRAM latency.
    float pf_mo[NI][5], pf_xs[NX], pf_g[NX], pf_y[NX];
    auto prefetch = [&](int tile2) {
        if (tile2 >= total) return;
        const int g2 = tile2 / p.ntiles, f2 = (tile2 - g2 * p.ntiles) * R;
        const int rows2 = min(R, p.S - f2);
        const size_t row2 = (size_t)g2 * p.S + f2;
        const float* mo2 = p.moments + row2 * 5 * M;
        const float *xs2 = p.x_s + row2 * F, *go2 = p.gout + row2 * F, *yp2 = p.y_pre + row2 * F;
#pragma unroll
        for (int n = 0; n < NI; ++n) {
            if (it_rr[n] < rows2) {
#pragma unroll
                for (int q = 0; q < 5; ++q) pf_mo[n][q] = __ldg(mo2 + it_go[n] + q * M);
            }
        }
#pragma unroll
        for (int n = 0; n < NX; ++n) {
            if (ix_rr[n] < rows2) pf_xs[n] = __ldg(xs2 + ix_go[n]);
            if (iy_rr[n] < rows2) {
                pf_g[n] = __ldg(go2 + iy_go[n]);
                pf_y[n] = p.mode == 1 ? __ldg(yp2 + iy_go[n]) : 0.f;
            }
        }
    };
#pragma unroll
    for (int n = 0; n < NI; ++n)
#pragma unroll
        for (int q = 0; q < 5; ++q) pf_mo[n][q] = 0.f;
#pragma unroll
    for (int n = 0; n < NX; ++n) pf_xs[n] = pf_g[n] = pf_y[n] = 0.f;
    prefetch(blockIdx.x);
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int g = tile / p.ntiles, lt = tile - g * p.ntiles;
        const int f0 = lt * R;
        const int rows = min(R, p.S - f0);
        const size_t row0 = (size_t)g * p.S + f0;
        // hidden activations of (r, chunk): in flight while the operands are built
        float a[C];
        load_row<C>(p.hidden + (row0 + (r < rows ? r : 0)) * J + off, a);   // rows beyond the tile: any valid row
        // ---- hcat = [x_s | mean | std | skew | kurt], split hi/lo (rows beyond the tile are zero) ----
        float m_mean[NI], m_vr[NI], m_c2[NI], m_c3[NI], m_c4[NI], m_i1[NI], m_is1[NI];
        unsigned m_fin[NI];      // bit 0..3: mean, var, skew, kurt were finite (nan_to_num passes their gradient)
#pragma unroll
        for (int n = 0; n < NI; ++n) {
            const int rr = it_rr[n];
            float mean_o = 0.f, std_o = 0.f, skew_o = 0.f, kurt_o = 0.f;
            m_fin[n] = 0u;
            m_mean[n] = m_vr[n] = m_c2[n] = m_c3[n] = m_c4[n] = m_i1[n] = m_is1[n] = 0.f;
            if (rr < rows) {
                const float mean = pf_mo[n][0], ex2 = pf_mo[n][1], c2 = pf_mo[n][2], c3 = pf_mo[n][3], c4 = pf_mo[n][4];
                const float vr = ex2 - mean * mean;
                const float var = vr > 0.f ? vr : kSlopeVar * vr;
                const float i1 = rsqrtf(var + kStdEps);          // 1 / std (NaN for var + eps < 0, like the sqrt)
                const float i2 = i1 * i1;
                const float skew = c3 * (i2 * i1), kurt = c4 * (i2 * i2);
                // |x| <= FLT_MAX is false for NaN and +-inf: one compare per statistic on the common path
                const bool fm = fabsf(mean) <= FLT_MAX, fv = fabsf(var) <= FLT_MAX;
                const bool fs = fabsf(skew) <= FLT_MAX, fk = fabsf(kurt) <= FLT_MAX;
                mean_o = mean; std_o = (var + kStdEps) * i1; skew_o = skew; kurt_o = kurt;
                float is1 = i1;
                if (!(fm && fv && fs && fk)) {                   // rare: torch.nan_to_num semantics
                    mean_o = nan_to_num(mean);
                    skew_o = nan_to_num(skew);
                    kurt_o = nan_to_num(kurt);
                    if (!fv) {
                        std_o = sqrtf(nan_to_num(var) + kStdEps);
                        is1 = 1.f / std_o;                       // 1 / std as recomputed after nan_to_num
                    }
                }
                m_fin[n] = (fm ? 1u : 0u) | (fv ? 2u : 0u) | (fs ? 4u : 0u) | (fk ? 8u : 0u);
                m_mean[n] = mean; m_vr[n] = vr; m_c2[n] = c2; m_c3[n] = c3; m_c4[n] = c4; m_i1[n] = i1;
                m_is1[n] = is1;
            }
            if (rr < R) {
                put(it_po[n], mean_o);
                put(it_po[n] + 4 * M, std_o);
                put(it_po[n] + 8 * M, skew_o);
                put(it_po[n] + 12 * M, kurt_o);
            }
        }
#pragma unroll
        for (int n = 0; n < NX; ++n) {
            const int rr = ix_rr[n];
            if (rr < R) put(ix_po[n], rr < rows ? pf_xs[n] : 0.f);
        }
        // ---- dy = BatchNorm backward of the upstream gradient ---------------------------------------
        {
            const float* sv = p.bn_save + (size_t)g * 4 * F;
            const float* st = p.bn_stat + (size_t)g * 2 * F;
            const float invS = 1.f / (float)p.S;
#pragma unroll
            for (int n = 0; n < NX; ++n) {
                const int rr = iy_rr[n], f = iy_f[n];
                if (rr >= R) continue;
                float dy = 0.f;
                if (rr < rows) {
                    const float gv = pf_g[n];
                    if (p.mode == 1) {
                        const float rstd = rsqrtf(sv[F + f] + p.eps);
                        const float xh = (pf_y[n] - sv[f]) * rstd;
                        dy = sv[2 * F + f] * (gv - st[f] * invS - xh * st[F + f] * invS);
                    } else if (p.mode == 2) {
                        dy = gv * sv[2 * F + f];
                    } else {
                        dy = gv;
                    }
                }
                DY[iy_so[n]] = dy;
            }
        }
        prefetch(tile + gridDim.x);      // next tile's scalar inputs: in flight under the rest of this tile
        __syncthreads();
        // ---- dh3 = (dy . W4) * lrelu'(h3): thread = (fibre, chunk of 2F hidden units) ---------------
        {
            float d[C];
#pragma unroll
            for (int c = 0; c < C; ++c) d[c] = 0.f;
            const float* y = DY + (r < R ? r : 0) * LDY;
            // the chunk is warp-uniform: one copy of the loop per chunk, weights as constant-bank immediates
            switch (chunk) {
                case 0: dh3_chunk<F, 0>(y, d); break;
                case 1: dh3_chunk<F, 1>(y, d); break;
                case 2: dh3_chunk<F, 2>(y, d); break;
                case 3: dh3_chunk<F, 3>(y, d); break;
                default: dh3_chunk<F, 4>(y, d); break;
            }
            const bool live = r < rows;
            if (r < R) {
#pragma unroll
                for (int q = 0; q < C / 4; ++q) {
                    float hi[4], lo[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int c = 4 * q + e;
                        const float v = live ? d[c] * (a[c] > 0.f ? 1.f : kSlope) : 0.f;
                        hi[e] = to_tf32(v);
                        lo[e] = to_tf32(v - hi[e]);
                        const int o2 = ((r >> 2) * MM::CS_D2 + (off + c) * 16 + (r & 3) * 4) >> 2;
                        Ehi[o2] = hi[e];
                        Elo[o2] = lo[e];
                    }
                    const int o = ((off / 4 + q) * MM::CS_D1 + r * 16) >> 2;
                    *reinterpret_cast<float4*>(Dhi + o) = make_float4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<float4*>(Dlo + o) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                    *reinterpret_cast<float4*>(A3 + r * LDA + off + 4 * q) =
                        live ? make_float4(a[4 * q], a[4 * q + 1], a[4 * q + 2], a[4 * q + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
        fence_proxy_async();      // operand writes (generic proxy) -> visible to the tensor core (async proxy)
        tc_fence_before();
        __syncthreads();
        // ---- MMAs (one thread); the other warps run the FMA-side reductions under them ----------------
        if (threadIdx.x == 0) {
            tc_fence_after();
            const uint32_t w_hi = smem_u32(Whi), w_lo = smem_u32(Wlo), d_hi = smem_u32(Dhi), d_lo = smem_u32(Dlo);
            const uint32_t e_hi = smem_u32(Ehi), e_lo = smem_u32(Elo), h_hi = smem_u32(Hhi), h_lo = smem_u32(Hlo);
            // GEMM1: D1[k, r] = sum_j W3c[k, j] dh3[r, j]   (K = j)
#pragma unroll 1
            for (int ks = 0; ks < JP / 8; ++ks) {
                const uint32_t ao = ks * 2 * MM::CS_W, bo = ks * 2 * MM::CS_D1;
                const uint64_t ah = umma_desc_ls(w_hi + ao, MM::CS_W, 128), al = umma_desc_ls(w_lo + ao, MM::CS_W, 128);
                const uint64_t bh = umma_desc_ls(d_hi + bo, MM::CS_D1, 128), bl = umma_desc_ls(d_lo + bo, MM::CS_D1, 128);
                umma_tf32(tmem_d1, al, bh, idesc1, ks > 0 ? 1u : 0u);   // small terms first
                umma_tf32(tmem_d1, ah, bl, idesc1, 1u);
                umma_tf32(tmem_d1, ah, bh, idesc1, 1u);
            }
            // GEMM2: D2[j, k] += sum_r dh3[r, j] hcat[r, k]   (K = r)
#pragma unroll 1
            for (int ks = 0; ks < R / 8; ++ks) {
                const uint32_t ao = ks * 2 * MM::CS_D2, bo = ks * 2 * MM::CS_H;
                const uint64_t ah = umma_desc_ls(e_hi + ao, MM::CS_D2, 128), al = umma_desc_ls(e_lo + ao, MM::CS_D2, 128);
                const uint64_t bh = umma_desc_ls(h_hi + bo, MM::CS_H, 128), bl = umma_desc_ls(h_lo + bo, MM::CS_H, 128);
                umma_tf32(tmem_d2, al, bh, idesc2, (first && ks == 0) ? 0u : 1u);
                umma_tf32(tmem_d2, ah, bl, idesc2, 1u);
                umma_tf32(tmem_d2, ah, bh, idesc2, 1u);
            }
            umma_commit(bar);
        }
        first = false;
        if (warp >= 5) {
            accw4.accumulate(DY, LDY, A3, LDA, rows);              // dW4[f][j] += dy[r][f] a3[r][j]
        } else if (warp >= 1) {
            const int j = threadIdx.x - 32;                        // column sums of dh3 (bias / u gradients)
            if (j < J) {
                const int o = ((j >> 2) * MM::CS_D1 + (j & 3) * 4) >> 2;
                float s = 0.f;
                for (int rr = 0; rr < rows; ++rr) s += Dhi[o + rr * 4] + Dlo[o + rr * 4];
                p.tot3_part[(size_t)tile * J + j] = s;
            }
            if (j < F) {
                float s = 0.f;
                for (int rr = 0; rr < rows; ++rr) s += DY[rr * LDY + j];
                db4 += s;
            }
        }
        __syncthreads();          // A3 is dead (dW4 done): it receives dhcat
        mbar_wait(bar, parity);
        parity ^= 1;
        tc_fence_after();
        // ---- dhcat out of TMEM: lane = hcat feature k, column = fibre ---------------------------------
        if (warp < 8 && (warp & 3) * 32 < K9) {
            const int quarter = warp & 3, half = warp >> 2;
            const int k = quarter * 32 + lane;
#pragma unroll
            for (int c0 = half * 32; c0 < (half * 32 + 32 < R ? half * 32 + 32 : R); c0 += 16) {
                float v[16];
                tmem_ld16(tmem_d1 + ((uint32_t)(quarter * 32) << 16) + c0, v);
                if (k < K9) {
#pragma unroll
                    for (int q = 0; q < 16; ++q) A3[(c0 + q) * LDC + k] = v[q];
                }
            }
        }
        tc_fence_before();
        __syncthreads();
        // ---- direct gradient of x_s, moment-polynomial coefficients ------------------------------------
        for (int i = threadIdx.x; i < rows * F; i += blockDim.x) {
            const int rr = i / F, k = i - rr * F;
            p.g_x_s[(row0 + rr) * F + k] = A3[rr * LDC + k];
        }
#pragma unroll
        for (int n = 0; n < NI; ++n) {
            const int rr = it_rr[n];
            if (rr >= rows) continue;
            const float* dh = A3 + it_do[n];
            const unsigned fin = m_fin[n];
            // torch: nan_to_num backward passes the gradient only where the value was finite
            const float d_mean = (fin & 1u) ? dh[0] : 0.f, d_std = (fin & 2u) ? dh[M] : 0.f;
            const float d_skew = (fin & 4u) ? dh[2 * M] : 0.f, d_kurt = (fin & 8u) ? dh[3 * M] : 0.f;
            const float i1 = m_i1[n], i2 = i1 * i1, i3 = i2 * i1, i4 = i2 * i2;
            const float c3 = m_c3[n], c4 = m_c4[n];
            const float d_c3 = d_skew * i3, d_c4 = d_kurt * i4;
            const float d_var = 0.5f * (d_std * m_is1[n] - (3.f * c3 * i4 * d_skew + 4.f * c4 * i4 * i1 * d_kurt) * i1);
            const float d_vr = d_var * (m_vr[n] > 0.f ? 1.f : kSlopeVar);
            const float d_mu = d_mean - 2.f * m_mean[n] * d_vr - 3.f * m_c2[n] * d_c3 - 4.f * c3 * d_c4;
            float* o = p.coefA + row0 * 4 * M + it_co[n];
            o[0] = d_mu;
            o[M] = 2.f * d_vr;
            o[2 * M] = 3.f * d_c3;
            o[3 * M] = 4.f * d_c4;
        }
        __syncthreads();
        tc_fence_after();
    }
    // ---- weight gradients of this CTA -------------------------------------------------------------------
    float* out = p.wpartial + (size_t)blockIdx.x * p.pstride;
    if (warp < 4) {
        // D2: lane = hidden unit j, column = hcat feature k
        const int j = warp * 32 + lane;
#pragma unroll 1
        for (int c0 = 0; c0 < KN; c0 += 16) {
            float v[16];
            if (!first) tmem_ld16(tmem_d2 + ((uint32_t)(warp * 32) << 16) + c0, v);
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int k = c0 + q;
                if (j < J && k < K9) out[j * K9 + k] = first ? 0.f : v[q];
            }
        }
    }
    tc_fence_before();
    accw4.flush(Dhi, out + J * K9, J, 0);     // starts with a __syncthreads()
    if (threadIdx.x >= 32 && threadIdx.x < 32 + F) out[J * K9 + F * J + threadIdx.x - 32] = db4;
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, MM::TMEM_COLS);
}

}  // namespace pfs
