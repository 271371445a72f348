// source_model.cuh -- SModel kernels (reference src/gnn.py:104-154).
//
// edge pass   : m = MLP1([x_t[tgt] | x_e]) per edge (class half pre-projected into Q_t), staged
//               transposed in shared memory; per (fibre, feature) two-pass moments in a fixed order
//               (replaces the four torch_scatter means of src/gnn.py:140-144).
// node pass   : moment finalisation (var, std, skew, kurt, nan_to_num) fused with MLP2 (10F->10F->F)
//               and the BatchNorm tile statistics.
// backward    : node pass (BatchNorm backward, MLP2 backward, moment-polynomial coefficients)
//               then an edge pass (recompute m, dm = A0 + A1 m + A2 d^2 + A3 d^3, MLP1 backward).
#pragma once
#include <cfloat>

#include "common.cuh"

namespace pfs {

// torch.nan_to_num(x, nan=0.0): nan -> 0, +-inf -> +-FLT_MAX
__device__ __forceinline__ float nan_to_num(float x) {
    if (x != x) return 0.f;
    if (isinf(x)) return x > 0.f ? FLT_MAX : -FLT_MAX;
    return x;
}
__device__ __forceinline__ bool finite_f(float x) { return (x == x) && !isinf(x); }

struct SourceEdgeFwdParams {
    Topo tp;
    const float* xe2;      // [G,E,F]
    const float* Qt;       // [G,T,2F] = x_t . W1[:, :F]^T + b1
    const float *w1, *w2, *b2;
    float* moments;        // [G,S,5,2F]: mean, E[m^2], c2, c3, c4
    const float* xaff;     // [G,4,F] (rows 2, 3: scale, shift) of a deferred EdgeModel norm, or null: xe2 then holds z
    float* xe_norm_out;    // [G,E,F] where x_e' = scale z + shift is stored (may alias xe2)
    float* split_rec;      // split tiles: [G,nslots,moment_record_floats(2F)] chunk records (k_split_moments -> moments)
};

// Chunk record of a split tile, per message feature j (rows of M floats): the sums of m and m^2, the sums of the
// 2nd, 3rd and 4th powers of m - (chunk mean), then the chunk's edge count.
__host__ __device__ constexpr int moment_record_floats(int M) { return 5 * M + 1; }

template <int F, bool SPLIT = false>
__global__ void __launch_bounds__(kThreads) k_source_edge_fwd(const SourceEdgeFwdParams p) {
    constexpr int M = 2 * F;
    constexpr int LDT = kTile + 1;
    using CW = MsgEdgeConst<F>;
    __shared__ float MT[M * LDT];   // messages, feature-major
    const Topo& tp = p.tp;
    const int total = tp.ntiles * tp.G;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const Tile t = get_tile<SPLIT>(tp, tile);
        if (threadIdx.x < t.ne) {
            const EdgeRef er = get_edge(tp, t, threadIdx.x);
            float x[F], h[M], m[M];
            load_row<F>(p.xe2 + ((size_t)t.g * tp.E + er.e) * F, x);
            if (p.xaff) {      // the EdgeModel's (double) BatchNorm affine, deferred to its first consumer
                const float* sc = p.xaff + (size_t)t.g * 4 * F + 2 * F;
#pragma unroll
                for (int j = 0; j < F; ++j) x[j] = fmaf(x[j], __ldg(sc + j), __ldg(sc + F + j));
                store_row<F>(p.xe_norm_out + ((size_t)t.g * tp.E + er.e) * F, x);
            }
            load_row<M>(p.Qt + ((size_t)t.g * tp.T + er.tgt) * M, h);
            dense_acc_c<F, M, CW::kW1t>(x, h);
#pragma unroll
            for (int j = 0; j < M; ++j) {
                h[j] = lrelu(h[j]);
                m[j] = c_w[CW::kB2 + j];
            }
            dense_acc_c<M, M, CW::kW2t>(h, m);
#pragma unroll
            for (int j = 0; j < M; ++j) MT[j * LDT + threadIdx.x] = m[j];
        }
        __syncthreads();
        for (int i = threadIdx.x; i < t.nfib * M; i += kThreads) {
            const int lf = i / M, j = i - lf * M;
            int e0, n;
            fibre_range<SPLIT>(tp, t, lf, e0, n);
            const float* col = MT + j * LDT + e0;
            float s1 = 0.f, s2 = 0.f;
            for (int e = 0; e < n; ++e) {
                const float v = col[e];
                s1 += v;
                s2 += v * v;
            }
            const float cnt = (float)max(n, 1);
            const float mean = s1 / cnt;
            float c2 = 0.f, c3 = 0.f, c4 = 0.f;
            for (int e = 0; e < n; ++e) {
                const float d = col[e] - mean;
                const float d2 = d * d;
                c2 += d2;
                c3 += d2 * d;
                c4 += d2 * d2;
            }
            if constexpr (SPLIT) {
                if (t.slot >= 0) {
                    float* r = p.split_rec + ((size_t)t.g * tp.nslots + t.slot) * moment_record_floats(M) + j;
                    r[0] = s1;
                    r[M] = s2;
                    r[2 * M] = c2;
                    r[3 * M] = c3;
                    r[4 * M] = c4;
                    if (j == 0) r[5 * M] = (float)n;
                    continue;
                }
            }
            float* o = p.moments + ((size_t)t.g * tp.S + t.fibre0 + lf) * 5 * M + j;
            o[0] = mean;
            o[M] = s2 / cnt;
            o[2 * M] = c2 / cnt;
            o[3 * M] = c3 / cnt;
            o[4 * M] = c4 / cnt;
        }
        __syncthreads();
    }
}

// Moment rows [mean, E[m^2], c2, c3, c4] of the split fibres from their chunk records: one thread per (graph, split
// fibre, feature) combines the records in slot order in fp64 with the pairwise update of the central moments
// (Chan, Golub and LeVeque; Pebay 2008), so the result does not depend on how the fibre was cut.
__global__ void k_split_moments(const Topo tp, int M, const float* __restrict__ rec, float* __restrict__ moments) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)tp.G * tp.nsplit * M) return;
    const int j = (int)(i % M);
    const long long gs = i / M;
    const int g = (int)(gs / tp.nsplit), sf = (int)(gs - (long long)g * tp.nsplit);
    const int R = 5 * M + 1;
    double n = 0.0, mean = 0.0, sq = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0;
    for (int s = tp.split_ptr[sf]; s < tp.split_ptr[sf + 1]; ++s) {
        const float* r = rec + ((size_t)g * tp.nslots + s) * R;
        const double nb = r[5 * M];
        const double mb = (double)r[j] / nb, b2 = r[2 * M + j], b3 = r[3 * M + j], b4 = r[4 * M + j];
        sq += (double)r[M + j];
        if (n == 0.0) {
            n = nb; mean = mb; m2 = b2; m3 = b3; m4 = b4;
            continue;
        }
        const double na = n, nn = na + nb, d = mb - mean, dn = d / nn, dn2 = dn * dn;
        m4 += b4 + d * dn2 * dn * na * nb * (na * na - na * nb + nb * nb) + 6.0 * dn2 * (na * na * b2 + nb * nb * m2) +
              4.0 * dn * (na * b3 - nb * m3);
        m3 += b3 + d * dn2 * na * nb * (na - nb) + 3.0 * dn * (na * b2 - nb * m2);
        m2 += b2 + d * dn * na * nb;
        mean += dn * nb;
        n = nn;
    }
    float* o = moments + ((size_t)g * tp.S + tp.split_fibre[sf]) * 5 * M + j;
    o[0] = (float)mean;
    o[M] = (float)(sq / n);
    o[2 * M] = (float)(m2 / n);
    o[3 * M] = (float)(m3 / n);
    o[4 * M] = (float)(m4 / n);
}

// ------------------------------------------------------------------------------------------
// node pass geometry: a tile of node_rows<F>() fibres, thread = (row pair, output chunk of 2F)
// ------------------------------------------------------------------------------------------
constexpr int kNodeChunks = 5;                               // 10F outputs = 5 chunks of 2F
template <int F> __host__ __device__ constexpr int node_pairs() { return F <= 10 ? kThreads / kNodeChunks : 25; }  // row pairs (shared memory bound for wide F)
template <int F> __host__ __device__ constexpr int node_rows() { return 2 * node_pairs<F>(); }                          // fibres per node tile

// hcat row (without the u columns): [x_s | mean | std | skew | kurt], finalised from raw moments
// exactly as reference src/gnn.py:141-151.  Writes HC[r][0..9F) for the rows of one tile.
template <int F>
__device__ __forceinline__ void build_hcat(const float* __restrict__ x_s, const float* __restrict__ moments,
                                           size_t row0, int rows, float* HC, int ld) {
    constexpr int M = 2 * F;
    for (int i = threadIdx.x; i < rows * F; i += kThreads) {
        const int r = i / F, k = i - r * F;
        HC[r * ld + k] = __ldg(x_s + (row0 + r) * F + k);
    }
    for (int i = threadIdx.x; i < rows * M; i += kThreads) {
        const int r = i / M, j = i - r * M;
        const float* mo = moments + (row0 + r) * 5 * M + j;
        const float mean = __ldg(mo), ex2 = __ldg(mo + M), c3 = __ldg(mo + 3 * M), c4 = __ldg(mo + 4 * M);
        const float vr = ex2 - mean * mean;
        const float var = vr > 0.f ? vr : kSlopeVar * vr;
        const float std0 = sqrtf(var + kStdEps);
        const float skew = c3 / (std0 * std0 * std0);
        const float kurt = c4 / (std0 * std0 * std0 * std0);
        float* h = HC + r * ld + F + j;
        h[0] = nan_to_num(mean);
        h[M] = sqrtf(nan_to_num(var) + kStdEps);
        h[2 * M] = nan_to_num(skew);
        h[3 * M] = nan_to_num(kurt);
    }
}

struct SourceNodeFwdParams {
    int G, S;
    const float *x_s, *u, *moments;
    const float *w3, *b3, *w4, *b4;
    float* hidden;      // [G,S,10F] saved lrelu(h3)
    float* y_pre;       // [G,S,F]
    float* bn_partial;  // [G,ntiles,2F+2] or null
    int ntiles;         // node tiles per graph
};

template <int F>
struct SourceNodeFwdSmem {
    static constexpr int K9 = 9 * F, J = 10 * F;
    static constexpr int LDH = K9 + 1, LDA = J + 1;
    static constexpr int kBuf = node_rows<F>() * LDA;   // HC, then reused for A3 (LDA >= LDH)
    static constexpr int kFloats = K9 * J + J * F + kBuf + J + F + node_rows<F>() * F;
    static constexpr size_t bytes = sizeof(float) * kFloats;
};

template <int F>
__global__ void __launch_bounds__(kThreads) k_source_node_fwd(const SourceNodeFwdParams p) {
    using SM = SourceNodeFwdSmem<F>;
    constexpr int K9 = SM::K9, J = SM::J, C = 2 * F, LDH = SM::LDH, LDA = SM::LDA;
    extern __shared__ __align__(16) float sm[];
    float* W3t = sm;                 // [k<9F][j<10F]
    float* W4t = W3t + K9 * J;       // [k<10F][f<F]
    float* BUF = W4t + J * F;        // HC [rows][LDH] then A3 [rows][LDA]
    float* b3e = BUF + SM::kBuf;     // [J] b3 + W3[:, 9F:] . u[g]
    float* b4s = b3e + J;            // [F]
    float* YS = b4s + F;             // [rows][F]
    load_w_inmajor<K9, J>(W3t, p.w3, J, 0);
    load_w_inmajor<J, F>(W4t, p.w4, J, 0);
    load_vec<F>(b4s, p.b4);
    __syncthreads();
    const int total = p.ntiles * p.G;
    const int rp = threadIdx.x / kNodeChunks, ch = threadIdx.x - rp * kNodeChunks;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int g = tile / p.ntiles, lt = tile - g * p.ntiles;
        const int f0 = lt * node_rows<F>();
        const int rows = min(node_rows<F>(), p.S - f0);
        const size_t row0 = (size_t)g * p.S + f0;
        build_hcat<F>(p.x_s, p.moments, row0, rows, BUF, LDH);
        for (int j = threadIdx.x; j < J; j += kThreads) {
            float s = __ldg(p.b3 + j);
            for (int k = 0; k < F; ++k) s = fmaf(__ldg(p.w3 + (size_t)j * J + K9 + k), __ldg(p.u + (size_t)g * F + k), s);
            b3e[j] = s;
        }
        __syncthreads();
        float a0[C], a1[C];
        const int r0 = 2 * rp, r1 = 2 * rp + 1;
        const bool live = rp < node_pairs<F>() && r0 < rows;
        if (live) {
            const float* h0 = BUF + r0 * LDH;
            const float* h1 = BUF + (r1 < rows ? r1 : r0) * LDH;
#pragma unroll
            for (int c = 0; c < C; ++c) a0[c] = a1[c] = b3e[ch * C + c];
#pragma unroll 2
            for (int k = 0; k < K9; ++k) {
                const float x0 = h0[k], x1 = h1[k];
                const float4* w = reinterpret_cast<const float4*>(W3t + k * J + ch * C);
#pragma unroll
                for (int c = 0; c < C / 4; ++c) {
                    const float4 v = w[c];
                    a0[4 * c] = fmaf(v.x, x0, a0[4 * c]);         a1[4 * c] = fmaf(v.x, x1, a1[4 * c]);
                    a0[4 * c + 1] = fmaf(v.y, x0, a0[4 * c + 1]); a1[4 * c + 1] = fmaf(v.y, x1, a1[4 * c + 1]);
                    a0[4 * c + 2] = fmaf(v.z, x0, a0[4 * c + 2]); a1[4 * c + 2] = fmaf(v.z, x1, a1[4 * c + 2]);
                    a0[4 * c + 3] = fmaf(v.w, x0, a0[4 * c + 3]); a1[4 * c + 3] = fmaf(v.w, x1, a1[4 * c + 3]);
                }
            }
        }
        __syncthreads();   // every thread is done reading HC: reuse the buffer for the activations
        if (live) {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                a0[c] = lrelu(a0[c]);
                a1[c] = lrelu(a1[c]);
                BUF[r0 * LDA + ch * C + c] = a0[c];
            }
            store_row<C>(p.hidden + (row0 + r0) * J + ch * C, a0);
            if (r1 < rows) {
#pragma unroll
                for (int c = 0; c < C; ++c) BUF[r1 * LDA + ch * C + c] = a1[c];
                store_row<C>(p.hidden + (row0 + r1) * J + ch * C, a1);
            }
        }
        __syncthreads();
        // second layer: y[r][f] for feature pairs
        for (int i = threadIdx.x; i < rows * (F / 2); i += kThreads) {
            const int r = i / (F / 2), f2 = i - r * (F / 2);
            float y0 = b4s[2 * f2], y1 = b4s[2 * f2 + 1];
            const float* a = BUF + r * LDA;
#pragma unroll 4
            for (int k = 0; k < J; ++k) {
                const float2 w = *reinterpret_cast<const float2*>(W4t + k * F + 2 * f2);
                y0 = fmaf(w.x, a[k], y0);
                y1 = fmaf(w.y, a[k], y1);
            }
            YS[r * F + 2 * f2] = y0;
            YS[r * F + 2 * f2 + 1] = y1;
            *reinterpret_cast<float2*>(p.y_pre + (row0 + r) * F + 2 * f2) = make_float2(y0, y1);
        }
        __syncthreads();
        if (p.bn_partial && threadIdx.x < F) {
            float s = 0.f;
            for (int r = 0; r < rows; ++r) s += YS[r * F + threadIdx.x];
            const float mean = s / (float)rows;
            float m2 = 0.f;
            for (int r = 0; r < rows; ++r) {
                const float d = YS[r * F + threadIdx.x] - mean;
                m2 += d * d;
            }
            float* o = p.bn_partial + (size_t)tile * bn_partial_stride(F);
            o[threadIdx.x] = mean;
            o[F + threadIdx.x] = m2;
            if (threadIdx.x == 0) o[2 * F] = (float)rows;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// backward, node pass
// ------------------------------------------------------------------------------------------
struct SourceNodeBwdParams {
    int G, S, ntiles;
    int mode;                 // 0 not normed, 1 train, 2 eval
    float eps;
    const float *x_s, *moments, *hidden, *y_pre, *gout;
    const float* bn_save;     // [G,4,F]
    const float* bn_stat;     // [G,2,F] sum g, sum g xhat (train)
    const float *w3, *w4;
    float* g_x_s;             // [G,S,F] direct part
    float* coefA;             // [G,S,4,2F]
    float* tot3_part;         // [G,ntiles,10F] column sums of dh3 per node tile
    float* wpartial;          // [ncta][pstride]: dW3 [10F*9F], dW4 [F*10F], db4 [F]
    int pstride;
};

template <int F>
struct SourceNodeBwdSmem {
    static constexpr int K9 = 9 * F, J = 10 * F;
    static constexpr int LDH = K9 + 1, LDA = J + 1, LDY = F + 1;
    // dW3 on threads [0, 224), dW4 on the last warp (F <= 14); F = 16 shares the first warp
    static_assert(F * F <= kThreads && 2 * F <= 32, "node kernels support Fdim <= 16");
    static constexpr int kNT3 = (F * F <= 224) ? 224 : kThreads;
    static constexpr int kT04 = (F * F <= 224) ? 224 : 0;
    using AccW3 = OuterAcc<J, K9, 10, 9, 0, kNT3>;
    static constexpr int kNT4 = ((F / 2) * 5 <= 32) ? 32 : 64;
    using AccW4 = OuterAcc<F, J, 2, 2 * F, kT04, kNT4>;
    static constexpr int kRows = node_rows<F>() * (LDH + 2 * LDA + LDY);
    static constexpr int kScr = AccW3::kScratchFloats > AccW4::kScratchFloats ? AccW3::kScratchFloats : AccW4::kScratchFloats;
    // the row buffers double as the cross-group scratch of the weight-gradient flush
    static constexpr int kRegion = kRows > kScr ? kRows : kScr;
    static constexpr int kFloats = J * K9 + F * J + kRegion;
    static constexpr size_t bytes = sizeof(float) * kFloats;
};

template <int F>
__global__ void __launch_bounds__(kThreads) k_source_node_bwd(const SourceNodeBwdParams p) {
    using SM = SourceNodeBwdSmem<F>;
    constexpr int K9 = SM::K9, J = SM::J, C = 2 * F, M = 2 * F, LDH = SM::LDH, LDA = SM::LDA, LDY = SM::LDY;
    extern __shared__ __align__(16) float sm[];
    float* W3o = sm;                      // [j<10F][k<9F]  (w3 rows, first 9F columns)
    float* W4o = W3o + J * K9;            // [f<F][j<10F]   (w4 as stored)
    float* HC = W4o + F * J;              // [rows][LDH]  hcat, later dhcat
    float* A3 = HC + node_rows<F>() * LDH;     // [rows][LDA]
    float* DH3 = A3 + node_rows<F>() * LDA;    // [rows][LDA]
    float* DY = DH3 + node_rows<F>() * LDA;    // [rows][LDY]
    load_w_outmajor<K9, J>(W3o, p.w3, J, 0);
    load_w_outmajor<J, F>(W4o, p.w4, J, 0);
    __syncthreads();
    using AccW3 = typename SM::AccW3;
    using AccW4 = typename SM::AccW4;
    AccW3 accw3;
    AccW4 accw4;
    accw3.init();
    accw4.init();
    float db4 = 0.f;   // thread f < F
    const int total = p.ntiles * p.G;
    const int rp = threadIdx.x / kNodeChunks, ch = threadIdx.x - rp * kNodeChunks;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int g = tile / p.ntiles, lt = tile - g * p.ntiles;
        const int f0 = lt * node_rows<F>();
        const int rows = min(node_rows<F>(), p.S - f0);
        const size_t row0 = (size_t)g * p.S + f0;
        build_hcat<F>(p.x_s, p.moments, row0, rows, HC, LDH);
        // dy = BatchNorm backward of the upstream gradient
        {
            const float* sv = p.bn_save + (size_t)g * 4 * F;
            const float* st = p.bn_stat + (size_t)g * 2 * F;
            const float invS = 1.f / (float)p.S;
            for (int i = threadIdx.x; i < rows * F; i += kThreads) {
                const int r = i / F, f = i - r * F;
                const float gv = __ldg(p.gout + (row0 + r) * F + f);
                float dy;
                if (p.mode == 1) {
                    const float rstd = rsqrtf(sv[F + f] + p.eps);
                    const float xh = (__ldg(p.y_pre + (row0 + r) * F + f) - sv[f]) * rstd;
                    dy = sv[2 * F + f] * (gv - st[f] * invS - xh * st[F + f] * invS);
                } else if (p.mode == 2) {
                    dy = gv * sv[2 * F + f];
                } else {
                    dy = gv;
                }
                DY[r * LDY + f] = dy;
            }
        }
        __syncthreads();
        // dh3 = (dy . W4) * lrelu'(h3), two rows x one chunk per thread
        {
            const int r0 = 2 * rp, r1 = 2 * rp + 1;
            if (rp < node_pairs<F>() && r0 < rows) {
                const bool two = r1 < rows;
                float a0[C], a1[C], d0[C], d1[C];
                load_row<C>(p.hidden + (row0 + r0) * J + ch * C, a0);
                load_row<C>(p.hidden + (row0 + (two ? r1 : r0)) * J + ch * C, a1);
#pragma unroll
                for (int c = 0; c < C; ++c) d0[c] = d1[c] = 0.f;
                const float* y0 = DY + r0 * LDY;
                const float* y1 = DY + (two ? r1 : r0) * LDY;
#pragma unroll
                for (int f = 0; f < F; ++f) {
                    const float v0 = y0[f], v1 = y1[f];
                    const float4* w = reinterpret_cast<const float4*>(W4o + f * J + ch * C);
#pragma unroll
                    for (int c = 0; c < C / 4; ++c) {
                        const float4 v = w[c];
                        d0[4 * c] = fmaf(v.x, v0, d0[4 * c]);         d1[4 * c] = fmaf(v.x, v1, d1[4 * c]);
                        d0[4 * c + 1] = fmaf(v.y, v0, d0[4 * c + 1]); d1[4 * c + 1] = fmaf(v.y, v1, d1[4 * c + 1]);
                        d0[4 * c + 2] = fmaf(v.z, v0, d0[4 * c + 2]); d1[4 * c + 2] = fmaf(v.z, v1, d1[4 * c + 2]);
                        d0[4 * c + 3] = fmaf(v.w, v0, d0[4 * c + 3]); d1[4 * c + 3] = fmaf(v.w, v1, d1[4 * c + 3]);
                    }
                }
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    A3[r0 * LDA + ch * C + c] = a0[c];
                    DH3[r0 * LDA + ch * C + c] = d0[c] * (a0[c] > 0.f ? 1.f : kSlope);
                }
                if (two) {
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        A3[r1 * LDA + ch * C + c] = a1[c];
                        DH3[r1 * LDA + ch * C + c] = d1[c] * (a1[c] > 0.f ? 1.f : kSlope);
                    }
                }
            }
        }
        __syncthreads();
        accw3.accumulate(DH3, LDA, HC, LDH, rows);
        accw4.accumulate(DY, LDY, A3, LDA, rows);
        if (threadIdx.x < F) {
            float s = 0.f;
            for (int r = 0; r < rows; ++r) s += DY[r * LDY + threadIdx.x];
            db4 += s;
        }
        __syncthreads();   // HC is dead from here: it receives dhcat
        // dhcat[r][k] = sum_j dh3[r][j] W3[j][k], item = (row pair, chunk of F columns)
        for (int i = threadIdx.x; i < ((rows + 1) / 2) * 9; i += kThreads) {
            const int pr = i / 9, kc = i - pr * 9;
            const int r0 = 2 * pr, r1 = (2 * pr + 1 < rows) ? 2 * pr + 1 : r0;
            float o0[F], o1[F];
#pragma unroll
            for (int k = 0; k < F; ++k) o0[k] = o1[k] = 0.f;
            const float* d0 = DH3 + r0 * LDA;
            const float* d1 = DH3 + r1 * LDA;
#pragma unroll 2
            for (int j = 0; j < J; ++j) {
                const float v0 = d0[j], v1 = d1[j];
                const float2* w = reinterpret_cast<const float2*>(W3o + j * K9 + kc * F);
#pragma unroll
                for (int k = 0; k < F / 2; ++k) {
                    const float2 v = w[k];
                    o0[2 * k] = fmaf(v.x, v0, o0[2 * k]);         o1[2 * k] = fmaf(v.x, v1, o1[2 * k]);
                    o0[2 * k + 1] = fmaf(v.y, v0, o0[2 * k + 1]); o1[2 * k + 1] = fmaf(v.y, v1, o1[2 * k + 1]);
                }
            }
#pragma unroll
            for (int k = 0; k < F; ++k) {
                HC[r0 * LDH + kc * F + k] = o0[k];
                if (r1 != r0) HC[r1 * LDH + kc * F + k] = o1[k];
            }
        }
        __syncthreads();
        // direct gradient of x_s, column sums of dh3, moment-polynomial coefficients
        for (int i = threadIdx.x; i < rows * F; i += kThreads) {
            const int r = i / F, k = i - r * F;
            p.g_x_s[(row0 + r) * F + k] = HC[r * LDH + k];
        }
        for (int j = threadIdx.x; j < J; j += kThreads) {
            float s = 0.f;
            for (int r = 0; r < rows; ++r) s += DH3[r * LDA + j];
            p.tot3_part[(size_t)tile * J + j] = s;
        }
        for (int i = threadIdx.x; i < rows * M; i += kThreads) {
            const int r = i / M, j = i - r * M;
            const float* mo = p.moments + (row0 + r) * 5 * M + j;
            const float mean = __ldg(mo), ex2 = __ldg(mo + M), c2 = __ldg(mo + 2 * M), c3 = __ldg(mo + 3 * M),
                        c4 = __ldg(mo + 4 * M);
            const float* dh = HC + r * LDH + F + j;
            float d_mean = dh[0], d_std = dh[M], d_skew = dh[2 * M], d_kurt = dh[3 * M];
            const float vr = ex2 - mean * mean;
            const float var = vr > 0.f ? vr : kSlopeVar * vr;
            const float std0 = sqrtf(var + kStdEps);
            const float s3 = std0 * std0 * std0, s4 = s3 * std0;
            // torch: nan_to_num backward passes the gradient only where the value was finite
            if (!finite_f(mean)) d_mean = 0.f;
            if (!finite_f(var)) d_std = 0.f;
            if (!finite_f(c3 / s3)) d_skew = 0.f;
            if (!finite_f(c4 / s4)) d_kurt = 0.f;
            const float std1 = sqrtf(nan_to_num(var) + kStdEps);
            const float d_c3 = d_skew / s3, d_c4 = d_kurt / s4;
            const float d_var = d_std / (2.f * std1) + (-3.f * c3 / s4 * d_skew - 4.f * c4 / (s4 * std0) * d_kurt) / (2.f * std0);
            const float d_vr = d_var * (vr > 0.f ? 1.f : kSlopeVar);
            const float d_mu = d_mean - 2.f * mean * d_vr - 3.f * c2 * d_c3 - 4.f * c3 * d_c4;
            // the count is recovered by the edge pass (it knows the fibre degree): store un-normalised
            float* o = p.coefA + (row0 + r) * 4 * M + j;
            o[0] = d_mu;
            o[M] = 2.f * d_vr;
            o[2 * M] = 3.f * d_c3;
            o[3 * M] = 4.f * d_c4;
        }
        __syncthreads();
    }
    float* out = p.wpartial + (size_t)blockIdx.x * p.pstride;
    accw3.flush(HC, out, K9, 0);
    accw4.flush(HC, out + J * K9, J, 0);
    if (threadIdx.x < F) out[J * K9 + F * J + threadIdx.x] = db4;
}

// ------------------------------------------------------------------------------------------
// backward, edge pass
// ------------------------------------------------------------------------------------------
struct SourceEdgeBwdParams {
    Topo tp;
    const float *xe2, *Qt;
    const float *w1, *w2, *b2;
    const float *moments, *coefA;   // [G,S,5,2F], [G,S,4,2F]
    float* g_x_e;                   // [G,E,F]
    const float* g_add;             // optional [G,E,F] added to g_x_e on store
    float* class_part;              // dense: [G,ntiles,T,2F] class sums of dhs
    float* dhs_rows;                // general: [G,E(q),2F]
    float* wpartial;                // [ncta][pstride]: dW1_e [2F*F], dW2 [2F*2F], db2 [2F]
    int pstride;
};

template <int F>
struct SourceEdgeBwdSmem {
    static constexpr int M = 2 * F;
    static constexpr int LDM = M + 4, LDF = F + 2;
    static constexpr int kWeights = 0;   // the weights live in the constant bank (MsgEdgeConst)
    static constexpr int kTiles = kTile * (3 * LDM + LDF);
    static constexpr size_t bytes = sizeof(float) * (kWeights + kTiles);
};

template <int F, bool SPLIT = false>
__global__ void __launch_bounds__(kThreads, (F <= 10 ? 2 : 1)) k_source_edge_bwd(const SourceEdgeBwdParams p) {
    using SM = SourceEdgeBwdSmem<F>;
    constexpr int M = 2 * F, LDM = SM::LDM, LDF = SM::LDF;
    extern __shared__ __align__(16) float sm[];
    using CW = MsgEdgeConst<F>;
    float* DM = sm;                  // [kTile][LDM]
    float* AS = DM + kTile * LDM;
    float* DHS = AS + kTile * LDM;
    float* XE = DHS + kTile * LDM;   // [kTile][LDF]
    using AccW2 = OuterAcc<M, M, 4, F / 2, 0, 160>;            // dW2[j][k]   = sum dm_j as_k
    using AccW1 = OuterAcc<M, F, 4, F / 2, 160, 96>;           // dW1_e[j][k] = sum dhs_j x_k
    AccW2 accw2;
    AccW1 accw1;
    accw2.init();
    accw1.init();
    float dmsum[M];
#pragma unroll
    for (int j = 0; j < M; ++j) dmsum[j] = 0.f;
    const Topo& tp = p.tp;
    const int total = tp.ntiles * tp.G;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const Tile t = get_tile<SPLIT>(tp, tile);
        if (threadIdx.x == 0 && tile + (int)gridDim.x < total && tp.layout == PFS_LAYOUT_DENSE) {   // next tile -> L2
            const Tile tn = get_tile<SPLIT>(tp, tile + gridDim.x);
            const size_t off = ((size_t)tn.g * tp.E + tn.q0) * F, bytes = (size_t)tn.ne * F * sizeof(float);
            const size_t frow = (size_t)tn.g * tp.S + tn.fibre0;
            bulk_prefetch_l2(p.xe2 + off, bytes);
            if (p.g_add) bulk_prefetch_l2(p.g_add + off, bytes);
            bulk_prefetch_l2(p.coefA + frow * 4 * M, (size_t)tn.nfib * 4 * M * sizeof(float));
            bulk_prefetch_l2(p.moments + frow * 5 * M, (size_t)tn.nfib * 5 * M * sizeof(float));
        }
        if (threadIdx.x < t.ne) {
            const EdgeRef er = get_edge(tp, t, threadIdx.x);
            const size_t row = ((size_t)t.g * tp.E + er.e) * F;
            float x[F], h[M], a[M], m[M];
            load_row<F>(p.xe2 + row, x);
            load_row<M>(p.Qt + ((size_t)t.g * tp.T + er.tgt) * M, h);
            dense_acc_c<F, M, CW::kW1t>(x, h);
#pragma unroll
            for (int j = 0; j < M; ++j) {
                a[j] = lrelu(h[j]);
                m[j] = c_w[CW::kB2 + j];
            }
            dense_acc_c<M, M, CW::kW2t>(a, m);
            // dm = (A0 + A1 m + A2 d^2 + A3 d^3) / count, count = the fibre's degree (a split tile holds a chunk of it)
            int n;
            if constexpr (SPLIT) {
                n = tp.rowptr[er.src + 1] - tp.rowptr[er.src];
            } else {
                int e0;
                fibre_range(tp, t, er.src - t.fibre0, e0, n);
            }
            const float inv = 1.f / (float)max(n, 1);
            const size_t frow = (size_t)t.g * tp.S + er.src;
            const float* cA = p.coefA + frow * 4 * M;
            const float* mo = p.moments + frow * 5 * M;
            float dm[M];
            {
                float c0[M], mu[M];
                load_row<M>(cA, c0);
                load_row<M>(mo, mu);
#pragma unroll
                for (int j = 0; j < M; ++j) {
                    dm[j] = c0[j];
                    mu[j] = m[j] - mu[j];   // d
                    c0[j] = mu[j] * mu[j];  // d^2
                }
                float c1[M];
                load_row<M>(cA + M, c1);
#pragma unroll
                for (int j = 0; j < M; ++j) dm[j] = fmaf(c1[j], m[j], dm[j]);
                load_row<M>(cA + 2 * M, c1);
#pragma unroll
                for (int j = 0; j < M; ++j) dm[j] = fmaf(c1[j], c0[j], dm[j]);
                load_row<M>(cA + 3 * M, c1);
#pragma unroll
                for (int j = 0; j < M; ++j) {
                    dm[j] = fmaf(c1[j], c0[j] * mu[j], dm[j]) * inv;
                    dmsum[j] += dm[j];
                }
            }
            store_row_smem<M>(DM + threadIdx.x * LDM, dm);
            store_row_smem<M>(AS + threadIdx.x * LDM, a);
            store_row_smem<F>(XE + threadIdx.x * LDF, x);
            float da[M];
#pragma unroll
            for (int k = 0; k < M; ++k) da[k] = 0.f;
            dense_acc_c<M, M, CW::kW2o>(dm, da);
#pragma unroll
            for (int k = 0; k < M; ++k) da[k] *= dlrelu(h[k]);   // dhs
            store_row_smem<M>(DHS + threadIdx.x * LDM, da);
            float dx[F];
#pragma unroll
            for (int k = 0; k < F; ++k) dx[k] = 0.f;
            dense_acc_c<M, F, CW::kW1o>(da, dx);
            if (p.g_add) add_row<F>(p.g_add + row, dx);
            store_row<F>(p.g_x_e + row, dx);
            if (p.dhs_rows) store_row<M>(p.dhs_rows + ((size_t)t.g * tp.E + t.q0 + threadIdx.x) * M, da);
        }
        __syncthreads();
        accw2.accumulate(DM, LDM, AS, LDM, t.ne);
        accw1.accumulate(DHS, LDM, XE, LDF, t.ne);
        if (p.class_part) tile_class_sums<M, LDM>(tp, t, DHS, p.class_part + (size_t)tile * tp.T * M);
        __syncthreads();
    }
    float* out = p.wpartial + (size_t)blockIdx.x * p.pstride;
    accw1.flush(DM, out, F, 0);
    accw2.flush(DM, out + M * F, M, 0);
    {
        float* red = DM;
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
        for (int j = 0; j < M; ++j) {
            const float v = warp_sum(dmsum[j]);
            if (lane == 0) red[w * M + j] = v;
        }
        __syncthreads();
        if (threadIdx.x < M) {
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < kWarps; ++i) s += red[i * M + threadIdx.x];
            out[M * F + M * M + threadIdx.x] = s;
        }
    }
}

}  // namespace pfs
