// target_model.cuh -- TModel kernels (reference src/gnn.py:157-192) and GlobalModel
// (reference src/gnn.py:195-223).
//
// The target message MLP's last Linear is commuted with the scatter-sum (both are linear):
//   agg[i] = sum_{e in class i} (W2 . a_e + b2) = W2 . (sum_e a_e) + count_i * b2,
// so the edge pass only sums the hidden activations a_e = lrelu(R_s[src] + W1_e . x_e) per class
// (deterministic per-tile class sums + a fixed-order second stage), and the tiny per-class tail
// (W2, MLP2, BatchNorm over the T classes) runs in one CTA per graph.
#pragma once
#include "common.cuh"

namespace pfs {

struct TargetEdgeFwdParams {
    Topo tp;
    const float* xe2;       // [G,E,F]
    const float* Rs;        // [G,S,2F] = x_s' . W1[:, :F]^T + b1
    const float* w1;        // [2F,2F]
    float* class_part;      // dense: [G,ntiles,T,2F]
    float* act_rows;        // general: [G,E(q),2F]
};

template <int F, bool SPLIT = false>
__global__ void __launch_bounds__(kThreads) k_target_edge_fwd(const TargetEdgeFwdParams p) {
    constexpr int M = 2 * F, LDM = M + 1;
    using CW = MsgEdgeConst<F>;      // only W1t / W1o of the layout are used by the TModel kernels
    __shared__ float AT[kTile * LDM];
    const Topo& tp = p.tp;
    const int total = tp.ntiles * tp.G;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const Tile t = get_tile<SPLIT>(tp, tile);
        if (threadIdx.x < t.ne) {
            const EdgeRef er = get_edge(tp, t, threadIdx.x);
            float x[F], h[M];
            load_row<F>(p.xe2 + ((size_t)t.g * tp.E + er.e) * F, x);
            load_row<M>(p.Rs + ((size_t)t.g * tp.S + er.src) * M, h);
            dense_acc_c<F, M, CW::kW1t>(x, h);
#pragma unroll
            for (int j = 0; j < M; ++j) h[j] = lrelu(h[j]);
            if (p.act_rows) {
                store_row<M>(p.act_rows + ((size_t)t.g * tp.E + t.q0 + threadIdx.x) * M, h);
            } else {
#pragma unroll
                for (int j = 0; j < M; ++j) AT[threadIdx.x * LDM + j] = h[j];
            }
        }
        if (p.class_part) {
            __syncthreads();
            float* cp = p.class_part + (size_t)tile * tp.T * M;
            for (int i = threadIdx.x; i < tp.T * M; i += kThreads) {
                const int c = i / M, k = i - c * M;
                float s = 0.f;
                for (int lf = 0; lf < t.nfib; ++lf) s += AT[(lf * tp.T + c) * LDM + k];
                cp[i] = s;
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------
// per-class tail, one CTA per graph.  Dynamic shared memory: T * (3F + 4F + F) + 4F floats.
// ------------------------------------------------------------------------------------------
struct TargetTailParams {
    int G, T, F;
    int mode;                    // 0 not normed, 1 train, 2 eval
    float eps;
    const float* x_t;            // [G,T,F]
    const float* u;              // [G,F]
    const float* act_sum;        // [G,T,2F]
    const int* colptr;           // class degrees (general layout) or null
    int dense_count;             // S for the dense layout
    const float *w2, *b2, *w3, *b3, *w4, *b4, *gamma, *beta, *rm, *rv;
    // forward
    float* y_pre;                // [G,T,F]
    float* x_t_out;              // [G,T,F]
    float* bn_save;              // [G,4,F]
    // backward
    const float* gout;           // [G,T,F]
    float* g_x_t;                // [G,T,F] direct part
    float* g_u;                  // [G,F]
    float* dasum;                // [G,T,2F] gradient table gathered by the edge pass
    float* gpartial;             // [G][tail_partial_floats(F)]
};

// layout of one graph's parameter-gradient partial (floats)
__host__ __device__ constexpr int tail_off_w2(int F) { return 0; }                       // [2F,2F]
__host__ __device__ constexpr int tail_off_b2(int F) { return 4 * F * F; }               // [2F]
__host__ __device__ constexpr int tail_off_w3(int F) { return 4 * F * F + 2 * F; }       // [4F,4F]
__host__ __device__ constexpr int tail_off_b3(int F) { return 20 * F * F + 2 * F; }      // [4F]
__host__ __device__ constexpr int tail_off_w4(int F) { return 20 * F * F + 6 * F; }      // [F,4F]
__host__ __device__ constexpr int tail_off_b4(int F) { return 24 * F * F + 6 * F; }      // [F]
__host__ __device__ constexpr int tail_off_gamma(int F) { return 24 * F * F + 7 * F; }   // [F]
__host__ __device__ constexpr int tail_off_beta(int F) { return 24 * F * F + 8 * F; }    // [F]
__host__ __device__ constexpr int tail_partial_floats(int F) { return 24 * F * F + 9 * F; }

__device__ __forceinline__ float class_count(const TargetTailParams& p, int i) {
    return p.colptr ? (float)(p.colptr[i + 1] - p.colptr[i]) : (float)p.dense_count;
}

// shared by forward and backward: hcat = [x_t | agg], b3e = b3 + W3[:, 3F:] . u, a3 = lrelu(h3)
__device__ __forceinline__ void tail_forward_core(const TargetTailParams& p, int g, float* HC, float* A3, float* b3e) {
    const int F = p.F, T = p.T, M = 2 * F, H = 4 * F, K3 = 3 * F;
    for (int i = threadIdx.x; i < T * F; i += blockDim.x) {
        const int r = i / F, k = i - r * F;
        HC[r * K3 + k] = p.x_t[((size_t)g * T + r) * F + k];
    }
    for (int i = threadIdx.x; i < T * M; i += blockDim.x) {
        const int r = i / M, j = i - r * M;
        const float* a = p.act_sum + ((size_t)g * T + r) * M;
        float s = class_count(p, r) * p.b2[j];
        for (int k = 0; k < M; ++k) s = fmaf(a[k], p.w2[j * M + k], s);
        HC[r * K3 + F + j] = s;
    }
    for (int j = threadIdx.x; j < H; j += blockDim.x) {
        float s = p.b3[j];
        for (int k = 0; k < F; ++k) s = fmaf(p.w3[j * H + K3 + k], p.u[(size_t)g * F + k], s);
        b3e[j] = s;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < T * H; i += blockDim.x) {
        const int r = i / H, j = i - r * H;
        float s = b3e[j];
        for (int k = 0; k < K3; ++k) s = fmaf(HC[r * K3 + k], p.w3[j * H + k], s);
        A3[r * H + j] = s > 0.f ? s : kSlope * s;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kThreads) k_target_tail_fwd(const TargetTailParams p) {
    extern __shared__ __align__(16) float sm[];
    const int F = p.F, T = p.T, H = 4 * F, K3 = 3 * F;
    const int g = blockIdx.x;
    float* HC = sm;               // [T][3F]
    float* A3 = HC + T * K3;      // [T][4F]
    float* Y = A3 + T * H;        // [T][F]
    float* b3e = Y + T * F;       // [4F]
    tail_forward_core(p, g, HC, A3, b3e);
    for (int i = threadIdx.x; i < T * F; i += blockDim.x) {
        const int r = i / F, f = i - r * F;
        float s = p.b4[f];
        for (int j = 0; j < H; ++j) s = fmaf(A3[r * H + j], p.w4[f * H + j], s);
        Y[i] = s;
        p.y_pre[(size_t)g * T * F + i] = s;
    }
    __syncthreads();
    float* sv = p.bn_save + (size_t)g * 4 * F;
    if (p.mode == 1) {
        if (threadIdx.x < F) {
            const int f = threadIdx.x;
            float s = 0.f;
            for (int r = 0; r < T; ++r) s += Y[r * F + f];
            const float mean = s / (float)T;
            float m2 = 0.f;
            for (int r = 0; r < T; ++r) {
                const float d = Y[r * F + f] - mean;
                m2 += d * d;
            }
            const float var = m2 / (float)T;
            const float scale = p.gamma[f] * (float)(1.0 / sqrt((double)var + (double)p.eps));
            sv[f] = mean;
            sv[F + f] = var;
            sv[2 * F + f] = scale;
            sv[3 * F + f] = p.beta[f] - mean * scale;
        }
    } else if (p.mode == 2) {
        if (threadIdx.x < F) {
            const int f = threadIdx.x;
            const float scale = p.gamma[f] * (float)(1.0 / sqrt((double)p.rv[f] + (double)p.eps));
            sv[f] = p.rm[f];
            sv[F + f] = p.rv[f];
            sv[2 * F + f] = scale;
            sv[3 * F + f] = p.beta[f] - p.rm[f] * scale;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < T * F; i += blockDim.x) {
        const int f = i % F;
        p.x_t_out[(size_t)g * T * F + i] = p.mode == 0 ? Y[i] : fmaf(Y[i], sv[2 * F + f], sv[3 * F + f]);
    }
}

// backward tail: dynamic shared memory T * (3F + 4F + 4F + F) + 4F + 2F floats
__global__ void __launch_bounds__(kThreads) k_target_tail_bwd(const TargetTailParams p) {
    extern __shared__ __align__(16) float sm[];
    const int F = p.F, T = p.T, M = 2 * F, H = 4 * F, K3 = 3 * F;
    const int g = blockIdx.x;
    float* HC = sm;               // [T][3F]  hcat, later dhcat
    float* A3 = HC + T * K3;      // [T][4F]  hidden activations, overwritten in place by dh3
    float* DH = A3;
    float* DY = A3 + T * H;       // [T][F]
    float* b3e = DY + T * F;      // [4F]
    float* st = b3e + H;          // [2F] sum g, sum g xhat
    tail_forward_core(p, g, HC, A3, b3e);
    float* gp = p.gpartial + (size_t)g * tail_partial_floats(F);
    const float* sv = p.bn_save + (size_t)g * 4 * F;
    const float* go = p.gout + (size_t)g * T * F;
    const float* yp = p.y_pre + (size_t)g * T * F;
    // BatchNorm backward over the T rows
    if (threadIdx.x < F) {
        const int f = threadIdx.x;
        float a = 0.f, b = 0.f, c = 0.f;
        if (p.mode == 1) {
            const float r = rsqrtf(sv[F + f] + p.eps);
            for (int i = 0; i < T; ++i) {
                const float gv = go[i * F + f];
                a += gv;
                b += gv * ((yp[i * F + f] - sv[f]) * r);
            }
            gp[tail_off_gamma(F) + f] = b;
            gp[tail_off_beta(F) + f] = a;
        } else if (p.mode == 2) {
            const float r = rsqrtf(p.rv[f] + p.eps);
            for (int i = 0; i < T; ++i) {
                const float gv = go[i * F + f];
                a += gv;
                c += gv * (yp[i * F + f] - p.rm[f]) * r;
            }
            gp[tail_off_gamma(F) + f] = c;
            gp[tail_off_beta(F) + f] = a;
        } else {
            gp[tail_off_gamma(F) + f] = 0.f;
            gp[tail_off_beta(F) + f] = 0.f;
        }
        st[f] = a;
        st[F + f] = b;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < T * F; i += blockDim.x) {
        const int f = i % F;
        const float gv = go[i];
        float dy;
        if (p.mode == 1) {
            const float xh = (yp[i] - sv[f]) * rsqrtf(sv[F + f] + p.eps);
            dy = sv[2 * F + f] * (gv - st[f] / (float)T - xh * st[F + f] / (float)T);
        } else if (p.mode == 2) {
            dy = gv * sv[2 * F + f];
        } else {
            dy = gv;
        }
        DY[i] = dy;
    }
    __syncthreads();
    // dW4, db4
    for (int i = threadIdx.x; i < F * H; i += blockDim.x) {
        const int f = i / H, j = i - f * H;
        float s = 0.f;
        for (int r = 0; r < T; ++r) s = fmaf(DY[r * F + f], A3[r * H + j], s);
        gp[tail_off_w4(F) + i] = s;
    }
    if (threadIdx.x < F) {
        float s = 0.f;
        for (int r = 0; r < T; ++r) s += DY[r * F + threadIdx.x];
        gp[tail_off_b4(F) + threadIdx.x] = s;
    }
    __syncthreads();              // dW4 has read every activation: dh3 may overwrite them
    // dh3 (in place over the activations: only their sign is needed)
    for (int i = threadIdx.x; i < T * H; i += blockDim.x) {
        const int r = i / H, j = i - r * H;
        float s = 0.f;
        for (int f = 0; f < F; ++f) s = fmaf(DY[r * F + f], p.w4[f * H + j], s);
        DH[i] = s * (A3[i] > 0.f ? 1.f : kSlope);
    }
    __syncthreads();
    // dW3 (all 4F columns: hcat columns then the u columns), db3, du
    for (int i = threadIdx.x; i < H * H; i += blockDim.x) {
        const int j = i / H, k = i - j * H;
        float s = 0.f;
        if (k < K3) {
            for (int r = 0; r < T; ++r) s = fmaf(DH[r * H + j], HC[r * K3 + k], s);
        } else {
            float tot = 0.f;
            for (int r = 0; r < T; ++r) tot += DH[r * H + j];
            s = tot * p.u[(size_t)g * F + (k - K3)];
        }
        gp[tail_off_w3(F) + i] = s;
    }
    for (int j = threadIdx.x; j < H; j += blockDim.x) {
        float tot = 0.f;
        for (int r = 0; r < T; ++r) tot += DH[r * H + j];
        gp[tail_off_b3(F) + j] = tot;
        b3e[j] = tot;   // reuse: column sums of dh3
    }
    __syncthreads();
    if (threadIdx.x < F) {
        float s = 0.f;
        for (int j = 0; j < H; ++j) s = fmaf(b3e[j], p.w3[j * H + K3 + threadIdx.x], s);
        p.g_u[(size_t)g * F + threadIdx.x] = s;
    }
    __syncthreads();
    // dhcat = dh3 . W3[:, :3F]  (overwrites HC after everyone is done with it)
    float* DHC = HC;   // hcat is dead after dW3: reuse as [T][3F]
    for (int i = threadIdx.x; i < T * K3; i += blockDim.x) {
        const int r = i / K3, k = i - r * K3;
        float s = 0.f;
        for (int j = 0; j < H; ++j) s = fmaf(DH[r * H + j], p.w3[j * H + k], s);
        DHC[i] = s;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < T * F; i += blockDim.x) {
        const int r = i / F, k = i - r * F;
        p.g_x_t[(size_t)g * T * F + i] = DHC[r * K3 + k];
    }
    // dW2 = dagg^T . act_sum, db2 = sum_i count_i dagg[i], dasum = dagg . W2
    for (int i = threadIdx.x; i < M * M; i += blockDim.x) {
        const int j = i / M, k = i - j * M;
        float s = 0.f;
        for (int r = 0; r < T; ++r) s = fmaf(DHC[r * K3 + F + j], p.act_sum[((size_t)g * T + r) * M + k], s);
        gp[tail_off_w2(F) + i] = s;
    }
    for (int j = threadIdx.x; j < M; j += blockDim.x) {
        float s = 0.f;
        for (int r = 0; r < T; ++r) s = fmaf(class_count(p, r), DHC[r * K3 + F + j], s);
        gp[tail_off_b2(F) + j] = s;
    }
    for (int i = threadIdx.x; i < T * M; i += blockDim.x) {
        const int r = i / M, k = i - r * M;
        float s = 0.f;
        for (int j = 0; j < M; ++j) s = fmaf(DHC[r * K3 + F + j], p.w2[j * M + k], s);
        p.dasum[(size_t)g * T * M + i] = s;
    }
}

// ------------------------------------------------------------------------------------------
// backward edge pass: dht = dasum[tgt] * lrelu'(ht); g_x_e = W1_e^T dht; fibre sums dRs; dW1_e
// ------------------------------------------------------------------------------------------
struct TargetEdgeBwdParams {
    Topo tp;
    const float *xe2, *Rs, *w1;
    const float* dasum;     // [G,T,2F]
    float* g_x_e;           // [G,E,F]
    const float* g_add;     // optional [G,E,F] added to g_x_e on store (gradient of x_e from its other consumers)
    float* dRs;             // [G,S,2F]
    float* wpartial;        // [ncta][pstride]: dW1_e [2F*F]
    int pstride;
    float* dRs_split;       // split tiles: [G,nslots,2F] partial fibre sums (k_split_sums -> dRs)
};

template <int F>
struct TargetEdgeBwdSmem {
    static constexpr int M = 2 * F, LDM = M + 4, LDF = F + 2;
    using AccW1 = OuterAcc<M, F, 4, F / 2>;
    static constexpr int kTiles = kTile * (LDM + LDF);
    // the tile region doubles as the cross-group scratch of the weight-gradient flush
    static constexpr int kRegion = kTiles > AccW1::kScratchFloats ? kTiles : AccW1::kScratchFloats;
    static constexpr int kFloats = kRegion;   // the weights live in the constant bank (MsgEdgeConst)
    static constexpr size_t bytes = sizeof(float) * kFloats;
};

template <int F, bool SPLIT = false>
__global__ void __launch_bounds__(kThreads) k_target_edge_bwd(const TargetEdgeBwdParams p) {
    using SM = TargetEdgeBwdSmem<F>;
    constexpr int M = 2 * F, LDM = SM::LDM, LDF = SM::LDF;
    extern __shared__ __align__(16) float sm[];
    using CW = MsgEdgeConst<F>;
    float* DHT = sm;               // [kTile][LDM]
    float* XE = DHT + kTile * LDM; // [kTile][LDF]
    using AccW1 = typename SM::AccW1;
    AccW1 accw1;
    accw1.init();
    const Topo& tp = p.tp;
    const int total = tp.ntiles * tp.G;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const Tile t = get_tile<SPLIT>(tp, tile);
        if (threadIdx.x == 0 && tile + (int)gridDim.x < total && tp.layout == PFS_LAYOUT_DENSE) {   // next tile -> L2
            const Tile tn = get_tile<SPLIT>(tp, tile + gridDim.x);
            const size_t off = ((size_t)tn.g * tp.E + tn.q0) * F, bytes = (size_t)tn.ne * F * sizeof(float);
            bulk_prefetch_l2(p.xe2 + off, bytes);
            if (p.g_add) bulk_prefetch_l2(p.g_add + off, bytes);
            bulk_prefetch_l2(p.Rs + ((size_t)tn.g * tp.S + tn.fibre0) * M, (size_t)tn.nfib * M * sizeof(float));
        }
        if (threadIdx.x < t.ne) {
            const EdgeRef er = get_edge(tp, t, threadIdx.x);
            const size_t row = ((size_t)t.g * tp.E + er.e) * F;
            float x[F], h[M], d[M];
            load_row<F>(p.xe2 + row, x);
            load_row<M>(p.Rs + ((size_t)t.g * tp.S + er.src) * M, h);
            dense_acc_c<F, M, CW::kW1t>(x, h);
            load_row<M>(p.dasum + ((size_t)t.g * tp.T + er.tgt) * M, d);
#pragma unroll
            for (int j = 0; j < M; ++j) d[j] *= dlrelu(h[j]);
            store_row_smem<M>(DHT + threadIdx.x * LDM, d);
            store_row_smem<F>(XE + threadIdx.x * LDF, x);
            float dx[F];
#pragma unroll
            for (int k = 0; k < F; ++k) dx[k] = 0.f;
            dense_acc_c<M, F, CW::kW1o>(d, dx);
            if (p.g_add) add_row<F>(p.g_add + row, dx);
            store_row<F>(p.g_x_e + row, dx);
        }
        __syncthreads();
        accw1.accumulate(DHT, LDM, XE, LDF, t.ne);
        tile_fibre_sums<M, LDM, 0, kThreads, SPLIT>(tp, t, DHT, fibre_sum_row<SPLIT>(tp, t, p.dRs, p.dRs_split, M));
        __syncthreads();
    }
    accw1.flush(DHT, p.wpartial + (size_t)blockIdx.x * p.pstride, F, 0);
}

// ------------------------------------------------------------------------------------------
// GlobalModel, one CTA per graph (reference src/gnn.py:195-223; RMSNorm applied twice)
// ------------------------------------------------------------------------------------------
struct GlobalParams {
    int G, F, S, T, normed;
    float rms_eps;
    const float *x_s, *x_t, *u;
    const float *w1, *b1, *w2, *b2, *rms_w;
    float* u_out;
    const float* gout;
    float *g_x_s, *g_x_t, *g_u;
    float* gpartial;   // [G][global_partial_floats(F)]
};
__host__ __device__ constexpr int glob_off_w1(int F) { return 0; }                        // [3F,3F]
__host__ __device__ constexpr int glob_off_b1(int F) { return 9 * F * F; }                // [3F]
__host__ __device__ constexpr int glob_off_w2(int F) { return 9 * F * F + 3 * F; }        // [F,3F]
__host__ __device__ constexpr int glob_off_b2(int F) { return 12 * F * F + 3 * F; }       // [F]
__host__ __device__ constexpr int glob_off_rms(int F) { return 12 * F * F + 4 * F; }      // [F]
__host__ __device__ constexpr int global_partial_floats(int F) { return 12 * F * F + 5 * F; }

// column means of x [rows, F] of graph g into out[0..F) (fixed order); blockDim.x threads.
// thread = (row lane, feature): consecutive threads read consecutive addresses, one pass over the rows
// (a single large graph has 1e5 rows here); scratch: blockDim.x floats
__device__ __forceinline__ void column_means(const float* x, int rows, int F, float* scratch, float* out) {
    const int lanes = blockDim.x / F;
    const int lr = threadIdx.x / F, f = threadIdx.x - lr * F;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (lr < lanes) {
        int r = lr;
        for (; r + 3 * lanes < rows; r += 4 * lanes) {      // four loads in flight per thread
            s0 += x[(size_t)r * F + f];
            s1 += x[(size_t)(r + lanes) * F + f];
            s2 += x[(size_t)(r + 2 * lanes) * F + f];
            s3 += x[(size_t)(r + 3 * lanes) * F + f];
        }
        for (; r < rows; r += lanes) s0 += x[(size_t)r * F + f];
    }
    scratch[threadIdx.x] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (threadIdx.x < F) {
        float s = 0.f;
        for (int i = 0; i < lanes; ++i) s += scratch[i * F + threadIdx.x];
        out[threadIdx.x] = s / (float)rows;
    }
    __syncthreads();
}

// forward core shared with the backward: hc [3F], h [3F] (pre-activation), y [F], o1 [F], r1, r2
__device__ __forceinline__ void global_core(const GlobalParams& p, int g, float* scratch, float* hc, float* h,
                                            float* y, float* o1, float* o2, float* rr) {
    const int F = p.F, K = 3 * F;
    if (threadIdx.x < F) hc[threadIdx.x] = p.u[(size_t)g * F + threadIdx.x];
    column_means(p.x_s + (size_t)g * p.S * F, p.S, F, scratch, hc + F);
    column_means(p.x_t + (size_t)g * p.T * F, p.T, F, scratch, hc + 2 * F);
    if (threadIdx.x < K) {
        float s = p.b1[threadIdx.x];
        for (int k = 0; k < K; ++k) s = fmaf(hc[k], p.w1[threadIdx.x * K + k], s);
        h[threadIdx.x] = s;
    }
    __syncthreads();
    if (threadIdx.x < F) {
        float s = p.b2[threadIdx.x];
        for (int k = 0; k < K; ++k) s = fmaf(lrelu(h[k]), p.w2[threadIdx.x * K + k], s);
        y[threadIdx.x] = s;
    }
    __syncthreads();
    if (p.normed) {
        if (threadIdx.x == 0) {
            float s = 0.f;
            for (int f = 0; f < F; ++f) s = fmaf(y[f], y[f], s);
            rr[0] = rsqrtf(s / (float)F + p.rms_eps);
        }
        __syncthreads();
        if (threadIdx.x < F) o1[threadIdx.x] = y[threadIdx.x] * rr[0] * p.rms_w[threadIdx.x];
        __syncthreads();
        if (threadIdx.x == 0) {
            float s = 0.f;
            for (int f = 0; f < F; ++f) s = fmaf(o1[f], o1[f], s);
            rr[1] = rsqrtf(s / (float)F + p.rms_eps);
        }
        __syncthreads();
        if (threadIdx.x < F) o2[threadIdx.x] = o1[threadIdx.x] * rr[1] * p.rms_w[threadIdx.x];
    } else if (threadIdx.x < F) {
        o2[threadIdx.x] = y[threadIdx.x];
    }
    __syncthreads();
}

// dynamic shared memory: kThreads scratch + 3F + 3F + F + F + F + 2 (+ 3F + F + F in the backward) floats
__global__ void __launch_bounds__(kThreads) k_global_fwd(const GlobalParams p) {
    extern __shared__ __align__(16) float sm[];
    const int F = p.F;
    float* scratch = sm;
    float* hc = scratch + kThreads;
    float* h = hc + 3 * F;
    float* y = h + 3 * F;
    float* o1 = y + F;
    float* o2 = o1 + F;
    float* rr = o2 + F;
    const int g = blockIdx.x;
    global_core(p, g, scratch, hc, h, y, o1, o2, rr);
    if (threadIdx.x < F) p.u_out[(size_t)g * F + threadIdx.x] = o2[threadIdx.x];
}

__global__ void __launch_bounds__(kThreads) k_global_bwd(const GlobalParams p) {
    extern __shared__ __align__(16) float sm[];
    const int F = p.F, K = 3 * F;
    float* scratch = sm;
    float* hc = scratch + kThreads;
    float* h = hc + 3 * F;
    float* y = h + 3 * F;
    float* o1 = y + F;
    float* o2 = o1 + F;
    float* rr = o2 + F;          // 2 floats
    float* dh = rr + 2;          // [3F]
    float* dy = dh + 3 * F;      // [F]
    float* d1 = dy + F;          // [F]
    const int g = blockIdx.x;
    global_core(p, g, scratch, hc, h, y, o1, o2, rr);
    float* gp = p.gpartial + (size_t)g * global_partial_floats(F);
    const float* go = p.gout + (size_t)g * F;
    if (p.normed) {
        // second RMSNorm: input o1, rstd rr[1]; first: input y, rstd rr[0]
        if (threadIdx.x == 0) {
            float s = 0.f;
            for (int f = 0; f < F; ++f) s += go[f] * p.rms_w[f] * o1[f];
            scratch[0] = s / (float)F;
        }
        __syncthreads();
        if (threadIdx.x < F) {
            const int f = threadIdx.x;
            d1[f] = rr[1] * go[f] * p.rms_w[f] - o1[f] * rr[1] * rr[1] * rr[1] * scratch[0];
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            float s = 0.f;
            for (int f = 0; f < F; ++f) s += d1[f] * p.rms_w[f] * y[f];
            scratch[1] = s / (float)F;
        }
        __syncthreads();
        if (threadIdx.x < F) {
            const int f = threadIdx.x;
            dy[f] = rr[0] * d1[f] * p.rms_w[f] - y[f] * rr[0] * rr[0] * rr[0] * scratch[1];
            gp[glob_off_rms(F) + f] = go[f] * o1[f] * rr[1] + d1[f] * y[f] * rr[0];
        }
    } else if (threadIdx.x < F) {
        dy[threadIdx.x] = go[threadIdx.x];
        gp[glob_off_rms(F) + threadIdx.x] = 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < F * K; i += blockDim.x) {
        const int f = i / K, k = i - f * K;
        gp[glob_off_w2(F) + i] = dy[f] * lrelu(h[k]);
    }
    if (threadIdx.x < F) gp[glob_off_b2(F) + threadIdx.x] = dy[threadIdx.x];
    if (threadIdx.x < K) {
        float s = 0.f;
        for (int f = 0; f < F; ++f) s = fmaf(dy[f], p.w2[f * K + threadIdx.x], s);
        dh[threadIdx.x] = s * dlrelu(h[threadIdx.x]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < K * K; i += blockDim.x) {
        const int j = i / K, k = i - j * K;
        gp[glob_off_w1(F) + i] = dh[j] * hc[k];
    }
    if (threadIdx.x < K) {
        gp[glob_off_b1(F) + threadIdx.x] = dh[threadIdx.x];
        float s = 0.f;
        for (int j = 0; j < K; ++j) s = fmaf(dh[j], p.w1[j * K + threadIdx.x], s);
        scratch[2 + threadIdx.x] = s;   // dcat
    }
    __syncthreads();
    const float* dcat = scratch + 2;
    if (threadIdx.x < F) p.g_u[(size_t)g * F + threadIdx.x] = dcat[threadIdx.x];
    for (int i = threadIdx.x; i < p.S * F; i += blockDim.x)
        p.g_x_s[(size_t)g * p.S * F + i] = dcat[F + i % F] / (float)p.S;
    for (int i = threadIdx.x; i < p.T * F; i += blockDim.x)
        p.g_x_t[(size_t)g * p.T * F + i] = dcat[2 * F + i % F] / (float)p.T;
}

// ------------------------------------------------------------------------------------------
// time head (reference src/gnn.py:307-312): softplus(MLP(F,F,1)(x_e)) * scale, plus the integer
// times visits = rint(time / hours[tgt]) (round-half-even, like torch.round), time_int = visits * hours
// ------------------------------------------------------------------------------------------
struct HeadParams {
    Topo tp;
    const float* x_e;
    const float *w1, *b1, *w2, *b2;
    float scale;
    const float* hours;
    const long long* edge_tgt;   // [E] class per edge id (general layout)
    float *time, *visits, *time_int;
    const float* g_time;
    float* g_x_e;
    float* wpartial;   // [ncta][pstride]: dW1 [F*F], db1 [F], dW2 [F], db2 [1]
    int pstride;
};

__device__ __forceinline__ float softplus_f(float x) {
    // torch.nn.functional.softplus, beta = 1, threshold = 20
    return x > 20.f ? x : log1pf(expf(x));
}

template <int F>
__global__ void __launch_bounds__(kThreads) k_head_fwd(const HeadParams p) {
    __shared__ __align__(16) float W1t[F * F];
    __shared__ float b1s[F], w2s[F];
    load_w_inmajor<F, F>(W1t, p.w1, F, 0);
    load_vec<F>(b1s, p.b1);
    load_vec<F>(w2s, p.w2);
    __syncthreads();
    const Topo& tp = p.tp;
    const float b2 = __ldg(p.b2);
    const long long N = (long long)tp.G * tp.E;
    for (long long n = (long long)blockIdx.x * kThreads + threadIdx.x; n < N; n += (long long)gridDim.x * kThreads) {
        float x[F], h[F];
        load_row<F>(p.x_e + n * F, x);
#pragma unroll
        for (int j = 0; j < F; ++j) h[j] = b1s[j];
        dense_acc<F, F>(W1t, x, h);
        float s = b2;
#pragma unroll
        for (int j = 0; j < F; ++j) s = fmaf(lrelu(h[j]), w2s[j], s);
        const float tm = softplus_f(s) * p.scale;
        p.time[n] = tm;
        if (p.hours) {
            const int e = (int)(n % tp.E);
            const int tgt = p.edge_tgt ? (int)p.edge_tgt[e] : e % tp.T;
            const float hv = __ldg(p.hours + tgt);
            const float v = rintf(tm / hv);
            if (p.visits) p.visits[n] = v;
            if (p.time_int) p.time_int[n] = v * hv;
        }
    }
}

template <int F>
__global__ void __launch_bounds__(kThreads) k_head_bwd(const HeadParams p) {
    constexpr int LDF = F + 2;
    __shared__ __align__(16) float W1t[F * F];
    __shared__ __align__(16) float W1o[F * F];
    __shared__ float b1s[F], w2s[F];
    using AccW1 = OuterAcc<F, F, 2, F / 2, 0, 128>;
    // one region: the two staging tiles, reused as the flush scratch and the final reduction buffer
    constexpr int kRegion = (2 * kTile * LDF > AccW1::kScratchFloats) ? 2 * kTile * LDF : AccW1::kScratchFloats;
    __shared__ float REGION[kRegion];
    float* DH = REGION;
    float* XE = REGION + kTile * LDF;
    load_w_inmajor<F, F>(W1t, p.w1, F, 0);
    load_w_outmajor<F, F>(W1o, p.w1, F, 0);
    load_vec<F>(b1s, p.b1);
    load_vec<F>(w2s, p.w2);
    __syncthreads();
    AccW1 acc;
    acc.init();
    float dw2[F], db1[F], db2 = 0.f;
#pragma unroll
    for (int j = 0; j < F; ++j) dw2[j] = db1[j] = 0.f;
    const Topo& tp = p.tp;
    const float b2 = __ldg(p.b2);
    const long long N = (long long)tp.G * tp.E;
    const long long ntile = (N + kTile - 1) / kTile;
    for (long long tile = blockIdx.x; tile < ntile; tile += gridDim.x) {
        const long long n = tile * kTile + threadIdx.x;
        const int rows = (int)min((long long)kTile, N - tile * kTile);
        if (n < N) {
            float x[F], h[F], dh[F];
            load_row<F>(p.x_e + n * F, x);
#pragma unroll
            for (int j = 0; j < F; ++j) h[j] = b1s[j];
            dense_acc<F, F>(W1t, x, h);
            float s = b2;
#pragma unroll
            for (int j = 0; j < F; ++j) s = fmaf(lrelu(h[j]), w2s[j], s);
            // d softplus = sigmoid(s) (1 above the threshold)
            const float sg = s > 20.f ? 1.f : 1.f / (1.f + expf(-s));
            const float ds = __ldg(p.g_time + n) * p.scale * sg;
            db2 += ds;
#pragma unroll
            for (int j = 0; j < F; ++j) {
                dw2[j] = fmaf(ds, lrelu(h[j]), dw2[j]);
                dh[j] = ds * w2s[j] * dlrelu(h[j]);
                db1[j] += dh[j];
            }
            store_row_smem<F>(DH + threadIdx.x * LDF, dh);
            store_row_smem<F>(XE + threadIdx.x * LDF, x);
            float dx[F];
#pragma unroll
            for (int k = 0; k < F; ++k) dx[k] = 0.f;
            dense_acc<F, F>(W1o, dh, dx);
            store_row<F>(p.g_x_e + n * F, dx);
        }
        __syncthreads();
        acc.accumulate(DH, LDF, XE, LDF, rows);
        __syncthreads();
    }
    float* out = p.wpartial + (size_t)blockIdx.x * p.pstride;
    acc.flush(DH, out, F, 0);
    // block-reduce the per-thread vectors: db1 [F], dW2 [F], db2
    {
        float* red = DH;   // [kWarps][2F+1]
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
        for (int j = 0; j < F; ++j) {
            const float a = warp_sum(db1[j]);
            const float b = warp_sum(dw2[j]);
            if (lane == 0) {
                red[w * (2 * F + 1) + j] = a;
                red[w * (2 * F + 1) + F + j] = b;
            }
        }
        const float c = warp_sum(db2);
        if (lane == 0) red[w * (2 * F + 1) + 2 * F] = c;
        __syncthreads();
        if (threadIdx.x < 2 * F + 1) {
            float s = 0.f;
            for (int i = 0; i < kWarps; ++i) s += red[i * (2 * F + 1) + threadIdx.x];
            out[F * F + threadIdx.x] = s;
        }
    }
}

}  // namespace pfs
