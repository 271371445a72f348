// loss.cu -- the training loss that follows the message-passing path (reference src/train.py:21-80;
// SURVEY.md section 8f row N1): softfloor, class / fibre sums, completeness, penalties, variance and the
// gradient w.r.t. the edge times, as five small kernels instead of ~45 ATen ops and two torch_scatter
// calls.  fp32, dense canonical edge order (the reference reshapes the times to [NFIBERS, NCLASSES],
// src/train.py:67), deterministic: every reduction has a fixed order.
//
// A leading graph dimension G batches independent graphs of the same S x T: graph g's rows start at g*S*T (edges),
// g*S (fibres), g*T (classes).  Every graph is reduced by the same code in the same order as a single-graph call
// (the row-block count depends on S alone), so graph g's results are bitwise those of a call on graph g by itself,
// and the launch count does not depend on G.
//
// One graph sharded over fibre ranges (DESIGN.md section 8b): each shard runs the same edge, fibre and class-partial kernels
// on its own fibres, then k_loss_shard_record reduces them to a record of 2 + 3T doubles (local fibre count and fibre
// penalty, per class sum of galaxies, mean and M2 of time2).  The caller exchanges the records, and k_loss_shard_merge
// combines them in rank order and runs the same tail as k_loss_scalars on the global totals.  The backward is the one-graph
// kernel with the variance taken over S_total fibres.
#include <cstdarg>
#include <cstdio>
#include <math_constants.h>

#include <cuda_runtime.h>

#include "../../include/pfs_b200.h"

namespace pfs_host {
int fail_msg(int code, const char* msg);
void mark_launch(const char* name, cudaStream_t st);
int sm_count();
}  // namespace pfs_host

namespace {

int lfail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    return pfs_host::fail_msg(code, buf);
}
#define L_REQUIRE(cond, msg)                                         \
    do {                                                             \
        if (!(cond)) return lfail(PFS_ERR_ARG, "%s (%s)", msg, #cond); \
    } while (0)
#define L_LAUNCH_CHECK(name)                                                                           \
    do {                                                                                              \
        cudaError_t e__ = cudaGetLastError();                                                         \
        if (e__ != cudaSuccess) return lfail(PFS_ERR_CUDA, "launch %s: %s", name, cudaGetErrorString(e__)); \
        pfs_host::mark_launch(name, st);                                                              \
    } while (0)

struct LossConst {
    int S, T, G;
    int class_stride;     // T: hours / counts are [G, T] tables; 0: one [T] table shared by every graph
    float total_time, wutils, wvar, pclass, pfiber, noiselevel;
    float r, atan_r;      // r = exp(-1 / sharpness) (0 when sharpness == 0), atan(r / (1 - r))
    const float* sharp_dev;   // optional device scalar overriding the sharpness (CUDA-graph replays with a schedule)
};
__device__ __forceinline__ void resolve_sharpness(LossConst& c) {
    if (c.sharp_dev) {
        const float sh = *c.sharp_dev;
        c.r = sh == 0.f ? 0.f : expf(-1.f / sh);
        c.atan_r = atanf(c.r / (1.f - c.r));
    }
}

// softfloor (reference src/train.py:21-27) of the noisy visit count and its derivative
__device__ __forceinline__ void softfloor_eval(float visited, float u, const LossConst& c, float& sf, float& dsf) {
    const float x = visited + c.noiselevel * (u - 0.5f);
    float sn, cs;
    sincosf(2.f * CUDART_PI_F * x, &sn, &cs);
    const float den = 1.f - c.r * cs;
    sf = x + (atanf(c.r * sn / den) - c.atan_r) * (1.f / CUDART_PI_F);
    dsf = 1.f + 2.f * c.r * (cs - c.r) / (1.f - 2.f * c.r * cs + c.r * c.r);
}

// edge e of the batch = row `row` (= g*S + k, the fibre over all graphs) and class i; g is only divided out when
// there is more than one graph
struct EdgeAt {
    long long row;
    int i, g;
};
__device__ __forceinline__ EdgeAt edge_at(long long e, const LossConst& c) {
    EdgeAt a;
    a.row = e / c.T;
    a.i = (int)(e - a.row * c.T);
    a.g = c.G > 1 ? (int)(a.row / c.S) : 0;
    return a;
}

// per edge: galaxies = max(0, softfloor(time / T_i)), time2 = galaxies * T_i      (src/train.py:43-49)
__global__ void __launch_bounds__(256) k_loss_edge_fwd(LossConst c, const float* __restrict__ time,
                                                       const float* __restrict__ noise, const float* __restrict__ hours,
                                                       float* __restrict__ galaxies, float* __restrict__ time2) {
    resolve_sharpness(c);
    const long long E = (long long)c.G * c.S * c.T;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
        const EdgeAt a = edge_at(e, c);
        const float h = hours[(size_t)a.g * c.class_stride + a.i];
        float sf, dsf;
        softfloor_eval(time[e] / h, noise[e], c, sf, dsf);
        const float g = fmaxf(sf, 0.f);
        galaxies[e] = g;
        time2[e] = g * h;
    }
}

// fibre sums of time2 (src/train.py:61): one warp per fibre, GS = G*S fibres over all graphs
__global__ void __launch_bounds__(256) k_loss_fibre_sums(long long GS, int T, const float* __restrict__ time2,
                                                         float* __restrict__ fibre_time) {
    const long long k = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (k >= GS) return;
    float s = 0.f;
    for (int i = lane; i < T; i += 32) s += time2[(size_t)k * T + i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) fibre_time[k] = s;
}

// class statistics over the fibres: partial[rb][0][i] = sum galaxies, [1] = sum (time2 - shift_i), [2] = sum (time2 - shift_i)^2,
// shift_i = time2 of fibre 0 (shifted sums do not cancel).  grid = nrb row blocks x G graphs, flattened into x
// (block = g * nrb + row block, so any G fits the grid), 256 threads = (row lane, class); partial is [G][nrb][3][T]
__global__ void __launch_bounds__(256) k_loss_class_partial(int S, int T, int nrb, const float* __restrict__ galaxies,
                                                            const float* __restrict__ time2, int rows_per_block,
                                                            float* __restrict__ partial) {
    __shared__ float red[3][256];
    const int g = blockIdx.x / nrb, rb = blockIdx.x - g * nrb;
    galaxies += (size_t)g * S * T;
    time2 += (size_t)g * S * T;
    partial += (size_t)g * nrb * 3 * T;
    const int tc = T < 256 ? T : 256;
    const int lanes = 256 / tc;
    const int lr = threadIdx.x / tc, lc = threadIdx.x - lr * tc;
    const int r0 = rb * rows_per_block, r1 = min(S, r0 + rows_per_block);
    for (int c0 = 0; c0 < T; c0 += tc) {
        const int i = c0 + lc;
        float a = 0.f, b = 0.f, q = 0.f;
        if (lr < lanes && i < T) {
            const float shift = time2[i];
            for (int k = r0 + lr; k < r1; k += lanes) {
                const size_t e = (size_t)k * T + i;
                a += galaxies[e];
                const float d = time2[e] - shift;
                b += d;
                q = fmaf(d, d, q);
            }
        }
        __syncthreads();
        red[0][threadIdx.x] = a; red[1][threadIdx.x] = b; red[2][threadIdx.x] = q;
        __syncthreads();
        if (lr == 0 && i < T) {
            float s0 = 0.f, s1 = 0.f, s2 = 0.f;
            for (int r = 0; r < lanes; ++r) {
                s0 += red[0][r * tc + lc]; s1 += red[1][r * tc + lc]; s2 += red[2][r * tc + lc];
            }
            float* o = partial + (size_t)rb * 3 * T;
            o[i] = s0; o[T + i] = s1; o[2 * T + i] = s2;
        }
    }
}

__device__ __forceinline__ double block_sum(double v, double* red) {     // fixed tree, blockDim.x == 1024
    red[threadIdx.x] = v;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    const double r = red[0];
    __syncthreads();
    return r;
}

// class i's totals over the fibres of graph g from its row blocks [g nrb, (g + 1) nrb) of `partial`, in row-block order:
// s0 = sum galaxies, mean and m2 (sum of squared deviations, unclamped) of time2, from the sums shifted by time2 of fibre 0
__device__ __forceinline__ void class_totals(const float* __restrict__ partial, int g, int nrb, int S, int T,
                                             const float* __restrict__ time2, int i, double& s0, double& mean, double& m2) {
    double s1 = 0.0, s2 = 0.0;
    s0 = 0.0;
    for (int b = g * nrb; b < (g + 1) * nrb; ++b) {
        s0 += partial[(size_t)b * 3 * T + i];
        s1 += partial[(size_t)b * 3 * T + T + i];
        s2 += partial[(size_t)b * 3 * T + 2 * T + i];
    }
    const double n = (double)S;
    mean = (double)time2[i] + s1 / n;
    m2 = s2 - s1 * s1 / n;
}

// sum over the graph's S fibres of lrelu_0.1(fibre_time - total_time)^2 (src/train.py:63): strided, then the fixed tree
__device__ __forceinline__ double fibre_penalty_sum(const LossConst& c, const float* __restrict__ fibre_time, double* red) {
    double fpen = 0.0;
    for (int k = threadIdx.x; k < c.S; k += blockDim.x) {
        const double ot = (double)fibre_time[k] - (double)c.total_time;
        const double l = ot > 0.0 ? ot : 0.1 * ot;                     // nn.LeakyReLU(0.1), src/train.py:63
        fpen += l * l;
    }
    return block_sum(fpen, red);
}

// Everything that follows the per-class totals, for one graph and one CTA of 1024 threads (src/train.py:51-71): n'_i, the
// class means, completeness and its minimum, penalties, variance, loss and the per-class gradient coefficient dL/dn'_i.
// totals(i, s0, mean, m2) gives class i's totals over all n fibres; fibre_penalty() the fibre-penalty sum (called by every
// thread, at the same point of the sequence).  scalars = {loss, totutils, class_penalty, fibre_penalty, variance, #minima}
template <class Totals, class FibrePenalty>
__device__ __forceinline__ void loss_tail(const LossConst& c, double n, const Totals& totals, const FibrePenalty& fibre_penalty,
                                          const float* __restrict__ counts, float* __restrict__ n_prime,
                                          float* __restrict__ class_mean, float* __restrict__ class_coef,
                                          float* __restrict__ scalars, double* red, float* s_min) {
    const int T = c.T;
    double var_sum = 0.0, cpen = 0.0;
    float my_min = CUDART_INF_F;
    for (int i = threadIdx.x; i < T; i += blockDim.x) {
        double s0, mean, m2;
        totals(i, s0, mean, m2);
        n_prime[i] = (float)s0;
        class_mean[i] = (float)mean;
        var_sum += (m2 > 0.0 ? m2 : 0.0) / (n - 1.0);                 // torch.var: unbiased
        const double over = s0 - (double)counts[i];
        if (over > 0.0) cpen += over * over;
        my_min = fminf(my_min, (float)s0 / counts[i]);
    }
    // minimum completeness and the number of classes attaining it (torch.min spreads the gradient evenly over ties)
    red[threadIdx.x] = (double)my_min;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] = fmin(red[threadIdx.x], red[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) *s_min = (float)red[0];
    __syncthreads();
    const float cmin = *s_min;
    double ties = 0.0;
    for (int i = threadIdx.x; i < T; i += blockDim.x)
        if (n_prime[i] / counts[i] == cmin) ties += 1.0;
    ties = block_sum(ties, red);
    var_sum = block_sum(var_sum, red);
    cpen = block_sum(cpen, red);
    const double fpen = fibre_penalty();
    for (int i = threadIdx.x; i < T; i += blockDim.x) {
        const float np = n_prime[i], N = counts[i];
        float coef = 2.f * c.pclass * fmaxf(np - N, 0.f);
        if (np / N == cmin) coef -= c.wutils / ((float)ties * N);
        class_coef[i] = coef;
    }
    if (threadIdx.x == 0) {
        const double class_penalty = c.pclass * cpen, fibre_penalty = c.pfiber * fpen;
        scalars[0] = (float)(-(double)c.wutils * cmin + fibre_penalty + class_penalty - (double)c.wvar * var_sum);
        scalars[1] = cmin;
        scalars[2] = (float)class_penalty;
        scalars[3] = (float)fibre_penalty;
        scalars[4] = (float)var_sum;
        scalars[5] = (float)ties;
    }
}

// one CTA per graph: the graph's class totals from its row blocks, then the loss tail
__global__ void __launch_bounds__(1024) k_loss_scalars(const LossConst c, const float* __restrict__ partial, int nrb,
                                                       const float* __restrict__ counts, const float* __restrict__ time2,
                                                       const float* __restrict__ fibre_time, float* __restrict__ n_prime,
                                                       float* __restrict__ class_mean, float* __restrict__ class_coef,
                                                       float* __restrict__ scalars) {
    __shared__ double red[1024];
    __shared__ float s_min;
    const int S = c.S, T = c.T;
    // graph blockIdx.x's rows (its row blocks of `partial` are indexed from the global row-block number: a pointer
    // offset there makes the unrolled loop spill at the 64 registers of a 1024-thread CTA)
    const size_t g = blockIdx.x;
    counts += g * c.class_stride;
    time2 += g * S * T;
    fibre_time += g * S;
    n_prime += g * T;
    class_mean += g * T;
    class_coef += g * T;
    scalars += g * 8;
    loss_tail(c, (double)S,
              [&](int i, double& s0, double& mean, double& m2) {
                  class_totals(partial, blockIdx.x, nrb, S, T, time2, i, s0, mean, m2);
              },
              [&] { return fibre_penalty_sum(c, fibre_time, red); },
              counts, n_prime, class_mean, class_coef, scalars, red, &s_min);
}

// Sharded loss, phase 1 (one graph, one CTA): this shard's record [2 + 3T] doubles = {n_r (local fibres), local fibre-penalty
// sum, per class: sum galaxies [T], mean of time2 [T], M2 of time2 [T]}, reduced in the order of k_loss_scalars
__global__ void __launch_bounds__(1024) k_loss_shard_record(const LossConst c, const float* __restrict__ partial, int nrb,
                                                            const float* __restrict__ time2,
                                                            const float* __restrict__ fibre_time, double* __restrict__ record) {
    __shared__ double red[1024];
    const int S = c.S, T = c.T;
    // graph blockIdx.x = 0 (one CTA), indexed as k_loss_scalars indexes it: with a constant 0 the unrolled loop spills
    for (int i = threadIdx.x; i < T; i += blockDim.x) {
        double s0, mean, m2;
        class_totals(partial, blockIdx.x, nrb, S, T, time2, i, s0, mean, m2);
        record[2 + i] = s0;
        record[2 + T + i] = mean;
        record[2 + 2 * T + i] = m2;
    }
    const double fpen = fibre_penalty_sum(c, fibre_time, red);
    if (threadIdx.x == 0) {
        record[0] = (double)S;
        record[1] = fpen;
    }
}

// Sharded loss, phase 2 (one CTA): the records [world][2 + 3T] of every shard combined in rank order -- sums added, (n, mean,
// M2) by the pairwise update (Chan et al.) -- then the loss tail over the S_total fibres.  Every rank reads the same records
// in the same order, so every rank writes bitwise the same results; with one rank they are those of k_loss_scalars.
__global__ void __launch_bounds__(1024) k_loss_shard_merge(const LossConst c, int S_total, int world,
                                                           const double* __restrict__ records, const float* __restrict__ counts,
                                                           float* __restrict__ n_prime, float* __restrict__ class_mean,
                                                           float* __restrict__ class_coef, float* __restrict__ scalars) {
    __shared__ double red[1024];
    __shared__ float s_min;
    const int T = c.T;
    const size_t R = 2 + 3 * (size_t)T;
    loss_tail(c, (double)S_total,
              [&](int i, double& s0, double& mean, double& m2) {
                  double n = records[0];
                  s0 = records[2 + i];
                  mean = records[2 + T + i];
                  m2 = records[2 + 2 * T + i];
#pragma unroll 1
                  for (int r = 1; r < world; ++r) {
                      const double* rec = records + r * R;
                      const double nb = rec[0], nab = n + nb, d = rec[2 + T + i] - mean;
                      s0 += rec[2 + i];
                      mean += d * nb / nab;
                      m2 = m2 + rec[2 + 2 * T + i] + d * d * n * nb / nab;
                      n = nab;
                  }
              },
              [&] {
                  double fpen = records[1];
                  for (int r = 1; r < world; ++r) fpen += records[r * R + 1];
                  return fpen;
              },
              counts, n_prime, class_mean, class_coef, scalars, red, &s_min);
}

// g_time[e] = gL_g * [softfloor > 0] * softfloor' / T_i * (dL/dn'_i + T_i * (dL/dfibre_time_k - 2 wvar (time2 - mean_i) / (S_var - 1)))
// S_var: the fibres the variance runs over (S, or S_total of a sharded graph)
__global__ void __launch_bounds__(256) k_loss_edge_bwd(LossConst c, int S_var, const float* __restrict__ time,
                                                       const float* __restrict__ noise, const float* __restrict__ hours,
                                                       const float* __restrict__ time2, const float* __restrict__ fibre_time,
                                                       const float* __restrict__ class_mean, const float* __restrict__ class_coef,
                                                       const float* __restrict__ g_loss, float* __restrict__ g_time) {
    resolve_sharpness(c);
    const long long E = (long long)c.G * c.S * c.T;
    const float vscale = 2.f * c.wvar / (float)(S_var - 1);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
        const EdgeAt a = edge_at(e, c);
        const size_t ci = (size_t)a.g * c.T + a.i;
        const float h = hours[(size_t)a.g * c.class_stride + a.i];
        float sf, dsf;
        softfloor_eval(time[e] / h, noise[e], c, sf, dsf);
        float g = 0.f;
        if (sf > 0.f) {
            const float gl = g_loss ? g_loss[a.g] : 1.f;
            const float ot = fibre_time[a.row] - c.total_time;
            const float dft = 2.f * c.pfiber * (ot > 0.f ? ot : 0.01f * ot);      // d/d ot of lrelu_0.1(ot)^2
            const float d_t2 = dft - vscale * (time2[e] - class_mean[ci]);
            g = gl * (class_coef[ci] + h * d_t2) * dsf / h;
        }
        g_time[e] = g;
    }
}

int make_const(const pfs_loss_args& a, LossConst& c) {
    if (a.S_total) {         // one shard of a graph: the graph needs 2 fibres, the shard 1
        L_REQUIRE(a.S >= 1 && a.S_total >= 2 && a.S <= a.S_total && a.T >= 1 && (long long)a.S * a.T < (1ll << 31),
                  "loss: bad shard sizes (at least 1 local fibre, 2 over all shards)");
        L_REQUIRE(a.G == 0 || a.G == 1, "loss: a sharded graph is one graph per call (G 0 or 1)");
    } else {
        L_REQUIRE(a.S >= 2 && a.T >= 1 && (long long)a.S * a.T < (1ll << 31), "loss: bad graph sizes (at least 2 fibres)");
    }
    L_REQUIRE(a.G >= 0, "loss: negative graph count");
    L_REQUIRE(a.class_tables == 0 || a.class_tables == 1, "loss: class_tables is 0 (one [T] table) or 1 ([G, T])");
    c.S = a.S; c.T = a.T;
    c.G = a.G > 1 ? a.G : 1;
    c.class_stride = a.class_tables ? a.T : 0;
    c.total_time = a.total_time; c.wutils = a.wutils; c.wvar = a.wvar; c.pclass = a.pclass; c.pfiber = a.pfiber;
    c.noiselevel = a.noiselevel;
    c.r = a.sharpness == 0.f ? 0.f : expf(-1.f / a.sharpness);
    c.atan_r = atanf(c.r / (1.f - c.r));
    c.sharp_dev = a.sharpness_dev;
    return PFS_OK;
}
int class_row_blocks(int S) {
    int nrb = (S + 255) / 256;
    const int cap = 4 * pfs_host::sm_count();
    return nrb > cap ? cap : (nrb < 1 ? 1 : nrb);
}
int edge_grid(long long E) {
    long long b = (E + 255) / 256;
    const long long cap = 8LL * pfs_host::sm_count();
    return (int)(b > cap ? cap : (b < 1 ? 1 : b));
}

// the edge pass, the fibre sums and the class partials of pfs_loss_fwd / pfs_loss_shard_fwd; the partials go to *partial
int loss_edges_and_partials(const pfs_loss_args* a, const LossConst& c, cudaStream_t st, int nrb, float** partial) {
    L_REQUIRE((long long)nrb * c.G < (1ll << 31), "loss: too many graphs for one launch");
    if (a->workspace_bytes < (size_t)c.G * nrb * 3 * c.T * sizeof(float))
        return lfail(PFS_ERR_WORKSPACE, "loss: workspace too small (%zu bytes for %d graph(s))", a->workspace_bytes, c.G);
    *partial = (float*)(((uintptr_t)a->workspace + 255) & ~(uintptr_t)255);
    const long long GS = (long long)c.G * c.S;
    k_loss_edge_fwd<<<edge_grid(GS * c.T), 256, 0, st>>>(c, a->time, a->noise, a->hours, a->galaxies, a->time2);
    L_LAUNCH_CHECK("k_loss_edge_fwd");
    k_loss_fibre_sums<<<(unsigned)((GS * 32 + 255) / 256), 256, 0, st>>>(GS, c.T, a->time2, a->fibre_time);
    L_LAUNCH_CHECK("k_loss_fibre_sums");
    const int rpb = (c.S + nrb - 1) / nrb;
    k_loss_class_partial<<<nrb * c.G, 256, 0, st>>>(c.S, c.T, nrb, a->galaxies, a->time2, rpb, *partial);
    L_LAUNCH_CHECK("k_loss_class_partial");
    return PFS_OK;
}

}  // namespace

extern "C" {

size_t pfs_sizeof_loss_args(void) { return sizeof(pfs_loss_args); }
size_t pfs_loss_workspace_bytes(int32_t S, int32_t T) { return (size_t)class_row_blocks(S) * 3 * T * sizeof(float) + 256; }


int pfs_loss_fwd(const pfs_loss_args* a) {
    L_REQUIRE(a && a->time && a->noise && a->hours && a->counts && a->galaxies && a->time2 && a->fibre_time && a->n_prime &&
                  a->class_mean && a->class_coef && a->scalars && a->workspace, "null pointer");
    L_REQUIRE(a->S_total == 0, "pfs_loss_fwd: S_total is set; a sharded graph runs pfs_loss_shard_fwd and pfs_loss_shard_merge");
    LossConst c;
    if (int rc = make_const(*a, c)) return rc;
    cudaStream_t st = (cudaStream_t)a->stream;
    pfs_host::mark_launch(nullptr, st);
    const int nrb = class_row_blocks(c.S);
    float* partial;
    if (int rc = loss_edges_and_partials(a, c, st, nrb, &partial)) return rc;
    k_loss_scalars<<<c.G, 1024, 0, st>>>(c, partial, nrb, a->counts, a->time2, a->fibre_time, a->n_prime, a->class_mean,
                                         a->class_coef, a->scalars);
    L_LAUNCH_CHECK("k_loss_scalars");
    return PFS_OK;
}

int pfs_loss_shard_fwd(const pfs_loss_args* a) {
    L_REQUIRE(a && a->time && a->noise && a->hours && a->galaxies && a->time2 && a->fibre_time && a->shard_record &&
                  a->workspace, "null pointer");
    L_REQUIRE(a->S_total > 0, "pfs_loss_shard_fwd: S_total (fibres over all shards) is not set");
    LossConst c;
    if (int rc = make_const(*a, c)) return rc;
    cudaStream_t st = (cudaStream_t)a->stream;
    pfs_host::mark_launch(nullptr, st);
    const int nrb = class_row_blocks(c.S);
    float* partial;
    if (int rc = loss_edges_and_partials(a, c, st, nrb, &partial)) return rc;
    k_loss_shard_record<<<1, 1024, 0, st>>>(c, partial, nrb, a->time2, a->fibre_time, a->shard_record);
    L_LAUNCH_CHECK("k_loss_shard_record");
    return PFS_OK;
}

int pfs_loss_shard_merge(const pfs_loss_args* a) {
    L_REQUIRE(a && a->counts && a->n_prime && a->class_mean && a->class_coef && a->scalars && a->shard_records, "null pointer");
    L_REQUIRE(a->S_total > 0, "pfs_loss_shard_merge: S_total (fibres over all shards) is not set");
    L_REQUIRE(a->world >= 1, "pfs_loss_shard_merge: world (ranks, records) is not set");
    LossConst c;
    if (int rc = make_const(*a, c)) return rc;
    cudaStream_t st = (cudaStream_t)a->stream;
    pfs_host::mark_launch(nullptr, st);
    k_loss_shard_merge<<<1, 1024, 0, st>>>(c, a->S_total, a->world, a->shard_records, a->counts, a->n_prime, a->class_mean,
                                           a->class_coef, a->scalars);
    L_LAUNCH_CHECK("k_loss_shard_merge");
    return PFS_OK;
}

int pfs_loss_bwd(const pfs_loss_args* a) {
    L_REQUIRE(a && a->time && a->noise && a->hours && a->time2 && a->fibre_time && a->class_mean && a->class_coef && a->g_time,
              "null pointer");
    LossConst c;
    if (int rc = make_const(*a, c)) return rc;
    cudaStream_t st = (cudaStream_t)a->stream;
    pfs_host::mark_launch(nullptr, st);
    const int S_var = a->S_total ? a->S_total : c.S;
    k_loss_edge_bwd<<<edge_grid((long long)c.G * c.S * c.T), 256, 0, st>>>(c, S_var, a->time, a->noise, a->hours, a->time2,
                                                                    a->fibre_time, a->class_mean, a->class_coef, a->g_loss,
                                                                    a->g_time);
    L_LAUNCH_CHECK("k_loss_edge_bwd");
    return PFS_OK;
}

}  // extern "C"
