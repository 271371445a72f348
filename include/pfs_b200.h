/*
 * pfs_b200.h -- C ABI of libpfs_b200.so: the B200 (sm_100a) message-passing layer.
 *
 * The reference (joshua-lintropic/pfs-neural-net) has no FFI: its boundary for this path is the
 * nn.Module surface of src/gnn.py.  The Python package `pfs-neural-net_b200/gnn.py` mirrors that
 * surface and lowers every module `forward`/`backward` onto the entry points below (ctypes; see
 * INTEGRATION.md for the stub a reference maintainer would add).  Each entry point names the
 * reference code it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated otherwise;
 *   - the caller allocates every output and the workspace (size from pfs_workspace_bytes);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden streams, no
 *     device synchronisation, no host allocation inside a call;
 *   - ONE STREAM AND ONE HOST THREAD PER DEVICE AT A TIME: the module-level entry points stage their
 *     small MLP weights in one per-device __constant__ bank (uploaded on `stream` ahead of the kernels
 *     that read it) and the caller passes one workspace per topology, so calls on the same device
 *     must be serialised on a single stream by a single host thread.  The library checks this
 *     cheaply: a call on a different stream than the previous call on that device first makes the
 *     new stream wait for everything enqueued so far (an event wait, no host sync), so switching
 *     streams between steps is safe; truly concurrent use of two streams is not supported;
 *   - return value 0 = ok, negative = error; pfs_last_error() gives the message (thread local);
 *   - nothing throws across the ABI; there is no CPU fallback: without a CUDA device every
 *     compute entry point returns PFS_ERR_CUDA;
 *   - tensors are row-major and contiguous, fp32; a leading "graph" dimension G batches
 *     independent graphs that share one topology and one set of weights: x_s [G,S,F],
 *     x_t [G,T,F], x_e [G,E,F], u [G,F].  BatchNorm statistics are per graph (the reference
 *     processes one graph per step), running buffers are updated graph by graph in order, and
 *     parameter gradients are summed over the G graphs in a fixed order (deterministic).
 */
#ifndef PFS_B200_H
#define PFS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PFS_ABI_VERSION 11

enum {
    PFS_OK = 0,
    PFS_ERR_ARG = -1,        /* bad argument (null pointer, unsupported F, ...) */
    PFS_ERR_CUDA = -2,       /* CUDA runtime error (message has the cudaGetErrorString) */
    PFS_ERR_UNSUPPORTED = -3,/* valid request this build cannot serve (e.g. an Fdim without kernels) */
    PFS_ERR_WORKSPACE = -4   /* workspace too small */
};

enum { PFS_LAYOUT_DENSE = 0, PFS_LAYOUT_CSR = 1 };

/* edges processed by one CTA tile.  A tile holds whole fibres; a fibre with more edges is split
 * over consecutive tiles of its own (see the split fields of pfs_topology). */
#define PFS_TILE_EDGES 256

/*
 * Topology of the bipartite graph (reference: `edge_index` [2,E] int64, src/gnn.py:98,135,187).
 *   PFS_LAYOUT_DENSE: the canonical complete graph of src/train.py:94, edge e = k*T + i
 *                     (src = e / T, tgt = e % T); no index arrays are read.
 *   PFS_LAYOUT_CSR:   any edge list.  Arrays come from pfs_build_topology (int32, device):
 *                     edges are visited in fibre-sorted ("CSR") order q = 0..E-1.
 */
typedef struct pfs_topology {
    int32_t layout;
    int32_t G;                 /* graphs in the batch (>= 1) */
    int32_t F;                 /* feature width Fdim */
    int32_t S, T, E;           /* fibres, classes, edges (per graph) */
    const int32_t* csr_rowptr; /* [S+1]  first CSR position of each fibre                     */
    const int32_t* csr_eid;    /* [E]    original edge id (row of x_e) at CSR position q      */
    const int32_t* csr_src;    /* [E]    fibre at CSR position q                              */
    const int32_t* csr_tgt;    /* [E]    class at CSR position q                              */
    const int32_t* tile_fibre; /* [ntiles+1] first fibre of every tile (<= PFS_TILE_EDGES edges)           */
    int32_t ntiles;            /* tiles per graph (CSR layout; dense layout derives it)       */
    const int32_t* csc_colptr; /* [T+1]  first CSC position of each class                     */
    const int32_t* csc_q;      /* [E]    CSR position of the k-th class-sorted edge           */
    /* ABI 7: split tiles (from pfs_build_split_tiles, used when a fibre has more than PFS_TILE_EDGES
     * edges).  A split tile holds one chunk [tile_q[i], tile_q[i+1]) of one fibre's edges; its per-fibre
     * results go to a partial-record slot and are combined per fibre in slot order.  All NULL / 0: every
     * tile holds whole fibres (the table of pfs_build_topology). */
    const int32_t* tile_q;     /* [ntiles+1] first CSR position of every tile                 */
    const int32_t* tile_slot;  /* [ntiles]   partial-record slot of a split tile, -1 for whole fibres */
    const int32_t* split_fibre;/* [nsplit]   the split fibres, ascending                      */
    const int32_t* split_ptr;  /* [nsplit+1] slots of split fibre i: [split_ptr[i], split_ptr[i+1]) */
    int32_t nsplit;            /* split fibres                                                 */
    int32_t nslots;            /* partial-record slots (= split tiles) per graph               */
} pfs_topology;

/* -------------------------------------------------------------------------------------------
 * misc
 * ---------------------------------------------------------------------------------------- */
int pfs_abi_version(void);
const char* pfs_last_error(void);
/* 1 if feature width F has compiled kernels in this build, else 0 */
int pfs_supports_fdim(int32_t F);
/* sizeof() of the argument structs, so a binding can check its own layout */
size_t pfs_sizeof_topology(void);
size_t pfs_sizeof_edge_args(void);
size_t pfs_sizeof_source_args(void);
size_t pfs_sizeof_target_args(void);
size_t pfs_sizeof_global_args(void);
size_t pfs_sizeof_head_args(void);

/* Launch accounting and optional per-kernel timing (used by bench.py; not part of the reference
 * surface).  pfs_launch_count: kernels launched by this library so far.  pfs_profile_enable(1)
 * starts recording a CUDA event after every kernel on its launch stream; pfs_profile_report waits
 * for them and writes one line "kernel launches total_ms" per kernel (returns bytes written). */
long long pfs_launch_count(void);
int pfs_profile_enable(int on);
int pfs_profile_report(char* buf, size_t buflen);

/* Workspace (bytes) sufficient for any forward/backward call on this topology. */
size_t pfs_workspace_bytes(const pfs_topology* topo);

/* -------------------------------------------------------------------------------------------
 * topology (replaces the implicit advanced-indexing / torch_scatter index handling of
 * reference src/gnn.py:98-100,135-144,187-190)
 * ---------------------------------------------------------------------------------------- */
/* Writes 1 to *flag_dev (device int32) when edge_index [2,E] int64 is exactly the canonical
 * dense order src = e / T, tgt = e % T with E = S*T, else 0. */
int pfs_detect_dense(const int64_t* edge_index, int64_t E, int32_t S, int32_t T, int32_t* flag_dev, void* stream);

/* Bytes of temporary device storage pfs_build_topology needs. */
size_t pfs_build_topology_temp_bytes(int64_t E, int32_t S, int32_t T);
/* Builds the int32 CSR/CSC arrays (stable counting sort, deterministic).  Outputs (device):
 * csr_rowptr [S+1], csr_eid [E], csr_src [E], csr_tgt [E], csc_colptr [T+1], csc_q [E],
 * tile_fibre [S+1] (capacity), *ntiles_dev and *max_degree_dev (device int32 each). */
int pfs_build_topology(const int64_t* edge_index, int64_t E, int32_t S, int32_t T,
                       int32_t* csr_rowptr, int32_t* csr_eid, int32_t* csr_src, int32_t* csr_tgt,
                       int32_t* csc_colptr, int32_t* csc_q, int32_t* tile_fibre,
                       int32_t* ntiles_dev, int32_t* max_degree_dev,
                       void* temp, size_t temp_bytes, void* stream);
/* Tile table for a topology with fibres of more than PFS_TILE_EDGES edges, over the CSR order of
 * pfs_build_topology.  Whole fibres are packed greedily as pfs_build_topology packs them; a fibre of
 * d > PFS_TILE_EDGES edges gets ceil(d / PFS_TILE_EDGES) consecutive tiles of its own with balanced
 * chunk sizes (sizes differ by at most one, the larger ones first).  Capacities (device int32):
 * tile_fibre, tile_q [S + E/PFS_TILE_EDGES + 2], tile_slot [S + E/PFS_TILE_EDGES + 1], split_fibre [S],
 * split_ptr [S+1]; counts_dev [3] receives ntiles, nsplit and nslots.  Sequential, once per topology. */
int pfs_build_split_tiles(const int32_t* csr_rowptr, int32_t S, int32_t* tile_fibre, int32_t* tile_q,
                          int32_t* tile_slot, int32_t* split_fibre, int32_t* split_ptr, int32_t* counts_dev,
                          void* stream);

/* -------------------------------------------------------------------------------------------
 * EdgeModel  (reference src/gnn.py:73-101: gather + cat + MLP(4F,4F,F) + BatchNorm1d applied twice)
 * ---------------------------------------------------------------------------------------- */
typedef struct pfs_edge_args {
    pfs_topology topo;
    /* inputs */
    const float *x_s, *x_t, *x_e, *u;            /* [G,S,F] [G,T,F] [G,E,F] [G,F] */
    const float *w1, *b1, *w2, *b2;              /* `0.weight` [4F,4F], `0.bias` [4F], `2.weight` [F,4F], `2.bias` [F] */
    const float *gamma, *beta;                   /* `norm.weight/bias` [F]; ignored when normed == 0 */
    float *running_mean, *running_var;           /* `norm.running_*` [F]; updated in place when training */
    int64_t* num_batches_tracked;                /* += 2 per graph when training (double norm)  */
    int32_t training, normed;
    float eps, momentum;
    /* forward outputs */
    float* x_e_out;                              /* [G,E,F] */
    float* bn_save;                              /* [G,4,F]: mean, biased var, combined scale, shift */
    /* backward inputs (x_e_out and bn_save as written by the forward) */
    const float* g_out;                          /* dL/dx_e_out [G,E,F] */
    /* backward outputs (overwritten) */
    float *g_x_s, *g_x_t, *g_x_e, *g_u;          /* [G,S,F] [G,T,F] [G,E,F] [G,F] */
    float *g_w1, *g_b1, *g_w2, *g_b2, *g_gamma, *g_beta;
    void* workspace; size_t workspace_bytes;
    void* stream;
    /* ABI 5 */
    int32_t defer_affine;                        /* forward, normed: x_e_out receives the PRE-norm z and bn_save the per-graph
                                                    (scale, shift); the caller hands bn_save to the next consumer of x_e_out
                                                    (pfs_source_args.x_e_affine), whose edge pass normalises the rows in place
                                                    as it reads them -- one pass over [G,E,F] and one launch less per Block */
    int32_t reserved0;
    float *table_s, *table_t;                    /* optional [G,S,4F], [G,T,4F]: node tables of the first-layer split.  The
                                                    forward writes them here instead of its workspace; a backward given the
                                                    same buffers reads them instead of recomputing them */
} pfs_edge_args;
int pfs_edge_fwd(const pfs_edge_args* a);
int pfs_edge_bwd(const pfs_edge_args* a);

/* -------------------------------------------------------------------------------------------
 * SModel  (reference src/gnn.py:104-154: message MLP(2F,2F,2F), per-fibre mean/std/skew/kurtosis
 * via torch_scatter, node MLP(10F,10F,F), BatchNorm1d over the fibres)
 * ---------------------------------------------------------------------------------------- */
typedef struct pfs_source_args {
    pfs_topology topo;
    const float *x_s, *x_t, *x_e, *u;            /* x_e is the UPDATED edge embedding */
    const float *w1, *b1, *w2, *b2;              /* node_mlp_1: [2F,2F] [2F] [2F,2F] [2F] */
    const float *w3, *b3, *w4, *b4;              /* node_mlp_2: [10F,10F] [10F] [F,10F] [F] */
    const float *gamma, *beta;
    float *running_mean, *running_var;
    int64_t* num_batches_tracked;
    int32_t training, normed;
    float eps, momentum;
    float* x_s_out;                              /* [G,S,F] */
    float* moments;                              /* [G,S,5,2F] saved: mean, E[m^2], c2, c3, c4 */
    float* hidden;                               /* [G,S,10F] saved: lrelu of the node MLP hidden layer */
    float* y_pre;                                /* [G,S,F] saved: node MLP output before the norm */
    float* bn_save;                              /* [G,4,F] */
    const float* g_out;                          /* dL/dx_s_out [G,S,F] */
    const float* g_x_e_add;                      /* optional [G,E,F]: g_x_e = (this module's dL/dx_e) + g_x_e_add, fused into the store */
    float *g_x_s, *g_x_t, *g_x_e, *g_u;
    float *g_w1, *g_b1, *g_w2, *g_b2, *g_w3, *g_b3, *g_w4, *g_b4, *g_gamma, *g_beta;
    void* workspace; size_t workspace_bytes;
    void* stream;
    /* ABI 5 */
    const float* x_e_affine;                     /* optional, forward: bn_save [G,4,F] of a pfs_edge_fwd run with defer_affine;
                                                    x_e then holds the pre-norm z, and the edge pass stores
                                                    x_e' = scale z + shift back into x_e_norm_out as it goes */
    float* x_e_norm_out;                         /* [G,E,F], may alias x_e (every row is read and written by one thread) */
} pfs_source_args;
int pfs_source_fwd(const pfs_source_args* a);
int pfs_source_bwd(const pfs_source_args* a);

/* -------------------------------------------------------------------------------------------
 * TModel  (reference src/gnn.py:157-192: message MLP(2F,2F,2F), scatter-sum over classes,
 * node MLP(4F,4F,F), BatchNorm1d over the classes)
 * ---------------------------------------------------------------------------------------- */
typedef struct pfs_target_args {
    pfs_topology topo;
    const float *x_s, *x_t, *x_e, *u;            /* x_s, x_e are the UPDATED embeddings */
    const float *w1, *b1, *w2, *b2;              /* node_mlp_1 */
    const float *w3, *b3, *w4, *b4;              /* node_mlp_2: [4F,4F] [4F] [F,4F] [F] */
    const float *gamma, *beta;
    float *running_mean, *running_var;
    int64_t* num_batches_tracked;
    int32_t training, normed;
    float eps, momentum;
    float* x_t_out;                              /* [G,T,F] */
    float* act_sum;                              /* [G,T,2F] saved: per-class sum of the hidden activations */
    float* y_pre;                                /* [G,T,F] saved */
    float* bn_save;                              /* [G,4,F] */
    const float* g_out;                          /* dL/dx_t_out [G,T,F] */
    const float* g_x_e_add;                      /* optional [G,E,F]: g_x_e = (this module's dL/dx_e) + g_x_e_add, fused into the store */
    float *g_x_s, *g_x_t, *g_x_e, *g_u;
    float *g_w1, *g_b1, *g_w2, *g_b2, *g_w3, *g_b3, *g_w4, *g_b4, *g_gamma, *g_beta;
    void* workspace; size_t workspace_bytes;
    void* stream;
    /* ABI 5 */
    float* table_s;                              /* optional [G,S,2F]: the fibre table of the first-layer split, written by the
                                                    forward and read back by a backward given the same buffer */
} pfs_target_args;
int pfs_target_fwd(const pfs_target_args* a);
int pfs_target_bwd(const pfs_target_args* a);

/* -------------------------------------------------------------------------------------------
 * GlobalModel  (reference src/gnn.py:195-223: mean-pool, MLP(3F,3F,F), RMSNorm applied twice)
 * ---------------------------------------------------------------------------------------- */
typedef struct pfs_global_args {
    int32_t G, F, S, T;
    const float *x_s, *x_t, *u;                  /* [G,S,F] [G,T,F] [G,F] (updated node embeddings) */
    const float *w1, *b1, *w2, *b2;              /* [3F,3F] [3F] [F,3F] [F] */
    const float* rms_weight;                     /* `norm.weight` [F]; ignored when normed == 0 */
    int32_t normed;
    float rms_eps;                               /* torch.finfo(float32).eps for nn.RMSNorm(eps=None) */
    float* u_out;                                /* [G,F] */
    const float* g_out;                          /* dL/du_out [G,F] */
    float *g_x_s, *g_x_t, *g_u;                  /* [G,S,F] [G,T,F] [G,F] */
    float *g_w1, *g_b1, *g_w2, *g_b2, *g_rms_weight;
    void* workspace; size_t workspace_bytes;
    void* stream;
} pfs_global_args;
int pfs_global_fwd(const pfs_global_args* a);
int pfs_global_bwd(const pfs_global_args* a);

/* -------------------------------------------------------------------------------------------
 * Time head  (reference GNN.edge_prediction, src/gnn.py:307-312: MLP(F,F,1), round (identity,
 * src/gnn.py:321-325), softplus * scale) plus the integer times adopted in DESIGN.md:
 * visits = rint(time / hours[tgt]), time_int = visits * hours[tgt] (src/train.py:257).
 * ---------------------------------------------------------------------------------------- */
typedef struct pfs_head_args {
    pfs_topology topo;
    const float* x_e;                            /* [G,E,F] */
    const float *w1, *b1, *w2, *b2;              /* decoder_e: [F,F] [F] [1,F] [1] */
    float scale;
    const float* class_hours;                    /* [T] hours per visit, or NULL (no integer outputs) */
    const int64_t* edge_tgt;                     /* [E] class of every edge (edge_index[1]); NULL for the dense layout */
    float* time;                                 /* [G,E] */
    float* visits;                               /* [G,E] integer-valued, or NULL */
    float* time_int;                             /* [G,E] or NULL */
    const float* g_time;                         /* dL/dtime [G,E] */
    float* g_x_e;                                /* [G,E,F] */
    float *g_w1, *g_b1, *g_w2, *g_b2;
    void* workspace; size_t workspace_bytes;
    void* stream;
} pfs_head_args;
int pfs_time_head_fwd(const pfs_head_args* a);
int pfs_time_head_bwd(const pfs_head_args* a);

/* -------------------------------------------------------------------------------------------
 * Wide-feature path (Fdim >= 32, bf16 storage, fp32 accumulation and statistics; BASELINE
 * configs C4 / C5b).  At these widths every MLP layer of src/gnn.py:65-71 is a dense contraction
 * and runs on tcgen05 tensor cores; the Python host (`pfs-neural-net_b200/wide.py`) composes the
 * module forward/backward passes of src/gnn.py:73-223 from the primitives below, one graph per
 * call (G = 1).  bf16 tensors are passed as void*; rows are row-major with the stated leading
 * dimension in ELEMENTS; all pointers must be 16-byte aligned and leading dimensions multiples of 8.
 * ---------------------------------------------------------------------------------------- */

/* C[M,N] = epilogue(A[M,K] . B[N,K]^T): one Linear layer (B = torch weight [out,in] or a column
 * slice of it), forward or input-gradient direction (reference src/gnn.py:65-71).  Epilogue, in
 * order: + bias[n] * (bias_rowscale ? bias_rowscale[m] : 1); + tab0[row0(m)][n]; + tab1[row1(m)][n]
 * (row0 = idx0 ? idx0[m] : m / div0, row1 = idx1 ? idx1[m] : m % mod1 -- the gathered first-layer
 * node tables replacing the concatenations of src/gnn.py:100,136,188); LeakyReLU(0.1) if act;
 * * (mask[m][n] > 0 ? 1 : 0.1) if mask (LeakyReLU derivative from the saved activation).
 * Outputs: bf16 [M,ldc] and/or fp32 [M,ldf].  Optional dense-layout operands: see the last fields. */
typedef struct pfs_wide_gemm_args {
    const void* A; int64_t lda;                  /* bf16 [M,K] */
    const void* B; int64_t ldb;                  /* bf16 [N,K] */
    int32_t M, N, K;
    const float* bias;                           /* [N] or NULL */
    const float* bias_rowscale;                  /* [M] or NULL */
    const float* tab0; const int32_t* idx0; int32_t div0;   /* fp32 [*,N] or NULL */
    const float* tab1; const int32_t* idx1; int32_t mod1;   /* fp32 [*,N] or NULL */
    const void* mask; int64_t ldmask;            /* bf16 [M,ldmask] or NULL */
    int32_t act;
    void* out_bf16; int64_t ldc;                 /* or NULL */
    float* out_f32; int64_t ldf;                 /* or NULL */
    void* stream;
    /* dense-layout fast path (canonical order, T % 128 == 0), replacing the gathered tables:
     * K-concatenation C = [A2[m % a2_mod] | A[m]] . B^T with B [N, K2 + K] (x_t[tgt] as a second operand), and
     * per-tile bias rows + bias_rows[m / bias_rows_div][n] (P_s[src] is constant over a 128-row tile) */
    const void* A2; int64_t lda2; int32_t K2; int32_t a2_mod;     /* bf16 [a2_mod, K2] or NULL */
    const float* bias_rows; int32_t bias_rows_div;                /* fp32 [*, N] or NULL */
} pfs_wide_gemm_args;
size_t pfs_sizeof_wide_gemm_args(void);
int pfs_wide_gemm_nt(const pfs_wide_gemm_args* a);

/* W[J, Kx] (+)= D[E,J]^T . X[E,Kx]: a weight gradient, contraction over edges / nodes
 * (autograd of src/gnn.py:65-71).  Split over row ranges, partial sums reduced in a fixed order.
 * out is fp32 with leading dimension ldo; workspace from pfs_wide_gemm_tn_workspace. */
size_t pfs_wide_gemm_tn_workspace(int64_t E, int32_t J, int32_t Kx);
int pfs_wide_gemm_tn(const void* D, int64_t ldd, const void* X, int64_t ldx, int64_t E, int32_t J, int32_t Kx,
                     float* out, int64_t ldo, int32_t accumulate, void* workspace, size_t workspace_bytes,
                     void* stream);

/* Row segments for the segmented reductions that replace torch_scatter (src/gnn.py:140-144,190):
 * mode 0 = dense fibres (rows seg*T + i), 1 = dense classes (rows i*T + seg), 2 = listed rows
 * list[ptr[seg] .. ptr[seg+1]) (list NULL: the positions themselves). */
typedef struct pfs_wide_segments {
    int32_t mode, nseg, S, T;
    const int32_t* ptr;
    const int32_t* list;
} pfs_wide_segments;
size_t pfs_sizeof_wide_segments(void);

/* Column statistics over rows (dtype codes: 0 = bf16, 1 = fp32).
 * kind 0: out[0][c] = mean, out[1][c] = sum of squared deviations of x (BatchNorm forward);
 * kind 1: out[0][c] = sum_r w[r] g[r][c], out[1][c] = sum_r w[r] g[r][c] (v[r][c] - p0[c]) p1[c]
 *         (BatchNorm backward sums, bias gradients; v, p0, p1, w optional). */
size_t pfs_wide_colstats_workspace(int64_t R, int32_t C);
int pfs_wide_colstats(int32_t kind, const void* g, int32_t g_dtype, int64_t ldg, const void* v, int32_t v_dtype,
                      int64_t ldv, const float* p0, const float* p1, const float* roww, int64_t R, int32_t C,
                      float* out, void* workspace, size_t workspace_bytes, void* stream);
/* kind 0: out = a[c] x + b[c];  kind 1: out = a[c] (x - b[c] - (v - p0[c]) p1[c] c2[c])  -> bf16 */
int pfs_wide_rowmap(int32_t kind, const void* x, int32_t x_dtype, int64_t ldx, const void* v, int32_t v_dtype,
                    int64_t ldv, const float* a, const float* b, const float* p0, const float* p1, const float* c2,
                    int64_t R, int32_t C, void* out_bf16, int64_t ldo, void* stream);
/* out[seg][c] = sum of x[row][c] over the segment's rows -> fp32 and/or bf16 [nseg, C] */
size_t pfs_wide_segsum_workspace(const pfs_wide_segments* sd, int32_t C);
int pfs_wide_segsum(const pfs_wide_segments* sd, const void* x, int32_t x_dtype, int64_t ldx, int32_t C, float* out_f32,
                    void* out_bf16, void* workspace, size_t workspace_bytes, void* stream);
/* SModel moment statistics (src/gnn.py:140-151) of the messages m [E,2F] per fibre:
 * moments [S,5,2F] = {mean, E[m^2], c2, c3, c4}; hcat [S,9F] = [x_s|mean|std|skew|kurt] */
int pfs_wide_moments_fwd(const pfs_wide_segments* sd, const void* m, int32_t m_dtype, int32_t C, float* moments, void* stream);
int pfs_wide_source_hcat(const void* x_s_bf16, const float* moments, int32_t S, int32_t F, void* hcat_bf16, int64_t ldo,
                         int32_t with_lo, void* stream);
/* with_lo: rows of 17F columns, [hcat | bf16 remainders of the 8F statistics columns]; contracted against
 * [W3[:, :9F] | W3[:, F:9F]] the fibre MLP sees the statistics to ~2^-17 instead of 2^-9.
 * pfs_wide_split: out[r] = [hi(x[r]) | lo(x[r])] (bf16 [R, 2C]) for any node-level fp32 GEMM operand */
int pfs_wide_split(const float* x, int64_t ldx, int64_t R, int32_t C, void* out_bf16, int64_t ldo, void* stream);
/* backward of the statistics: dh [S,9F] fp32 -> dx_s bf16 [S,F] and cubic coefficients coef [S,4,2F];
 * dm[e] = A0 + A1 m + A2 d^2 + A3 d^3 per edge (src = fibre of every edge, NULL: e / T) */
int pfs_wide_source_coef(const pfs_wide_segments* sd, const float* dh, const float* moments, int32_t S, int32_t F,
                         void* dx_s_bf16, float* coef, void* stream);
int pfs_wide_source_dm(const void* m, int32_t m_dtype, const float* moments, const float* coef, const int32_t* src, int32_t T,
                       int64_t E, int32_t C, void* dm_bf16, void* stream);
/* the same, one CTA per fibre segment (coefficients stay in registers over the fibre's edges) */
int pfs_wide_source_dm_seg(const pfs_wide_segments* fibres, const void* m, int32_t m_dtype, const float* moments,
                           const float* coef, int32_t C, void* dm_bf16, void* stream);
/* out[e] = tab[idx ? idx[e] : e % mod] * (act[e] > 0 ? 1 : 0.1)   (TModel backward, src/gnn.py:188-190) */
int pfs_wide_gather_mask(const float* tab, const int32_t* idx, int32_t mod, const void* act_bf16, int64_t E, int32_t C,
                         void* out_bf16, void* stream);
/* Time head on the wide path (src/gnn.py:307-312): a [E,F] = lrelu(x_e W1^T + b1) from pfs_wide_gemm_nt;
 * pred = a . w2 + b2, time = softplus(pred) * scale; optional integer outputs (NULL to skip):
 * visits = rint(time / class_hours[tgt]), time_int = visits * class_hours[tgt] (tgt NULL: e % T).
 * Backward: gp[e] = g_time[e] sigmoid(pred[e]) scale and da = gp w2 lrelu'(a) (bf16 [E,F]); the weight
 * gradients follow from pfs_wide_colstats (roww = gp) and pfs_wide_gemm_tn / _nt on da. */
int pfs_wide_head_fwd(const void* a_bf16, const float* w2, const float* b2, float scale, int64_t E, int32_t F,
                      const float* class_hours, const int32_t* tgt, int32_t T, float* pred, float* time, float* visits,
                      float* time_int, void* stream);
int pfs_wide_head_bwd(const void* a_bf16, const float* w2, const float* pred, const float* g_time, float scale, int64_t E,
                      int32_t F, float* gp, void* da_bf16, void* stream);
/* dtype conversion (0 = bf16, 1 = fp32) and bf16 transpose out[c][r] = in[r][c] */
int pfs_wide_cast(const void* in, int32_t in_dtype, void* out, int32_t out_dtype, int64_t n, void* stream);
int pfs_wide_transpose(const void* in_bf16, int32_t R, int32_t C, int64_t ld, void* out_bf16, void* stream);

/* -------------------------------------------------------------------------------------------
 * Training loss that consumes the edge times (reference src/train.py:21-80: softfloor + loss_function
 * from `time = gnn.edge_prediction(...)` on; SURVEY.md section 8f row N1).  fp32, dense canonical edge
 * order e = k*T + i (the reference reshapes the times to [NFIBERS, NCLASSES], src/train.py:67), or any edge
 * list (E > 0, ABI 10, below).  `noise`
 * is the uniform [0,1) draw of softfloor (torch.rand_like, src/train.py:22), supplied by the caller so the
 * result is reproducible.
 *   forward : galaxies = max(0, softfloor(time / T_i)), time2 = galaxies T_i, n'_i, fibre times, and
 *             scalars = {loss, totutils (min completeness), class_penalty, fibre_penalty, variance, #minima}
 *   backward: g_time = dloss/dtime * g_loss (g_loss: device vector [G], NULL = 1)
 * Graph dimension (ABI 8): G independent graphs of the same S x T in one call; every per-graph array below
 * gains a leading [G] (G = 0 or 1: one graph, the shapes without it).  S*T < 2^31 per graph; G*S*T may
 * exceed it.  A forward + backward is 5 launches whatever G is.  Graph g's results depend on graph g's
 * inputs alone (not on G or on g's position): a batched call is bitwise equal to G single-graph calls.
 * The batched forward needs G * pfs_loss_workspace_bytes(S, T) bytes of workspace.
 * Fibre-sharded graph (ABI 9): one graph whose fibres are split over `world` ranks, each calling with its own
 * contiguous fibre range (S local fibres, S_total over all ranks, one graph per call).  The forward is
 *   1. pfs_loss_shard_fwd: the per-edge and per-fibre outputs of the local fibres and this rank's record
 *      shard_record [2 + 3T] doubles = {n_r, local fibre-penalty sum, per class: sum galaxies [T], mean [T] and
 *      M2 [T] of time2 over the local fibres} (4 launches);
 *   2. the caller makes every rank's record visible to every rank as shard_records [world][2 + 3T], rank order;
 *   3. pfs_loss_shard_merge: n_prime, class_mean, class_coef and scalars of the whole graph (1 launch).  The records
 *      are combined in rank order, so every rank gets bitwise the same results; with world = 1 they are bitwise those
 *      of pfs_loss_fwd.
 * pfs_loss_bwd with S_total set takes the variance over S_total fibres; time, noise, time2, fibre_time and g_time are
 * the local rows, class_mean and class_coef the merged ones.
 * Any edge list (ABI 10): E > 0 edges per graph in any order (duplicates, fibres and classes without edges allowed),
 * edge e = (fibre csr_src, class csr_tgt) as listed by the CSR / CSC arrays of pfs_build_topology, shared by the G graphs.
 * Every per-edge array is then [G, E] in edge-list order (E replaces S*T above).  The variance runs over the fibre x class
 * matrix of cells c_ki = sum of time2 over the edges (k, i), 0 where fibre k has no edge to class i; a fibre without edges
 * has fibre time 0, a class without edges n'_i = 0.  The forward is 4 launches and also writes cell_time [G, E] (the cell
 * value of every edge), which the backward (1 launch) reads.  Workspace: G * pfs_loss_list_workspace_bytes(T).  Graph g's
 * results are bitwise those of a one-graph call.  E > 0 with S_total set, or with a NULL edge array or cell_time, and
 * E = 0 with an edge array set, are refused (PFS_ERR_ARG).
 * Edge list sharded over fibre ranges (ABI 11): each rank holds the edges of its contiguous fibre range (S local fibres,
 * fibres renumbered from 0, S_total over all ranks, E > 0 local edges and their CSR / CSC arrays, one graph per call).
 *   1. pfs_loss_list_shard_fwd: the per-edge and per-fibre outputs of the local edges (cell_time included) and this
 *      rank's record shard_record [2 + 3T] = {S, local fibre-penalty sum, per class: sum galaxies, mean and M2 of the
 *      cells over the S local fibres, zero cells included} (4 launches, workspace pfs_loss_list_workspace_bytes(T));
 *   2. the records exchanged as for ABI 9;
 *   3. pfs_loss_shard_merge with E = 0 and every edge array NULL (the records mean what ABI 9's mean).
 *   With world = 1 the results are bitwise those of pfs_loss_fwd on the same edge list.
 * pfs_loss_list_shard_bwd: the edge-list backward with the variance over S_total fibres (1 launch).  Both refuse
 * (PFS_ERR_ARG, before any CUDA call) a NULL array, E <= 0, S_total unset, S > S_total and G > 1.
 * ---------------------------------------------------------------------------------------- */
typedef struct pfs_loss_args {
    int32_t S, T;                                /* fibres, classes (per graph) */
    const float* time;                           /* [G, S*T] */
    const float* noise;                          /* [G, S*T] uniform [0,1) */
    const float* hours;                          /* [T] or [G, T] (class_tables): T_i = class_info[:,0] */
    const float* counts;                         /* [T] or [G, T] (class_tables): N_i = class_info[:,1] / NFIELDS */
    float total_time, wutils, wvar, pclass, pfiber, sharpness, noiselevel;   /* src/config.py:19,27-28; train.py:21,29 */
    float* galaxies;                             /* [G, S*T] */
    float* time2;                                /* [G, S*T] galaxies * T_i (the `time` of finaloutput) */
    float* fibre_time;                           /* [G, S] */
    float* n_prime;                              /* [G, T] */
    float* class_mean;                           /* [G, T] mean over fibres of time2 */
    float* class_coef;                           /* [G, T] dloss/dn'_i */
    float* scalars;                              /* [G, 8] */
    const float* g_loss;                         /* backward: device vector [G] (upstream gradient of each graph's loss)
                                                    or NULL (1 for every graph) */
    float* g_time;                               /* backward: [G, S*T] */
    void* workspace; size_t workspace_bytes;     /* forward: G * pfs_loss_workspace_bytes(S, T) */
    void* stream;
    const float* sharpness_dev;                  /* optional device scalar overriding `sharpness` (a sharpness schedule
                                                    under CUDA-graph replay, src/train.py:139) */
    int32_t G;                                   /* ABI 8: graphs in the batch; 0 or 1 = one graph */
    int32_t class_tables;                        /* ABI 8: 0 = hours / counts are one [T] table shared by every graph,
                                                    1 = one [G, T] table per graph */
    int32_t S_total;                             /* ABI 9: fibres over all shards; 0 = not sharded (the ABI 8 behaviour).
                                                    With S_total set, S >= 1, S_total >= 2 and G is 0 or 1 */
    int32_t world;                               /* ABI 9: ranks of the sharded graph (pfs_loss_shard_merge) */
    double* shard_record;                        /* ABI 9: pfs_loss_shard_fwd output, [2 + 3T] */
    const double* shard_records;                 /* ABI 9: pfs_loss_shard_merge input, [world][2 + 3T] in rank order */
    int32_t E;                                   /* ABI 10: edges per graph of an edge list; 0 = the dense canonical order
                                                    e = k*T + i (the ABI 9 behaviour, every array below NULL) */
    const int32_t* csr_rowptr;                   /* ABI 10: [S+1]  pfs_build_topology's CSR range of each fibre */
    const int32_t* csr_eid;                      /* ABI 10: [E]    edge id at CSR position q */
    const int32_t* csr_src;                      /* ABI 10: [E]    fibre at CSR position q */
    const int32_t* csr_tgt;                      /* ABI 10: [E]    class at CSR position q */
    const int32_t* csc_colptr;                   /* ABI 10: [T+1]  CSC range of each class */
    const int32_t* csc_q;                        /* ABI 10: [E]    CSR position of the j-th class-sorted edge */
    float* cell_time;                            /* ABI 10: [G, E] forward output, backward input: the cell value c_ki of
                                                    every edge */
} pfs_loss_args;
size_t pfs_sizeof_loss_args(void);
size_t pfs_loss_workspace_bytes(int32_t S, int32_t T);
size_t pfs_loss_list_workspace_bytes(int32_t T);      /* per graph, E > 0 */
int pfs_loss_fwd(const pfs_loss_args* a);
int pfs_loss_bwd(const pfs_loss_args* a);
int pfs_loss_shard_fwd(const pfs_loss_args* a);
int pfs_loss_shard_merge(const pfs_loss_args* a);
int pfs_loss_list_shard_fwd(const pfs_loss_args* a);     /* ABI 11 */
int pfs_loss_list_shard_bwd(const pfs_loss_args* a);     /* ABI 11 */

#ifdef __cplusplus
}
#endif
#endif /* PFS_B200_H */
