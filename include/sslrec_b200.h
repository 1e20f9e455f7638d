/*
 * sslrec_b200 -- C ABI of the B200 (sm_100a) general_cf training hot path.
 *
 * The reference (HKUDS/SSLRec) has no FFI: its "operator interface" for this path is the set of
 * PyTorch calls made by models/general_cf/*.py, models/loss_utils.py, models/aug_utils.py and
 * trainer/trainer.py.  Each entry point below names the reference call site(s) it replaces
 * (file:line, relative to the reference checkout).  INTEGRATION.md shows the ctypes binding a
 * maintainer adds on the reference side.
 *
 * Conventions
 *   - plain C: raw device pointers, sizes, a cudaStream_t passed as void*; no torch types.
 *   - every function returns 0 on success, a negative SSL_E_* code otherwise; the message is
 *     available from ssl_last_error() (thread-local).  No C++ exception crosses the boundary.
 *   - the caller owns every buffer it passes; the library owns only what lives inside an
 *     ssl_plan (work lists + split-row scratch).  Kernels are enqueued on the given stream and
 *     never synchronise it (ssl_plan_create synchronises once, for its uploads).
 *   - all floating point is fp32; node / item ids inside batches are int64 (trainer.py:64),
 *     CSR indices are int32.
 *   - "table view": a [rows, dim] fp32 matrix addressed as base + row * stride (stride in
 *     floats), so one view of the interleaved [N, V, dim] propagation output is
 *     (E + v*dim, V*dim) without a copy.
 */
#ifndef SSLREC_B200_H
#define SSLREC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SSL_API __attribute__((visibility("default")))
#else
#define SSL_API
#endif

#define SSL_OK 0
#define SSL_E_ARG (-1)     /* bad argument (shape, null pointer, unsupported dim) */
#define SSL_E_CUDA (-2)    /* a CUDA runtime call or kernel launch failed */
#define SSL_E_ALLOC (-3)

#define SSL_MAX_VIEWS 4
#define SSL_MAX_SUM_SRC 6
#define SSL_MAX_DIM 128    /* embedding_size must be a multiple of 4 and <= 128 */
#define SSL_MAX_PEERS 7    /* other GPUs of the node whose tables a kernel stores to over NVLink (8-GPU NVSwitch domain) */

SSL_API int ssl_version(void);
SSL_API const char *ssl_last_error(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
SSL_API int64_t ssl_launch_count(void);
/* process-wide switches for tests and A/B profiling (value 0 / 1):
 *   "prop_view_major"  propagation with grid.y = view and one accumulator per thread: DRAM traffic at 1.03x compulsory instead of
 *                      1.3x, but 25-40 % slower on B200 (profiles/r02_prop_variants.md); default 0
 *   "kmeans_rows_per_round"  1 selects kmeans_assign_kernel<1> (one row per warp and round, the round-1 form); default 4 rows per round --
 *                      same arithmetic per (row, centroid), same summation order: bit-identical results (csrc/kmeans_assign.cuh)
 *   "predict_tiled"    ssl_predict_mask as a register-tiled product (128 x 128 score tiles, csrc/predict_tile.cuh); 0 selects the
 *                      round-1 warp-per-item kernel (4 % of the FFMA rate, profiles/r02_ncu_kernels.md), kept as the cross-check; default 1 */
SSL_API int ssl_set_option(const char *name, int64_t value);

/* ------------------------------------------------------------------------------------------
 * a1/a2  adjacency plan -- replaces the torch sparse COO tensor built by
 * data_utils/data_handler_general_cf.py:53-73 as the operand of t.spmm (lightgcn.py:28-29).
 * CSR of the (row block of the) normalised adjacency; the structure and values are symmetric,
 * so the same plan serves A and A^T.
 *   h_rowptr  host  int32 [n_rows+1]   (read during create only)
 *   d_colidx  device int32 [nnz]       global column (node) ids, ascending inside a row
 *   d_vals    device fp32  [nnz]
 *   d_rev     device int32 [nnz] or NULL: position of the reverse entry (col,row); only needed
 *             when an *injected* edge mask is used together with transpose = 1
 *   row_offset  global id of local row 0 (row-sharded multi-GPU; 0 on one GPU)
 *   side_split  global row id where the second side of the bipartite graph starts (|U|), or 0: the work list
 *               then runs all rows of one side before the other, so concurrently running CTAs gather from one
 *               half of the table only (user rows read item rows and vice versa) -- halves the L2 working set
 * ------------------------------------------------------------------------------------------ */
typedef struct ssl_plan ssl_plan;

SSL_API int ssl_plan_create(ssl_plan **out, const int32_t *h_rowptr, const int32_t *d_colidx, const float *d_vals,
                    const int32_t *d_rev, int64_t n_rows, int64_t n_cols, int64_t nnz, int64_t row_offset,
                    int64_t side_split, void *stream);
/* Row-sharded multi-GPU (SURVEY.md 8e): the plan owns the global rows [a0, a1) followed by [b0, b1) -- a GPU's share
 * of the user rows and of the item rows, so every GPU gets the same mix of both sides; h_rowptr runs over the
 * n_rows = (a1-a0) + (b1-b0) local rows in that order, column ids stay global.  ssl_plan_create is the single-range
 * case [row_offset, row_offset + n_rows). */
SSL_API int ssl_plan_create_ranges(ssl_plan **out, const int32_t *h_rowptr, const int32_t *d_colidx, const float *d_vals,
                           const int32_t *d_rev, int64_t n_rows, int64_t n_cols, int64_t nnz, int64_t a0, int64_t a1,
                           int64_t b0, int64_t b1, int64_t side_split, void *stream);
SSL_API int ssl_plan_destroy(ssl_plan *plan);
/* work-list statistics: out[0]=items, out[1]=split rows, out[2]=segments, out[3]=max row nnz */
SSL_API int ssl_plan_stats(const ssl_plan *plan, int64_t out[4]);

/* ------------------------------------------------------------------------------------------
 * a2-a10  one propagation layer for up to SSL_MAX_VIEWS augmented views at once.
 *
 *   acc_v[r]  = sum_p  m_v(p) * s_v * val[p] * x_in[col[p], v]          (CSR row r)
 *   x_v[r]    = acc_v[r] + residual[r, v]                                 (residual optional)
 *   x_v[r]   += eps * sign(x_v[r]) * u / max(|u|_2, 1e-12)                (noise_mode != 0)
 *   x_out[r, v]   = x_v[r]                                                (x_out optional)
 *   sum_out[r, v] = x_v[r] + sum_i sum_src[i][r, v]                       (sum_out optional;
 *                   reduce_views: sum_out[r] = sum_v of the above, + reg_coef * [*reg_coef_dev] * reg_src[r] + reg_src2[r])
 *
 * replaces: t.spmm (lightgcn.py:29, hccf.py:36), the layer sum (lightgcn.py:41, simgcl.py:29,
 * sgl.py:34, ncl.py:41), EdgeDrop (aug_utils.py:18-31) as an in-kernel keep test so no second
 * adjacency is built, EmbedPerturb (aug_utils.py:125-132) as an epilogue, and -- with
 * transpose = 1 and residual = upstream gradient -- the autograd backward of all of them
 * (dX = A_v^T dY evaluated on the same CSR with the mask key swapped).
 *
 * Layouts: x_in [n_cols, in_views, dim] (in_views = 1: all views read the same rows, or
 * = n_views); x_out, residual [n_cols, n_views, dim]; sum_src[i] [n_cols, sum_src_views[i], dim]
 * with sum_src_views[i] in {1, n_views}; sum_out [n_cols, n_views, dim] or [n_cols, dim].
 * Every table is FULL height (n_cols = N rows) and addressed by the GLOBAL row id; a row-sharded
 * plan reads and writes only the rows it owns.
 *
 * Fused all-gather (row-sharded multi-GPU, one NVSwitch domain): with n_peers > 0 every finished
 * row of x_out / sum_out is also stored to the same row of x_out_peers[q] / sum_out_peers[q] --
 * the other GPUs' tables, mapped into this process (CUDA IPC / symmetric memory) -- so after the
 * launches of all ranks have completed (cross-GPU barrier, caller's job) every GPU holds the
 * whole layer output; the NVLink stores overlap the gathers of the rows still being computed.
 * This replaces "one NCCL allgather of the d-wide layer output per layer".
 *
 * edge_mode[v]: 0 keep all; 1 counter-based RNG: keep iff U(seed[v], edge_stream_id, row, col) >= 1-keep
 *               (floor(U + keep), aug_utils.py:28); 2 injected: edge_mask[v][p] != 0, p = CSR
 *               position (rev[p] when transpose).  edge_scale[v] multiplies kept values
 *               (1, or 1/keep for EdgeDrop(resize_val=True), hccf.py:33) of a view with edge_mode 1 or 2; a view with
 *               edge_mode 0 propagates the stored values unscaled.
 * noise_mode[v]: 0 none; 1 RNG uniform(seed[v], noise_stream_id, row, elem);
 *               2 injected: noise_u[v] is a [n_cols, dim] U[0,1) tensor (global row).
 * ------------------------------------------------------------------------------------------ */
typedef struct ssl_prop_args {
    int32_t dim, n_views, in_views, transpose;
    const float *x_in;
    float *x_out;
    float *sum_out;
    const float *residual;
    int32_t reduce_views;
    int32_t n_sum_src;
    const float *sum_src[SSL_MAX_SUM_SRC];
    int32_t sum_src_views[SSL_MAX_SUM_SRC];
    float reg_coef;
    const float *reg_src;             /* [n_rows, dim]; only with reduce_views */
    int32_t edge_mode[SSL_MAX_VIEWS];
    float edge_keep[SSL_MAX_VIEWS];
    float edge_scale[SSL_MAX_VIEWS];
    const uint8_t *edge_mask[SSL_MAX_VIEWS];
    int32_t noise_mode[SSL_MAX_VIEWS];
    const float *noise_u[SSL_MAX_VIEWS];
    float noise_eps;
    uint64_t seed[SSL_MAX_VIEWS];
    uint32_t edge_stream_id;          /* RNG sub-stream of the edge mask: constant over the layers of one forward
                                         (lightgcn.py:36-37, sgl.py:27-28) or the layer index (hccf.py:47) */
    uint32_t noise_stream_id;         /* RNG sub-stream of the perturbation: the layer index (simgcl.py:26-27) */
    int32_t n_peers;                  /* 0 on one GPU */
    float *x_out_peers[SSL_MAX_PEERS];    /* peers' copies of the x_out table (same shape, same row addressing) */
    float *sum_out_peers[SSL_MAX_PEERS];  /* peers' copies of the sum_out table */
    const float *reg_coef_dev;        /* optional device scalar multiplied into reg_coef (the upstream gradient of the
                                         regulariser term: d loss / d reg_params is only known on the device) */
    const float *reg_src2;            /* optional second [n_cols, dim] row source added with coefficient 1 (with reduce_views):
                                         gradient rows that losses wrote for layer 0 (ncl.py:75) */
    const uint64_t *seed_ptr[SSL_MAX_VIEWS];  /* optional: the view's seed is READ FROM THE DEVICE (overrides seed[v]) -- a step captured
                                         in a CUDA graph draws fresh masks / noise at every replay because the host rewrites these
                                         words, not the launch arguments */
} ssl_prop_args;

SSL_API int ssl_propagate_layer(const ssl_plan *plan, const ssl_prop_args *args, void *stream);

/* ------------------------------------------------------------------------------------------
 * a9  NodeDrop (aug_utils.py:40-50, sgl.py:24-25).
 * forward : out[r, v] = x[r] * m_v(r)            x [n, dim] -> out [n, n_views, dim]
 * backward: out[r]   += sum_v g[r, v] * m_v(r)   g [n, n_views, dim] -> out [n, dim]  (accumulate)
 * mode[v]: 0 keep all; 1 RNG keep iff U(seed[v], row) >= 1-keep; 2 injected mask[v][r] != 0.
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_node_drop(const float *x, float *out, int64_t n, int32_t dim, int32_t n_views, int32_t backward,
                  const int32_t *mode, const float *keep, const uint8_t *const *mask, const uint64_t *seed,
                  int64_t row_offset, void *stream);
/* the same with per-view seeds read from the device (seed_ptr[v] may be NULL: then seed[v] is used) */
SSL_API int ssl_node_drop_dev(const float *x, float *out, int64_t n, int32_t dim, int32_t n_views, int32_t backward,
                      const int32_t *mode, const float *keep, const uint8_t *const *mask, const uint64_t *seed,
                      const uint64_t *const *seed_ptr, int64_t row_offset, void *stream);

/* ------------------------------------------------------------------------------------------
 * a11+a12  gathers + BPR  (lightgcn.py:48-52, loss_utils.py:7-10; hccf.py:70-74 is the same
 * function written as -log sigmoid).  loss_b = softplus(a.n - a.p), coef_b = sigmoid(a.n - a.p).
 * users / items are table views; ancs index the user view, poss/negs the item view.
 * ssl_bpr_bwd adds scale * (*gscale) * d loss_b into the gradient views (atomicAdd: batch
 * indices repeat; the reference's index_put_(accumulate) does the same).
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_bpr_fwd(const float *users, int64_t u_stride, const float *items, int64_t i_stride,
                const int64_t *ancs, const int64_t *poss, const int64_t *negs, int64_t batch, int32_t dim,
                float *loss_b, float *coef_b, void *stream);
SSL_API int ssl_bpr_bwd(const float *users, int64_t u_stride, const float *items, int64_t i_stride,
                const int64_t *ancs, const int64_t *poss, const int64_t *negs, int64_t batch, int32_t dim,
                const float *coef_b, const float *gscale, float scale,
                float *g_users, int64_t gu_stride, float *g_items, int64_t gi_stride, void *stream);

/* ------------------------------------------------------------------------------------------
 * a13/a14  InfoNCE, never materialising the [B, N_side] logits
 * (loss_utils.py:30-39 cal_infonce_loss; :42-51 cal_infonce_loss_spec_nodes with norm_mode 1).
 *
 * ssl_rows_normalize  x^ = x / sqrt(1e-8 + |x|^2)  (norm_mode 0, loss_utils.py:33-35) or
 *                     F.normalize(x + 1e-8)        (norm_mode 1, loss_utils.py:45-46) or
 *                     F.normalize(x)               (norm_mode 2, loss_utils.py:78,85) or
 *                     x itself                     (norm_mode 3: LightGCL contracts raw rows, lightgcl.py:112);
 *   optional gather (idx != NULL: row i of the output is x[idx[i]]), optional scale of the
 *   output (alpha), writes row-major out [n, dim], the K-major tile copy out_t
 *   [ceil(n/64), dim, 64] the streaming side of ssl_softmax_gemm reads (may be NULL),
 *   rinv [n] (the 1/norm used, needed by the backward), and optionally the tf32 split
 *   out_hi = tf32_rna(out), out_lo = tf32_rna(out - out_hi) (cvt.rna: round to nearest, ties away from zero; the 13 low
 *   mantissa bits of both parts are zero), row-major [n, dim] each, plus their transposes
 *   out_thi / out_tlo [dim, t_pitch] (t_pitch >= ceil64(n), multiple of 4) that
 *   ssl_softmax_gemm_tf32x3 reads through TMA.
 * ssl_softmax_gemm    for every row r of R [n_r, dim] over the rows c of C (row-major C
 *   [n_c, dim] and its K-major tile copy C_t):   e = exp2(R_r . C_c - offset) * colscale[c]
 *   rowsum_part[s, r] = sum_c e   (optional)     o_part[s, r, :] = sum_c e * C_c
 *   for the s-th of n_split contiguous chunks of C: chunk s is the 64-row tiles [t0, t1) with t0 = n_ct*s/n_split,
 *   t1 = n_ct*(s+1)/n_split, n_ct = ceil(n_c/64) (1 <= n_split <= n_ct).  C and C_t are read in whole 64-row tiles: the
 *   caller supplies ceil64(n_c) rows of C and ceil(n_c/64) tiles of C_t [ceil(n_c/64), dim, 64] (the layout
 *   ssl_rows_normalize writes), and their padding rows must be finite -- they enter the products and are masked
 *   afterwards (ssl_rows_normalize writes them as zeros).  R, C, C_t 16-byte aligned; colscale is read for c < n_c
 *   only.  One launch does the forward of a term
 *   (R = scaled anchors, C = normalised table: log-sum-exp and the softmax-weighted table
 *   average that is the anchor gradient) and, with the roles swapped, its backward
 *   (R = table tile, C = anchors, colscale = g/rowsum: the dense table gradient).
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_rows_normalize(const float *x, int64_t stride, const int64_t *idx, int64_t n, int32_t dim, int32_t norm_mode,
                       float alpha, float *out, float *out_t, float *rinv, float *out_hi, float *out_lo,
                       float *out_thi, float *out_tlo, int64_t t_pitch, void *stream);
SSL_API int ssl_softmax_gemm(const float *R, int64_t n_r, const float *C, const float *C_t, int64_t n_c, int32_t dim,
                     const float *colscale, float offset, int32_t n_split, float *rowsum_part, float *o_part,
                     void *stream);
/* The same contraction on the tcgen05 tensor cores with 3xTF32 error compensation (fp32-grade
 * accuracy): operands are the hi / lo splits written by ssl_rows_normalize, row-major [n, dim],
 * and for the streamed operand also the transposed splits CT_hi / CT_lo [dim, ct_pitch];
 * dim must be 32 or 64.  colscale, when given, must be readable up to ceil64(n_c) floats (the
 * padded tail is loaded with the tile and masked).  Outputs and semantics are those of
 * ssl_softmax_gemm. */
SSL_API int ssl_softmax_gemm_tf32x3(const float *R_hi, const float *R_lo, int64_t n_r, const float *C_hi, const float *C_lo,
                            const float *CT_hi, const float *CT_lo, int64_t ct_pitch, int64_t n_c, int32_t dim,
                            const float *colscale, float offset, int32_t n_split, float *rowsum_part, float *o_part,
                            void *stream);
/* forward epilogue of one term: reduces the split partials and produces, per anchor b,
 *   rowsum[b] (+ deno_eps), obar[b,:] = o[b,:]/rowsum[b] and
 *   loss_b[b] = -(a^_b . p^_b)/tau + 1/tau + ln(rowsum[b])          */
SSL_API int ssl_nce_finalize(const float *rowsum_part, const float *o_part, int32_t n_split, int64_t batch, int32_t dim,
                     const float *a_hat, const float *p_hat, float tau, float deno_eps,
                     float *rowsum, float *obar, float *loss_b, void *stream);
/* backward w.r.t. the gathered rows: d a^ = g/tau (obar - p^), d p^ = -g/tau a^, pushed through
 * the normalisation (de = rinv (dx^ - x^ (x^ . dx^))) and atomically added to the gradient views.
 * g = scale * (*gscale).  g1 / g2 may be NULL (NCL prototypes, HCCF's detached side). */
SSL_API int ssl_nce_bwd_rows(const float *a_hat, const float *p_hat, const float *obar, const float *rinv1, const float *rinv2,
                     const int64_t *idx, int64_t batch, int32_t dim, float tau, const float *gscale, float scale,
                     float *g1, int64_t g1_stride, float *g2, int64_t g2_stride, void *stream);
/* backward w.r.t. the table: dt^ = sum of the split partials of the swapped ssl_softmax_gemm;
 * g_table[j] (+)= rinv_j (dt^_j - t^_j (t^_j . dt^_j)) */
SSL_API int ssl_nce_bwd_table(const float *dt_part, int32_t n_split, const float *t_hat, const float *rinv, int64_t n,
                      int32_t dim, float *g_table, int64_t g_stride, int32_t accumulate, void *stream);
/* the epilogue of a term without a positive pair, log(sum_j exp(a_b . t_j / temp) + eps) (lightgcl.py:112-113):
 * rowsum[b] = sum of the partials + eps, obar = o / rowsum, loss_b[b] = ln(rowsum[b]) */
SSL_API int ssl_lse_finalize(const float *rowsum_part, const float *o_part, int32_t n_split, int64_t batch, int32_t dim, float eps,
                     float *rowsum, float *obar, float *loss_b, void *stream);
/* colscale[b] = scale * (*gscale) * ln2 / rowsum[b] for the swapped gemm */
SSL_API int ssl_nce_colscale(const float *rowsum, int64_t batch, const float *gscale, float scale, float *colscale, void *stream);

/* ------------------------------------------------------------------------------------------
 * a15  reg_params (loss_utils.py:20-24): out[0] = sum x^2, deterministic two-stage reduction.
 * ssl_sum: out[0] = alpha * sum x (same reduction; used for the per-sample loss vectors).
 * ssl_axpy: y += alpha * (*gscale) * x  (gradient of the regulariser, 2 * reg_weight * W).
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_sumsq(const float *x, int64_t n, float *out, void *stream);
SSL_API int ssl_sum(const float *x, int64_t n, float alpha, float *out, void *stream);
SSL_API int ssl_axpy(const float *x, float *y, int64_t n, const float *gscale, float alpha, void *stream);

/* ------------------------------------------------------------------------------------------
 * a20  Adam (trainer.py:45-49,68 -> torch.optim.Adam, amsgrad off): one fused pass over
 * p, g, m, v.  step is 1-based; weight_decay is folded into g as torch does.  Hyper-parameters are
 * doubles (Python floats): 1 - beta and the bias corrections are formed in double, then rounded once.
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_adam_step(float *p, const float *g, float *m, float *v, int64_t n, int64_t step, double lr, double beta1,
                  double beta2, double eps, double weight_decay, void *stream);
/* Row-sharded Adam: the same update on the n elements p[0..n) this GPU owns (p, g, m, v already point at the owned
 * range), with every new parameter value also stored to the same position of p_peers[q] (the other GPUs' replicas of
 * the table, mapped over NVLink) -- the all-gather of the updated table fused into the optimizer kernel. */
SSL_API int ssl_adam_step_peers(float *p, float *const *p_peers, int32_t n_peers, const float *g, float *m, float *v, int64_t n,
                        int64_t step, double lr, double beta1, double beta2, double eps, double weight_decay, void *stream);
/* The step count read from the device: *step_dev (>= 1) is the 1-based step of THIS update; the bias corrections are formed on the
 * device (double precision, as the host path) into scratch2 (2 floats) by a one-thread launch, so that a CUDA graph holding the
 * optimizer step replays with a counter the graph itself increments. */
SSL_API int ssl_adam_step_dev(float *p, float *const *p_peers, int32_t n_peers, const float *g, float *m, float *v, int64_t n,
                      const int64_t *step_dev, float *scratch2, double lr, double beta1, double beta2, double eps, double weight_decay,
                      void *stream);

/* ------------------------------------------------------------------------------------------
 * a18  full_predict + _mask_predict (lightgcn.py:58-66, base_model.py:35-36) and the top-k that
 * consumes it (metrics.py:108).
 * ssl_predict_mask: preds[b, i] = (U[users[b]] . I[i]) * (1 - M[b,i]) - 1e8 * M[b,i]; the mask is
 *   either the dense int64 [n_b, n_item] tensor the reference passes (mask_dense) or, when that
 *   is NULL, the training CSR (trn_rowptr int32 [n_user+1], trn_cols int32) read on device.  Every score is one
 *   sequential fp32 FMA chain over k = 0 .. dim-1; masked positions read exactly -1e8.
 * ssl_topk: the k largest entries of every row, descending, ties broken by the lower index.
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_predict_mask(const float *users_tab, int64_t u_stride, const float *items_tab, int64_t i_stride,
                     const int64_t *users, int64_t n_b, int64_t n_item, int32_t dim, const int64_t *mask_dense,
                     const int32_t *trn_rowptr, const int32_t *trn_cols, float *preds, void *stream);
/* Opt-in evaluation mode (test.exact_order): Y = A X with the accumulation order of the reference's CPU t.spmm (lightgcn.py:29) -- every output
 * element one sequential fp32 FMA chain over the CSR row in ascending column order, no row splitting -- so that, with the layer sum formed in
 * the reference's order and ssl_predict_mask's sequential score chains, full_predict reproduces the reference's CPU full_predict bit for bit.
 * rowptr: DEVICE int32 [n_rows + 1]; x [*, dim] / y [n_rows, dim] with row strides in floats.  Not on the training path (csrc/spmm_exact.cuh). */
SSL_API int ssl_spmm_exact(const int32_t *rowptr, const int32_t *colidx, const float *vals, int64_t n_rows, const float *x, int64_t x_stride,
                   int32_t dim, float *y, int64_t y_stride, void *stream);
SSL_API int ssl_topk(const float *preds, int64_t n_b, int64_t n_item, int32_t k, int64_t *out_idx, float *out_val, void *stream);

/* ------------------------------------------------------------------------------------------
 * SURVEY 8(f) row 4  DirectAU's losses (loss_utils.py:75-86) on unit rows x^ = F.normalize(x)
 * (ssl_rows_normalize with norm_mode 2).
 * ssl_align_fwd: loss_b[b] = |x^_b - y^_b|^2 (alignment, alpha = 2; the caller averages).
 * uniformity(x) = log mean_{i<j} exp(-2 |x^_i - x^_j|^2): the pair sum is ssl_softmax_gemm[_tf32x3]
 *   with R = 4 log2(e) x^, C = x^, offset = 4 log2(e); ssl_uniform_finalize reduces its split partials
 *   and removes the i == j term: pair_sum[i] = sum_{j!=i} e_ij, w[i,:] = sum_{j!=i} e_ij x^_j.
 * ssl_unit_rows_bwd: dx^_b = scale * (*gscale) * (c1 d1_b + c2 d2_b) pushed through the normalisation,
 *   g_out[idx[b]] += rinv_b (dx^_b - x^_b (x^_b . dx^_b))   (d2 may be NULL; idx NULL = identity).
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_align_fwd(const float *xhat, const float *yhat, int64_t batch, int32_t dim, float *loss_b, void *stream);
SSL_API int ssl_uniform_finalize(const float *rowsum_part, const float *o_part, int32_t n_split, int64_t batch, int32_t dim,
                         const float *r_scaled, const float *xhat, float offset, float *pair_sum, float *w, void *stream);
SSL_API int ssl_unit_rows_bwd(const float *xhat, const float *rinv, const int64_t *idx, int64_t batch, int32_t dim, const float *d1,
                      float c1, const float *d2, float c2, const float *gscale, float scale, float *g_out, int64_t g_stride,
                      void *stream);

/* ------------------------------------------------------------------------------------------
 * a7  HCCF's hyper-graph branch (hccf.py:43-49 + HGNNLayer :100-108) and its autograd backward without library GEMMs.
 * All products are skinny (n rows x {dim, hyper_num} <= 128), so two kernel shapes cover them:
 * ssl_rowgemm   out[r, :n_out] (+)= leaky( scale * ( in1[r, :k1] M1 + in2[r, :k2] M2 ), slope )     row-local
 *     M1 [k1, n_out] row-major (m1_trans: given as [n_out, k1]); the second product is optional (in2 = NULL);
 *     pre_ref: in1[r, j] is multiplied by act'(pre_ref[r, j]) = (pre_ref > 0 ? 1 : pre_slope) while it is loaded
 *     (dZ = dY * act'(Y): LeakyReLU keeps the sign, so the saved OUTPUT tells the derivative); slope = 1: no activation.
 *     replaces  E_side @ W * mult (:43-44), adj @ hids (:106) and, in the backward, dZ @ lat^T + X @ dlat^T, H @ dlat, dA @ W^T.
 * ssl_colgemm   out[k1, k2] = post( scale * sum_r in1[r, :k1]^T (x) in2[r, :k2] )                   reduction over rows
 *     per-CTA partials part[ssl_colgemm_parts(n_rows), k1, k2] are reduced in a fixed order (bit-reproducible);
 *     pre_ref acts on in2 as above; mode 0: out_act (optional) = leaky(out); mode 1: out *= act'(ref).
 *     replaces  adj.T @ embeds (:105) and, in the backward, H^T dZ and E^T dA.
 * ssl_hyper_dropout  F.dropout(A, p = 1 - keep) (:48-49): out = x * m / keep (accumulate: out += ..., the backward);
 *     mode 1: m = floor(U + keep) from the in-kernel counter-based generator keyed (seed, stream_id; row, 4-column group);
 *     mode 2: m = mask [n, h] fp32 of 0 / 1 (injected draws).
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_rowgemm(const float *in1, int64_t in1_stride, int32_t k1, const float *m1, int32_t m1_trans, const float *in2,
                int64_t in2_stride, int32_t k2, const float *m2, int32_t m2_trans, const float *pre_ref, int64_t pre_stride,
                float pre_slope, float *out, int64_t out_stride, int32_t n_out, float scale, float slope, int32_t accumulate, int64_t n_rows,
                void *stream);
SSL_API int ssl_colgemm_parts(int64_t n_rows);
SSL_API int ssl_colgemm(const float *in1, int64_t in1_stride, int32_t k1, const float *in2, int64_t in2_stride, int32_t k2,
                const float *pre_ref, int64_t pre_stride, float slope, int64_t n_rows, float *part, float scale, int32_t mode,
                const float *ref, float *out, float *out_act, void *stream);
SSL_API int ssl_hyper_dropout(const float *x, float *out, int64_t n, int32_t h, float keep, int32_t mode, const float *mask, uint64_t seed,
                      uint32_t stream_id, int32_t accumulate, void *stream);
/* seed read from the device (CUDA-graph replay, see ssl_prop_args.seed_ptr) */
SSL_API int ssl_hyper_dropout_dev(const float *x, float *out, int64_t n, int32_t h, float keep, int32_t mode, const float *mask,
                          const uint64_t *seed_ptr, uint32_t stream_id, int32_t accumulate, void *stream);

/* ------------------------------------------------------------------------------------------
 * a17  KMeansClustering (aug_utils.py:142-157, NCL): one Lloyd iteration = assignment
 *   idx[r] = argmin_k sum_j (x_rj - c_kj)^2 (ties -> lowest k) and the centroid update
 *   c_k = sum_{idx[r]=k} x_r / (count_k + 1e-6), in place.  Deterministic (static row partition,
 *   ordered partial sums, no floating-point atomics).  ssl_kmeans_workspace gives the launch
 *   shape: part_sum must hold n_cta * k * dim floats and part_cnt n_cta * k.  *changed is
 *   incremented by the number of rows whose assignment changed (initialise assign to -1).
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_kmeans_workspace(int64_t n, int32_t dim, int32_t k, int32_t *n_cta, int32_t *n_warps);
SSL_API int ssl_kmeans_iter(const float *x, int64_t stride, int64_t n, int32_t dim, int32_t k, float *centroids, int64_t *assign,
                    float *part_sum, float *part_cnt, float *counts, int32_t *changed, void *stream);

/* ------------------------------------------------------------------------------------------
 * a21  PairwiseTrnData.sample_negs (datasets_general_cf.py:13-26): negs[e] = an item drawn uniformly
 *   until users[e] has no training interaction with it (membership by binary search in the sorted
 *   training CSR, int32).  Counter-based: a pure function of (seed, epoch, e).
 * ------------------------------------------------------------------------------------------ */
SSL_API int ssl_sample_negs(const int64_t *users, int64_t n_pairs, const int32_t *trn_rowptr, const int32_t *trn_cols,
                    int64_t n_item, uint64_t seed, uint32_t epoch, int64_t *negs, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SSLREC_B200_H */
