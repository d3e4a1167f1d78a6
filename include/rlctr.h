/*
 * rlctr.h -- C ABI of librlctr_sm100a.so: the B200 (sm_100a) hot path of
 * jqsl2012/RL_CTR_Prediction.
 *
 * The reference has no operator/FFI layer of its own (SURVEY.md section 8b): its seam
 * is the nn.Module surface of src/models/p_model.py, src/models/Feature_embedding.py and
 * the loop functions of src/main/pretrain_main.py / src/all_main/main.py.  Each entry
 * point below names the reference lines whose ATen op sequence it replaces; the Python
 * package rl_ctr_prediction_b200 binds these symbols with ctypes behind drop-in classes of
 * the same names, constructors and state_dict keys (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - the caller owns every buffer (tables, optimizer state, outputs, workspaces); the
 *     library never allocates or frees device memory and keeps no global mutable state;
 *   - all work is enqueued on the `stream` argument: no implicit synchronisation, no use
 *     of the default stream, safe to capture into a CUDA graph;
 *   - return value: 0 = success, negative = RLCTR_E* argument error, positive = cudaError_t;
 *   - all device pointers must be 16-byte aligned unless noted; ids are int64 as in the
 *     reference's LongTensor contract (src/models/creat_data.py:15-19);
 *   - an id outside [0, n_rows) is treated as an all-zero row (no fault, no update).
 *
 * Table layout ("fused row"): one row per feature id, `row_stride` floats (multiple of 4,
 * or exactly 1 for the LR table), column `lin_col` = first-order weight (nn.Embedding(N,1),
 * p_model.py:14,34,69,263; -1 if the model has none), columns emb_col .. emb_col+dim-1 =
 * the latent vector (p_model.py:38,267; for FFM the F per-field vectors of p_model.py:76-78
 * interleaved, dim = F*D), remaining columns zero padding.  The 128-bit aligned fused row
 * turns the reference's two gathers per field (4 B + 4*D B, two DRAM sectors each) into
 * one aligned vector read (SURVEY H3).
 */
#ifndef RLCTR_H_
#define RLCTR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RLCTR_VERSION 100

#define RLCTR_OK            0
#define RLCTR_EINVAL       (-1)   /* bad argument (NULL, negative size, ...)            */
#define RLCTR_EUNSUPPORTED (-2)   /* shape outside what the kernels are built for        */
#define RLCTR_EWORKSPACE   (-3)   /* workspace too small                                 */
#define RLCTR_EALIGN       (-4)   /* pointer not 16-byte aligned / stride not allowed    */

typedef struct CUstream_st* rlctr_stream_t;   /* == cudaStream_t */

/* One embedding table in the fused-row layout described above. */
#define RLCTR_MAX_WORLD 8
typedef struct rlctr_table {
    float*  data;        /* [n_rows, row_stride] */
    int64_t n_rows;      /* feature_nums */
    int32_t row_stride;  /* floats per row: 1, or a multiple of 4 */
    int32_t lin_col;     /* column of the first-order weight, -1 = none */
    int32_t emb_col;     /* first column of the latent vector */
    int32_t dim;         /* latent_dims (FFM: field_nums*latent_dims), 0 = none */
    int32_t row_pitch;   /* floats between consecutive rows, >= row_stride (0 means row_stride).  A trainable
                          * table is laid out [ p | exp_avg | exp_avg_sq ] per row (row_pitch = 3*row_stride,
                          * rlctr_adam.exp_avg = data + row_stride, .exp_avg_sq = data + 2*row_stride) so the
                          * optimizer touches ONE contiguous 3*row_stride*4-byte record per row instead of three
                          * random 64 B blocks: random HBM accesses are activation-rate bound, not byte bound
                          * (profiles/r1_gather_probe.md).  The Adam arrays always use the table's pitch. */
    /* Row sharding over the GPUs of one box (SURVEY section 8e).  world <= 1: not sharded.  world = 2, 4 or 8: row `id`
     * lives on rank id % world at local row id / world; peers[r] is the base of rank r's shard as mapped into THIS
     * process (CUDA peer / symmetric memory over NVLink; peers[own rank] == data); n_rows is then the GLOBAL row
     * count.  Only the forward gathers (rlctr_embed_fwd) read through peers[]; the optimizer kernels always run on
     * the owner against a table struct that describes the local shard (world = 0). */
    int32_t world;
    float*  peers[RLCTR_MAX_WORLD];
} rlctr_table;

/* torch.optim.Adam state for one table (src/main/pretrain_main.py:181).  `sched[t]` holds
 * the two Python-double scalars torch derives at step t, cast to fp32:
 * (lr / (1 - beta1^t), sqrt(1 - beta2^t)).  `step` is a DEVICE scalar holding the number of
 * COMPLETED optimizer steps (0 after construction), so a captured CUDA graph can be replayed
 * while the step advances (rlctr_step_advance, +1 after the update kernels of a step). */
typedef struct rlctr_adam {
    float*         exp_avg;      /* [n_rows, row_stride] at the table's row_pitch */
    float*         exp_avg_sq;   /* [n_rows, row_stride] at the table's row_pitch */
    int32_t*       stamp;        /* [n_rows] last step at which the row is up to date; NULL in sparse mode */
    const float*   sched;        /* [sched_len][2], index = step (entry 0 unused) */
    const int32_t* step;         /* device scalar: completed steps t; update kernels apply step t+1 */
    int32_t        sched_len;
    int32_t        stamp_col;    /* >= 0: the row's stamp is the int32 stored at float offset stamp_col of the row RECORD
                                  * itself (a padding column of the row, or the 4th float of an LR record [w|m|v|stamp]);
                                  * `stamp` is then ignored.  The stamp rides along with data the kernels touch anyway:
                                  * no second random HBM access per row.  -1: separate `stamp` array (NULL = not lazy). */
    /* hyper-parameters as the Python DOUBLES torch.optim.Adam holds: the kernels use float(1 - beta1),
     * float(1 - beta2), float(eps), float(weight_decay) exactly as torch derives them in double and casts
     * at the op (1.0f - 0.999f differs from float(1 - 0.999) by 1.3e-5 relative) */
    double         beta1, beta2, eps, weight_decay;
    /* rlctr_rows_lookup's staging array, or NULL.  Non-NULL (rlctr_rows_adam only): the (p | exp_avg | exp_avg_sq) of the
     * row at sorted position k are read from stage[k * rlctr_lookup_stage_floats(table)] -- already current through *step --
     * instead of from the table record, and nothing is replayed; the updated record is written to the table as usual. */
    const float*   stage;
} rlctr_adam;

/* Where rlctr_rows_lookup leaves the rows of a batch.  gathered[r] is rank r's [n_per_rank, row_stride] lookup buffer as
 * mapped into THIS process (world <= 1: gathered[0], indexed by slot); a slot of the sorted view is a GLOBAL slot
 * src_rank * n_per_rank + slot, as in rlctr_rowgrad. */
typedef struct rlctr_lookup {
    float*   stage;                       /* [n, rlctr_lookup_stage_floats(table)], 16-byte aligned */
    int32_t  world;
    uint32_t n_per_rank;
    float*   gathered[RLCTR_MAX_WORLD];
} rlctr_lookup;

/* Where the gradient of a gathered row comes from.  For sorted position k with
 * slot = sorted_slots[k], b = slot / fields, f = slot % fields, the row gradient is
 *     staged[slot]                                   (generic, row_stride floats)
 *   + dlogit[b] at lin_col                           (d z / d w = 1)
 *   + dlogit[b] * (sums[b] - row) on the latent cols (FM: d z / d v_f = S - v_f)
 *   + extra[b, f*dim .. ]          on the latent cols (dense tail, e.g. the DeepFM tower)
 * any of the four pointers may be NULL. */
#define RLCTR_STAGED_PARTNER 1   /* staged[slot] = d logit / d row (rlctr_ffm_fwd `partners`): the row
                                  * gradient is dlogit[b] * staged[slot] and nothing else            */
#define RLCTR_DZ_IN_SUMS     2   /* dlogit[b] is ALSO stored in the last (padding) column of sums[b, :] and is read from
                                  * there: for a sharded table the owner then pulls ONE aligned 64-byte line per occurrence
                                  * over NVLink instead of a 4-byte and a 64-byte one (needs row_stride > used columns)  */
typedef struct rlctr_rowgrad {
    const float* staged;   /* [n, row_stride] */
    const float* dlogit;   /* [B] */
    const float* sums;     /* [B, row_stride] from rlctr_embed_fwd */
    const float* extra;    /* [B, fields*dim] */
    int32_t      fields;
    int32_t      flags;    /* 0 or RLCTR_STAGED_PARTNER */
    /* Sharded tables: the owner reduces the gradients of ALL ranks' batches.  world > 1: a slot is a GLOBAL slot
     * g = src_rank * n_per_rank + slot, and the four arrays above are read from rank src_rank's buffers through
     * peer_*[src_rank] (peer-mapped memory, the pull side of the gradient exchange over NVLink); the plain pointers are
     * ignored (NULL-ness of peer_*[0] decides which terms exist). */
    int32_t      world;
    uint32_t     n_per_rank;                       /* slots per rank (batch * fields, equal on every rank) */
    const float* peer_staged[RLCTR_MAX_WORLD];
    const float* peer_dlogit[RLCTR_MAX_WORLD];
    const float* peer_sums[RLCTR_MAX_WORLD];
    const float* peer_extra[RLCTR_MAX_WORLD];
} rlctr_rowgrad;

int         rlctr_version(void);
/* kernels launched by this library in this process so far (host-side tally; bench.py's gpu_launches) */
unsigned long long rlctr_launch_count(void);
const char* rlctr_strerror(int code);

/* ------------------------------------------------------------------------------------
 * K1  fused gather + first order + FM second order.
 * Replaces, per batch: nn.Embedding gathers p_model.py:23,47,54,303,311,320 and the
 * sum/pow/sub/mul temporaries of LR.forward :18-26, FM.forward :40-57, DeepFM.to_fm
 * :296-313 (one gather feeds the FM term and the tower input, reference gathers twice).
 *   logit[b]   = bias + sum_f w[x_f] (+ 0.5*sum_d[(sum_f v)^2 - sum_f v^2] if RLCTR_FM_TERM)
 *   pctr[b*pctr_stride] = sigmoid(logit)          (optional; stride lets M models fill [B,M])
 *   sums[b, :] = column sums over the F gathered rows (saved for the backward; optional)
 *   rows_out[b*rows_pitch + f*dim + d] = v_f[d]   (bit-exact copy; optional; rows_pitch = 0 means fields*dim;
 *                                                  a pitch that is a multiple of 4 floats lets the tower's first
 *                                                  GEMM fetch the rows by TMA; pad columns are never written)
 * ids == NULL: the rows are already in sample order (table->data = rlctr_rows_lookup's `gathered`, [batch*fields, row_stride]):
 * row (b, f) is row b*fields + f -- the streamed forward of the training step.
 * ------------------------------------------------------------------------------------ */
#define RLCTR_FM_TERM 1
int rlctr_embed_fwd(const int64_t* ids, const rlctr_table* table, const float* bias,
                    float* logit, float* pctr, int64_t pctr_stride, float* sums, float* rows_out,
                    int64_t rows_pitch, int64_t batch, int32_t fields, int32_t flags, rlctr_stream_t stream);

/* Pairwise inner products over already-gathered rows: the InnerPNN tower input (p_model.py:178-198)
 *   out[b, :] = [ E (fields*dim) | ip (P = fields*(fields-1)/2) ]   (ip_first != 0: [ ip | E ], Feature_embedding.py:51-59)
 *   ip[p] = <E[i], E[j]> for the p-th pair (i < j, row-major)      rows: [batch, fields*dim] at pitch ld_rows
 * and its backward  grows[b, i, :] = g_E[i, :] + sum_{j != i} g_ip[pair(i, j)] * E[j, :].  fields <= 23. */
int rlctr_pairdots_fwd(const float* rows, int64_t ld_rows, float* out, int64_t ld_out, int64_t batch,
                       int32_t fields, int32_t dim, int32_t ip_first, rlctr_stream_t stream);
int rlctr_pairdots_bwd(const float* rows, int64_t ld_rows, const float* gout, int64_t ld_g, float* grows,
                       int64_t ld_grows, int64_t batch, int32_t fields, int32_t dim, int32_t ip_first,
                       rlctr_stream_t stream);

/* DCN cross network (p_model.py:408-419,423-428) over gathered rows x0 [batch, dim] (pitch ldx):
 *   x_{l+1} = x0 * <x_l, w_l> + b_l + x_l, l = 0..layers-1;  out = x_layers;  s_saved[batch, layers] = <x_l, w_l> (for bwd)
 *   w, b: [layers, dim] (cross_net_w.{l}.weight, cross_net_b.{l} stacked).  dim <= 256, layers <= 6.
 * bwd: gx0 = dL/dx0 (all paths), dw / db [layers, dim]; ws: rlctr_cross_ws_bytes bytes (per-block partials, fixed-order sum). */
size_t rlctr_cross_ws_bytes(int64_t batch, int32_t dim, int32_t layers);
int rlctr_cross_fwd(const float* x0, int64_t ldx, const float* w, const float* b, int32_t layers, float* out, int64_t ld_out,
                    float* s_saved, int64_t batch, int32_t dim, rlctr_stream_t stream);
int rlctr_cross_bwd(const float* x0, int64_t ldx, const float* w, const float* b, const float* s_saved, int32_t layers,
                    const float* gout, int64_t ld_g, float* gx0, int64_t ld_gx, float* dw, float* db, int64_t batch,
                    int32_t dim, void* ws, size_t ws_bytes, rlctr_stream_t stream);

/* OuterPNN product term (p_model.py:236,245-251; the reference's kernel matrix is a constant torch.ones((D, D))):
 *   out[b, :] = [ rows[b, :fields*dim] | cross[dim] ],  cross[d] = sum_{i<dim} (S_d * 1) * S_d,  S = sum_f v_f
 * bwd: grows[b, f*dim+d] = gout[b, f*dim+d] + gout[b, fields*dim+d] * 2 * dim * S_d. */
int rlctr_fieldsq_fwd(const float* rows, int64_t ld_rows, float* out, int64_t ld_out, int64_t batch, int32_t fields,
                      int32_t dim, rlctr_stream_t stream);
int rlctr_fieldsq_bwd(const float* rows, int64_t ld_rows, const float* gout, int64_t ld_g, float* grows, int64_t ld_grows,
                      int64_t batch, int32_t fields, int32_t dim, rlctr_stream_t stream);

/* AFM attention tail (p_model.py:472-481) over gathered rows [batch, fields*dim] (pitch ld_rows):
 *   ip_p = v_i * v_j (i < j);  a_p = relu(W_a ip_p + b_a);  s_p = <w_s, a_p> + b_s;  score = softmax_p(s);
 *   attn = sum_p (score_p * m1_p) ip_p;  out[b] = <fc_w, attn * m2> + fc_b
 * params / dparams: packed [W_a (dim x dim, row = output) | b_a | w_s | b_s | fc_w | fc_b], dim*dim + 3*dim + 2 floats
 * (attention_net.weight/.bias, attention_softmax.weight/.bias, fc.weight/.bias).  m1 / m2: the two F.dropout masks of
 * the reference (always on, :477,479): 0 or 1/(1-p), drawn as hash(rng_state[0], rng_state[1] + b*(P+dim) + col) like
 * the tower's mask (rlctr_rng_advance by batch*(P+dim) after the forward; the backward takes the SAME rng_state values),
 * or read from `masks` [batch, P+dim] when given (mask-as-input parity tests); dropout_p == 0: no dropout.
 * dim in {4, 8, 10}; fields <= 23.  bwd: grows = d L / d rows (written, pitch ld_grows), ws: rlctr_afm_ws_bytes. */
size_t rlctr_afm_ws_bytes(int64_t batch, int32_t dim);
int rlctr_afm_fwd(const float* rows, int64_t ld_rows, const float* params, float* out, int64_t batch, int32_t fields,
                  int32_t dim, float dropout_p, const uint64_t* rng_state, const float* masks, rlctr_stream_t stream);
int rlctr_afm_bwd(const float* rows, int64_t ld_rows, const float* params, const float* gout, float* grows, int64_t ld_grows,
                  float* dparams, int64_t batch, int32_t fields, int32_t dim, float dropout_p, const uint64_t* rng_state,
                  const float* masks, void* ws, size_t ws_bytes, rlctr_stream_t stream);

/* Plain bit-exact row gather out[k, :] = table[ids[k], :] (nn.Embedding.forward); the owner
 * side of the sharded lookup.  out has row_stride floats per row. */
int rlctr_gather_rows(const int64_t* ids, int64_t n, const rlctr_table* table, float* out,
                      rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * K2  FFM over the interleaved table (dim = fields*latent; column block t of row id is
 * field_feature_embeddings[t].weight[id]): p_model.py:82-100.
 *   logit[b] = bias + sum_f w[x_f] + sum_{i<j} <T_j[x_i], T_i[x_j]>
 * partners (optional, training; [B*F, row_stride]): partners[b*F+i, block j] = T_i[x_j] for
 * j != i, 0 on the diagonal, 1 at lin_col -- d logit / d row_i, the autograd of :91 (SURVEY
 * section 3.7 FFM).  Feed it to rlctr_rows_adam as `staged` with RLCTR_STAGED_PARTNER.
 * ------------------------------------------------------------------------------------ */
int rlctr_ffm_fwd(const int64_t* ids, const rlctr_table* table, const float* bias,
                  float* logit, float* pctr, int64_t pctr_stride, float* partners,
                  int64_t batch, int32_t fields, int32_t latent, rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * K5  RL state encoder: Feature_Embedding.forward, Feature_embedding.py:51-59.
 *   out[b, 0:P]      = <v_i, v_j> for (i,j) in the order of :40-43, P = F(F-1)/2
 *   out[b, P:P+F*D]  = v_0 .. v_{F-1}
 * out_stride = floats between consecutive samples (>= P + F*D).
 * ------------------------------------------------------------------------------------ */
int rlctr_featemb_fwd(const int64_t* ids, const rlctr_table* table, float* out, int64_t out_stride,
                      int64_t batch, int32_t fields, rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * BatchNorm1d in TRAINING mode fused with the ReLU behind it: the hidden layers of the policy nets in their learn steps
 * (Linear -> BatchNorm1d -> ReLU: src/models/DDQN_model.py:32-46, DDPG_for_PG_model.py:27-40; torch runs native_batch_norm +
 * relu and three backward kernels there).
 *   fwd: mean / biased variance per column over the batch (two exact passes), y = [relu](gamma * (x - mean) * rsqrt(var + eps) + beta),
 *        running_mean / running_var updated like torch (momentum, UNBIASED variance), save_mean / save_invstd kept for the backward;
 *   bwd: dy_r = gy * (y > 0) if relu; dbeta = sum dy_r; dgamma = invstd * sum dy_r (x - mean);
 *        dx = gamma * invstd * (dy_r - dbeta / B - (x - mean) * invstd^2 * sum dy_r (x - mean) / B)     (batch_norm_backward).
 * x / y / gy / dx: [batch, n] at their pitches; batch <= 65536 (replay batches; RLCTR_EUNSUPPORTED beyond); gamma / beta /
 * running_* / dx / dgamma / dbeta optional.  Eval-mode BatchNorm never comes here: it is folded into the GEMM by the host.
 * ------------------------------------------------------------------------------------ */
int rlctr_bn_relu_fwd(const float* x, int64_t ldx, const float* gamma, const float* beta, float* running_mean, float* running_var,
                      float momentum, float eps, float* y, int64_t ldy, float* save_mean, float* save_invstd, int64_t batch,
                      int32_t n, int32_t relu, rlctr_stream_t stream);
int rlctr_bn_relu_bwd(const float* x, int64_t ldx, const float* y, int64_t ldy, const float* gy, int64_t ldg, const float* gamma,
                      const float* save_mean, const float* save_invstd, float* dx, int64_t lddx, float* dgamma, float* dbeta,
                      int64_t batch, int32_t n, int32_t relu, rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Loss head: torch.sigmoid + nn.BCELoss(mean) forward AND their autograd
 * (p_model.py:55; src/main/pretrain_main.py:167,98,101), with torch's exact clamp
 * semantics (log >= -100; (p-y)/max((1-p)p,1e-12); SURVEY N2):
 *   pctr = sigmoid(logit); loss[0] = mean BCE; dlogit[b] = dL/dlogit[b]; dbias[0] = sum_b dlogit[b].
 * Exactly one of labels_i64 / labels_f32 is non-NULL.  ws: RLCTR_REDUCE_WS_BYTES bytes,
 * zeroed once by the caller (the kernel leaves its counter zeroed).  The mean is a
 * fixed-shape two-level tree: bit-identical from run to run.
 * ------------------------------------------------------------------------------------ */
#define RLCTR_REDUCE_WS_BYTES 16640
int rlctr_bce_fwd_bwd(const float* logit, const int64_t* labels_i64, const float* labels_f32,
                      float* pctr, float* loss, float* dlogit, float* dbias, void* ws, int64_t batch,
                      rlctr_stream_t stream);
/* The drop-in loop keeps the caller's own loss (nn.BCELoss at src/main/pretrain_main.py:98), so
 * autograd hands back dL/dpctr: this is torch's sigmoid_backward, dlogit = grad_p*(1-p)*p, plus
 * dbias[0] = sum_b dlogit[b] (the gradient of the `bias` parameter, p_model.py:16,36) as a
 * fixed-shape tree.  grad_p == NULL: dlogit is an input and only the sum is taken.  dbias, ws
 * optional (ws as in rlctr_bce_fwd_bwd). */
int rlctr_sigmoid_bwd(const float* grad_p, const float* pctr, float* dlogit, float* dbias, void* ws,
                      int64_t batch, rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * K3  deterministic scatter: sort (id, slot) pairs, segment-reduce, fused Adam.
 * Replaces aten::embedding_dense_backward (dense [N,D] zero-fill + index_add) and the
 * dense foreach Adam over all N rows (src/main/pretrain_main.py:101-102; SURVEY a6, a7).
 * ------------------------------------------------------------------------------------ */
size_t rlctr_sort_ws_bytes(int64_t n, int64_t n_rows);
/* sorted_ids/sorted_slots [n]: stable ascending sort of ids (slot = position in `ids`). */
int rlctr_sort_ids(const int64_t* ids, int64_t n, int64_t n_rows,
                   uint32_t* sorted_ids, uint32_t* sorted_slots,
                   void* ws, size_t ws_bytes, rlctr_stream_t stream);

size_t rlctr_rows_ws_bytes(int64_t n);
/* For every distinct id: g = sum over its occurrences (slot order) of the row gradient,
 * then Adam step *step+1 with L2 (g += wd*p) on that row (after replaying the L2-only steps
 * stamp[id]+1 .. *step it missed); stamp[id] = *step+1.  No atomics on the data path;
 * bit-identical from run to run.  Follow with rlctr_step_advance(+1). */
/* Sharded variant: `ids_all` are the ids of EVERY rank's batch (all-gathered, n_all = world * n_per_rank, uint32).  Keys
 * are the LOCAL rows (id / world) of the ids this rank owns (id % world == rank); everything else sorts last as a
 * sentinel and is skipped by the consumers.  sorted_slots are GLOBAL slots (positions in ids_all).  No counts travel
 * to the host: the sorted arrays have n_all entries and rlctr_rows_catchup / rlctr_rows_adam are called with n = n_all. */
int rlctr_sort_ids_sharded(const uint32_t* ids_all, int64_t n_all, int32_t world, int32_t rank, int64_t n_rows_global,
                           uint32_t* sorted_rows, uint32_t* sorted_slots, void* ws, size_t ws_bytes,
                           rlctr_stream_t stream);

/* Gradient-side push (the write counterpart of the owner-side pull through rlctr_rowgrad.peer_*): rank `rank` writes row
 * `slot` of its src[n, width] (per-occurrence gradient rows: DeepFM's tower-input gradients, width = dim) to
 * peer_recv[owner(ids[slot])] + (rank * n + slot) * width.  peer_recv[r] = base of rank r's receive buffer
 * [world * n, width] as mapped into THIS process.  After the step's barrier the owner reads only local memory: it passes
 * rlctr_rowgrad.peer_extra[r] = its own receive buffer + r * n * width.  Posted NVLink writes instead of 2-3 us remote reads
 * on the dependent path of every row.  Out-of-range ids are skipped; width even: 8-byte stores. */
int rlctr_push_rows(const int64_t* ids, int64_t n, int32_t world, int32_t rank, int64_t n_rows_global, const float* src,
                    int32_t width, void* const* peer_recv, rlctr_stream_t stream);
/* Owner routing of a batch's ids (replaces the id all_gather + rlctr_sort_ids_sharded, whose per-rank work grows with the
 * number of GPUs): rank `rank` buckets its n ids by owner, stably, and WRITES (local row, global slot = rank * n + slot) of
 * bucket o into its segment [rank * cap, (rank + 1) * cap) of owner o's receive arrays peer_keys[o] / peer_vals[o]
 * (uint32 [world * cap] each, peer-mapped; unused slots get the sentinel key 0xffffffff).  After a barrier each owner
 * sorts its world * cap received pairs by row with rlctr_sort_routed (ws: rlctr_sort_ws_bytes(world * cap, n_rows_local)
 * bytes): the same sorted view as rlctr_sort_ids_sharded without the non-owned tail, same (row, source rank, slot) order.
 * A bucket with more than `cap` ids sets *overflow (device int32, never cleared by the library) != 0: the view is then
 * incomplete -- rerun with a larger cap.  ws: rlctr_route_ws_bytes(n, world) bytes. */
size_t rlctr_route_ws_bytes(int64_t n, int32_t world);
int rlctr_route_ids(const int64_t* ids, int64_t n, int32_t world, int32_t rank, int64_t n_rows_global, int64_t cap,
                    void* const* peer_keys, void* const* peer_vals, int32_t* overflow, void* ws, size_t ws_bytes,
                    rlctr_stream_t stream);
int rlctr_sort_routed(const uint32_t* keys, const uint32_t* vals, int64_t n_in, int64_t n_rows_local, uint32_t* sorted_rows,
                      uint32_t* sorted_slots, void* ws, size_t ws_bytes, rlctr_stream_t stream);
/* The same sort with the RECEIVE POSITION (index into keys / vals) as the value: sorted_pos[k] = r, the global slot is vals[r].
 * With it the gradient-side rows can travel in the routed order too: rlctr_push_rows_routed writes row `slot` of src[n, width]
 * (width even) to peer_recv[owner] + (rank * cap + bucket position) * width -- the position its (row, slot) pair got from
 * rlctr_route_ids, whose workspace `route_ws` (same ids, same n) still holds the bucket order -- so consecutive threads write
 * consecutive bytes over NVLink and an owner's receive buffer is [world * cap, width], dense.  ws (sort): rlctr_sort_ws_bytes. */
int rlctr_sort_routed_pos(const uint32_t* keys, int64_t n_in, int64_t n_rows_local, uint32_t* sorted_rows, uint32_t* sorted_pos,
                          void* ws, size_t ws_bytes, rlctr_stream_t stream);
int rlctr_push_rows_routed(const void* route_ws, int64_t n, int32_t world, int32_t rank, int64_t cap, const float* src,
                           int32_t width, void* const* peer_recv, rlctr_stream_t stream);
/* The same push for up to RLCTR_GROUP_MAX sources in one pass over the bucket order (the dense-tail members of a row-sharded
 * co-located group): source s is srcs[s] [n, widths[s]] (every width even, rows 8-byte aligned), and occurrence `slot` writes ONE
 * interleaved row peer_recv[owner] + (rank * cap + bucket position) * pitch + off_s, off_s = sum_{t<s} widths[t],
 * pitch = sum_s widths[s].  An owner's receive buffer is [world * cap, pitch]; member s of the update reads it with
 * rlctr_member.extra = buffer + off_s, extra_pitch = pitch.  rlctr_push_rows_routed is this call with n_src = 1. */
int rlctr_push_rows_routed_multi(const void* route_ws, int64_t n, int32_t world, int32_t rank, int64_t cap,
                                 const float* const* srcs, const int32_t* widths, int32_t n_src, void* const* peer_recv,
                                 rlctr_stream_t stream);
int rlctr_rows_adam(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n,
                    const rlctr_rowgrad* grad, const rlctr_table* table, const rlctr_adam* opt,
                    void* ws, size_t ws_bytes, rlctr_stream_t stream);
/* ------------------------------------------------------------------------------------
 * Co-located records: several models trained on the SAME id stream (the reference trains LR, FM, DeepFM ... one after the
 * other on the same encoded batches, src/main/pretrain_main.py:25-45,96-103; the RL ensemble scores M of them per sample,
 * src/all_main/main.py:183-271) keep the parameters of one id in ONE record:
 *     [ p: member columns .. | stamp ]  [ exp_avg ]  [ exp_avg_sq ]      three blocks, `block` floats apart
 * A random HBM access costs the same whether it returns 4 or 128 bytes (profiles/r2_rowprobe.md), so the gather of LR + FM +
 * DeepFM (4 + 44 + 44 bytes) is ONE 128-byte line instead of three, and the optimizer touches three lines per id instead of
 * seven.  The joint table is an ordinary rlctr_table (row_stride = active floats rounded to 4, <= RLCTR_GROUP_MAX_FLOATS;
 * lin_col = -1, emb_col = 0, dim = used columns; rlctr_adam.exp_avg / exp_avg_sq = data + block / + 2*block, stamp_col = the first
 * unused column), so rlctr_rows_catchup / rlctr_adam_flush serve it unchanged; the two calls below are its forward and its update.
 * A record whose row fits one 128-byte line keeps each block in its own line (block 32, pitch 96).  A wider row (up to four
 * lines, 128 floats) is packed [p | exp_avg | exp_avg_sq] with block = row_stride and the pitch rounded up to whole lines.
 * Past RLCTR_GROUP_MAX_FLOATS the calls below, rlctr_rows_catchup and rlctr_adam_flush return RLCTR_EUNSUPPORTED for a joint
 * table with an in-record stamp.
 * A member is one model's view of the record: the columns it owns, where its outputs go, where its gradient side comes from.
 * Members with an FM term keep the chunk alignment of their stand-alone row (emb_col % 4 as in the stand-alone table): their
 * logits and updates are then bit-identical to the stand-alone kernels'.
 * ------------------------------------------------------------------------------------ */
#define RLCTR_GROUP_MAX 4
#define RLCTR_GROUP_MAX_FLOATS 128      /* joint row: four 128-byte lines */
typedef struct rlctr_member {
    int32_t      lin_col;      /* column of the first-order weight in the joint row, -1 = none */
    int32_t      emb_col;      /* first latent column */
    int32_t      dim;          /* latent dims, 0 = none (LR) */
    int32_t      flags;        /* RLCTR_FM_TERM */
    const float* bias;         /* device scalar or NULL */
    /* forward outputs (rlctr_group_fwd), each optional */
    float*       logit;        /* [B] */
    float*       pctr;         /* [B * pctr_stride] */
    int64_t      pctr_stride;
    float*       rows_out;     /* [B, rows_pitch]: rows_out[b, f*dim + d] = v_f[d] (tower input) */
    int64_t      rows_pitch;   /* 0 = fields*dim */
    /* gradient side (rlctr_group_rows_adam) */
    const float* dlogit;       /* [B] dL/dlogit of this member; NULL: it rides in the sums rows, column sums_pitch - RLCTR_GROUP_MAX + m
                                * (one line per sample carries S and every member's dL/dlogit: what the row-sharded step all-gathers).
                                * Never read for a member without a first-order column and without RLCTR_FM_TERM (FNN, PNN, DCN:
                                * its row gradient is `extra` alone) */
    const float* extra;        /* [B, fields*dim] dense-tail gradient on the latent columns, or NULL */
    int64_t      extra_pitch;  /* floats between consecutive occurrences' rows of `extra`; 0 = dim (the [B, fields*dim] layout).
                                * The row-sharded group passes the interleaved receive rows of rlctr_push_rows_routed_multi:
                                * extra = receive buffer + off_m, extra_pitch = the receive row's pitch */
} rlctr_member;
/* One gather per (sample, field) for every member: logit / pctr / rows_out per member as rlctr_embed_fwd would produce them
 * from the member's stand-alone table (a member with lin_col = -1, no bias and no RLCTR_FM_TERM has a table logit of 0: it
 * usually asks for rows_out only); sums[b * sums_pitch + col] = column sums of the joint rows (optional: the backward's S;
 * sums_pitch = 0 means row_stride).  A row-sharded joint table (table->world > 1) is read through peers[] like rlctr_embed_fwd. */
int rlctr_group_fwd(const int64_t* ids, const rlctr_table* table, const rlctr_member* members, int32_t n_members,
                    float* sums, int32_t sums_pitch, int64_t batch, int32_t fields, rlctr_stream_t stream);
/* rlctr_rows_adam over the joint record: per column the gradient of the member that owns it
 * (first-order: dlogit_m[b]; latent: dlogit_m[b] * (sums[b, col] - row[col]) if RLCTR_FM_TERM, + extra_m[slot * extra_pitch + d]),
 * reduced over the occurrences of an id in slot order, then ONE Adam step on the record.  b = slot / fields: for a row-sharded
 * table the slots are GLOBAL (src rank * n_per_rank + slot), `sums` is the all-gathered [world * B, sums_pitch] array, extra_m the
 * owner's receive buffer of rlctr_push_rows, and `world` sizes the grid for the owned ~1/world of the sorted view (the rest are
 * sentinels).  ws: rlctr_rows_ws_bytes(n).
 * slot_of (optional, the routed exchange): sorted_slots then holds RECEIVE positions r of the owner's routing buffers
 * (rlctr_sort_routed_pos); the global slot is slot_of[r] (the `vals` rlctr_route_ids delivered) and extra_m is indexed by r (the rows
 * rlctr_push_rows_routed delivered): dense per-source segments instead of a [world * n, dim] buffer of which 1/world is used. */
int rlctr_group_rows_adam(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n, const rlctr_table* table,
                          const rlctr_adam* opt, const rlctr_member* members, int32_t n_members, const float* sums,
                          int32_t sums_pitch, int32_t fields, int32_t world, const uint32_t* slot_of, void* ws, size_t ws_bytes,
                          rlctr_stream_t stream);

/* Same reduction, but the sums are stored into a dense [n_rows,row_stride] gradient
 * (rows of untouched ids are not written): the literal embedding_dense_backward. */
int rlctr_rows_grad_dense(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n,
                          const rlctr_rowgrad* grad, const rlctr_table* table, float* dense_grad,
                          void* ws, size_t ws_bytes, rlctr_stream_t stream);
/* Lazy-exact mode, the owner-side LOOKUP of a training step (replaces rlctr_rows_catchup + the by-id gather of the forward;
 * the gather side of nn.Embedding, p_model.py:23,47,54,303,311,320, under the dense-Adam semantics of SURVEY N3).  For every
 * distinct id of the sorted view: read its record ONCE, replay in registers the L2-only Adam steps it missed (stamp+1 .. *step),
 * leave (p | exp_avg | exp_avg_sq) in lookup->stage at its sorted position (rlctr_rows_adam takes them from there through
 * rlctr_adam.stage: nothing is replayed twice and the table is written once per step), and WRITE the current row to every
 * sample that gathered it: lookup->gathered[src rank][slot, :] -- for a row-sharded table that is the lookup exchange, as
 * posted NVLink writes into the requester's buffer.  The forward then runs rlctr_embed_fwd with ids == NULL over `gathered`
 * (sample-ordered, streamed).  The table itself is not written.  Vector rows need the in-record stamp (stamp_col >= 0) or a
 * non-lazy optimizer, row_stride <= 16; LR records any stamp.  ws: rlctr_rows_ws_bytes(n) bytes. */
int64_t rlctr_lookup_stage_floats(const rlctr_table* table);
int rlctr_rows_lookup(const uint32_t* sorted_ids, const uint32_t* sorted_slots, int64_t n, const rlctr_table* table,
                      const rlctr_adam* opt, const rlctr_lookup* lookup, void* ws, size_t ws_bytes, rlctr_stream_t stream);
/* Lazy-exact mode: bring every distinct id of the batch up to *step (the completed steps) by
 * replaying the L2-only Adam steps it missed (g = wd*p), so the forward reads exactly what the
 * reference's dense Adam would have produced (SURVEY N3). */
int rlctr_rows_catchup(const uint32_t* sorted_ids, int64_t n, const rlctr_table* table,
                       const rlctr_adam* opt, rlctr_stream_t stream);
/* Replay the missed L2-only steps of rows [row_begin,row_end) up to *step.  Called once per
 * step this IS dense Adam (SURVEY N3, mode A); called before eval/state_dict/epoch end it is
 * the flush of the lazy mode (mode B). */
/* The same catch-up from the batch's ids in BATCH order (int64 [n], duplicates and out-of-range ids allowed): no sorted view is
 * needed, so a training step can sort on another stream while catch-up, gather and tower run (p_model.py:270's read needs current rows,
 * the scatter only needs the sorted view at the end).  Occurrences of one id are told apart by a claim bit per table row (`claim`:
 * rlctr_rows_claim_bytes(n_rows) bytes of scratch, zeroed by the call); the result is independent of which occurrence wins.
 * In-record stamps and co-located records (5..8 active 16-byte chunks) only; RLCTR_EUNSUPPORTED otherwise. */
size_t rlctr_rows_claim_bytes(int64_t n_rows);
int rlctr_rows_catchup_ids(const int64_t* ids, int64_t n, const rlctr_table* table, const rlctr_adam* opt, void* claim,
                           size_t claim_bytes, rlctr_stream_t stream);
int rlctr_adam_flush(const rlctr_table* table, const rlctr_adam* opt,
                     int64_t row_begin, int64_t row_end, rlctr_stream_t stream);
/* Dense Adam for the replicated parameters (bias, tower, policy nets): applies step *step+1
 * with torch semantics. */
int rlctr_dense_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                     const float* sched, const int32_t* step, double beta1, double beta2, double eps,
                     double weight_decay, rlctr_stream_t stream);
/* The same step for up to RLCTR_DENSE_MAX tensors in one launch (host arrays of device pointers / sizes; torch's foreach Adam).
 * torch.optim.Adam keeps one step counter PER PARAMETER (a parameter without a gradient is skipped and its counter stays):
 * `steps` is a device int32 array of completed-step counters and tensor t uses steps[step_index[t]] (step_index: host array,
 * NULL = every tensor uses steps[0]).  rlctr_steps_advance adds 1 to the listed counters (count <= RLCTR_DENSE_MAX). */
#define RLCTR_DENSE_MAX 24
int rlctr_dense_adam_multi(float* const* params, const float* const* grads, float* const* exp_avgs, float* const* exp_avg_sqs,
                           const int64_t* sizes, int32_t count, const float* sched, const int32_t* steps,
                           const int32_t* step_index, double beta1, double beta2, double eps, double weight_decay,
                           rlctr_stream_t stream);
int rlctr_steps_advance(int32_t* steps, const int32_t* step_index, int32_t count, rlctr_stream_t stream);
int rlctr_step_advance(int32_t* step, int32_t delta, rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * K6  ensemble scoring + reward: generate_preds.
 *   variant 0: src/all_main/main.py:183-271 (action in 2..M, reward +1/-1)
 *   variant 1: src/all_main/hybrid_td3_main_per.py:56-133 (action in 1..M, reward 1/0)
 * pctr, w, w_out are [B, M] row-major, M <= 8.
 * ------------------------------------------------------------------------------------ */
int rlctr_generate_preds(const float* pctr, const float* w, const int64_t* action, const int64_t* label,
                         float* y, float* w_out, float* reward, int64_t batch, int32_t models,
                         int32_t variant, rlctr_stream_t stream);
/* The v10 form, src/all_main/hybrid_td3_main_per_v10.py:54-164: models chosen by descending `w` (prob_weights), softmax over the
 * k largest `c_actions` in their own descending order, reward 1/0 on strict comparisons with the all-model mean, and
 * return_c_actions -> c_out [B, M].  As in the reference (:117) the c_out entries of a partial ensemble (action < M) come from the
 * sorted c_actions of batch row r, r = the sample's rank among the samples with the same action.  ws: _ws_bytes(batch) bytes. */
size_t rlctr_generate_preds_v10_ws_bytes(int64_t batch);
int rlctr_generate_preds_v10(const float* pctr, const float* w, const float* c_actions, const int64_t* action,
                             const int64_t* label, float* y, float* c_out, float* reward, int64_t batch, int32_t models,
                             void* ws, size_t ws_bytes, rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * REINFORCE head: PG_model.py:53-58,104-107 (softmax, -log pi(a), loss, and its autograd).
 *   variant 0: literal  loss = (sum_b -logp_b) * mean_b(vt_b)
 *   variant 1: per-sample loss = mean_b(-logp_b * vt_b)
 * act in 1..A (A <= 32).  ws: RLCTR_REDUCE_WS_BYTES bytes zeroed once by the caller.
 * ------------------------------------------------------------------------------------ */
int rlctr_reinforce_loss_bwd(const float* logits, const int64_t* act, const float* vt,
                             float* logp, float* loss, float* dlogits, void* ws,
                             int64_t batch, int32_t actions, int32_t variant, rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Evaluation metrics on the device (replaces the per-batch .tolist() + sklearn.metrics.roc_auc_score of test() /
 * submission(), src/main/pretrain_main.py:110-139):
 *   out[0] = ROC AUC of `pred` against the binary labels (ties get average ranks, as sklearn; NaN if one class only)
 *   out[1] = mean BCE log-loss with torch's clamped logs
 * Deterministic (fixed-order partial sums in double).  ws: rlctr_auc_ws_bytes(n) bytes, 16-byte aligned.
 * ------------------------------------------------------------------------------------ */
size_t rlctr_auc_ws_bytes(int64_t n);
int rlctr_auc_logloss(const float* pred, const int64_t* labels_i64, const float* labels_f32, int64_t n, float* out,
                      void* ws, size_t ws_bytes, rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * K4  dense layers on the tcgen05 tensor cores (3xTF32 split: fp32-grade accuracy; SURVEY H2).
 * nn.Linear of the DeepFM tower (p_model.py:276-293) and of the policy networks
 * (PG_model.py:42-51, DDQN_model.py:20-52, DDPG_for_PG_model.py:20-81): weight [out,in] row-major,
 * bias [out], activations [batch, features] row-major; the layer INPUT x may be padded: ldx floats between its
 * rows (0 = in_dim).  y, gy, dx, dw, db are dense.  When x, gy and the workspace are 16-byte aligned with
 * ldx % 4 == 0 (and out_dim % 4 == 0 for the backward) the operands are fetched by TMA (csrc/mlp_tma.cu);
 * any other shape takes the software-staged kernel (csrc/mlp.cu) -- same numbers, slower.
 *   fwd: y = x w^T + bias, ReLU fused if RLCTR_MLP_RELU (ws: rlctr_mlp_ws_bytes bytes, or NULL = no TMA path)
 *   bwd: with RLCTR_MLP_RELU, gy is first masked IN PLACE by (y > 0) (y = the saved forward output);
 *        dx = gy w (optional), dw = gy^T x (optional, split-K with a fixed-order reduction),
 *        db = column sums of gy (optional).  ws: rlctr_mlp_ws_bytes(batch, in, out) bytes.
 * ------------------------------------------------------------------------------------ */
#define RLCTR_MLP_RELU 1
#define RLCTR_MLP_DROPOUT 2     /* fwd: y = keep ? y / (1-p) : 0 after bias / ReLU (nn.Dropout in train mode, p_model.py:284) */
#define RLCTR_MLP_DX_MASK 4     /* bwd: dx *= (x > 0 ? dx_scale : 0): the ReLU (+dropout) backward of the layer that
                                   produced x, fused into this layer's dgrad epilogue */
#define RLCTR_MLP_FP32 8        /* exact fp32 on the CUDA cores (one FFMA per product, k ascending: the reference's SGEMM arithmetic)
                                   instead of 3xTF32 on the tensor cores.  For the small-batch learn steps of the BatchNorm policy
                                   nets, whose backward cancels the dominant part of the gradient (csrc/mlp.cu `simt`) */
#define RLCTR_MLP_W_PRESPLIT 16 /* bwd: `ws` is the workspace the forward call of this layer ran with (same batch / dims / flags, weights
                                 * unchanged since): the (W_hi, W_lo) images it left there feed the dgrad GEMM, the split kernel is skipped.
                                 * Only meaningful where the forward took the 3xTF32 path (not RLCTR_MLP_FP32, out_dim > 1). */
size_t rlctr_mlp_ws_bytes(int64_t batch, int32_t in_dim, int32_t out_dim);
/* ---- replay memory of the RL agents, sampled on the device (SURVEY 8f.4) ----------------------------------------------------
 * The reference samples on the host: random.sample (DDQN_model.py:183-185) and np.random.choice(n, batch, p=P, replace=False)
 * after a D2H copy of every priority (v10_Hybrid_TD3_model_PER.py:62-85).  Randomness here: the counter hash under rng_state
 * (device {seed, counter}; advance it with rlctr_rng_advance by the number the call consumed: 1 for uniform, n_valid for PER).
 *   store   memory[(counter + i) % memory_size, :] = src[i, :]  (Memory.add :44-60 / store_transition DDQN_model.py:105-120)
 *   gather  out[i, :] = memory[idx[i], :];   update  priorities[idx[i] * ld] = td[i]  (batch_update :107-108)
 *   sample_uniform  `batch` DISTINCT indices of [0, n_valid): images of 0..batch-1 under a keyed permutation (random.sample)
 *   sample_per      greedy == 0: weighted sampling without replacement, w_i = (|priorities[i*ld]| + eps)^alpha
 *                   (stochastic_sample :62-85; exponential clocks -log(u_i)/w_i, the `batch` smallest);
 *                   greedy != 0: the `batch` largest raw priorities[i*ld] (greedy_sample :87-105).
 *                   out_isw[i] = (p_i / min_j p_j)^(-beta), p = w (stochastic) or the raw priority (greedy), j over [0, n_valid). */
int rlctr_replay_store(float* memory, int64_t memory_size, int32_t width, int64_t counter, const float* src, int64_t n,
                       int64_t ld_src, rlctr_stream_t stream);
int rlctr_replay_gather(const float* memory, int32_t width, const int64_t* idx, int64_t n, float* out, rlctr_stream_t stream);
int rlctr_replay_update(float* priorities, int32_t ld, const int64_t* idx, const float* td, int64_t n, rlctr_stream_t stream);
int rlctr_replay_sample_uniform(int64_t n_valid, int64_t batch, const uint64_t* rng_state, int64_t* out_idx, rlctr_stream_t stream);
size_t rlctr_replay_per_ws_bytes(int64_t n_valid);
int rlctr_replay_sample_per(const float* priorities, int32_t ld, int64_t n_valid, float eps, float alpha, float beta, int32_t greedy,
                            int64_t batch, const uint64_t* rng_state, int64_t* out_idx, float* out_isw, void* ws, size_t ws_bytes,
                            rlctr_stream_t stream);

/* Generalised advantage estimate of the PPO agent (Hybrid_PPO_model.py:206-212): the reference's reversed Python loop with a
 * host synchronisation per sample, as one fp64 scan:  adv = 0; for i, d in enumerate(reversed(deltas)): adv = c*adv + d;
 * advantages[i] = adv  (c = gamma * lambda; advantages[i] belongs to sample n-1-i, as written in the reference). */
size_t rlctr_gae_ws_bytes(int64_t n);
int rlctr_gae_scan(const float* deltas, int64_t n, double gamma_lambda, float* advantages, void* ws, size_t ws_bytes,
                   rlctr_stream_t stream);

/* Dropout mask: keep(element i) = r16(rng_state[0] (seed), rng_state[1] (counter) + i) >= p * 2^16, i = row * out_dim + col
 * (16 random bits per element, two elements per 32-bit hash: csrc/common.cuh).
 * rng_state is DEVICE memory so that a captured CUDA graph draws a new mask on every replay; rlctr_rng_advance moves the
 * counter (call it with batch * out_dim after each forward that used the state).  The mask is not stored: the backward
 * recovers it from the saved output (y == 0 <=> clipped by ReLU or dropped; gy_scale = 1 / (1-p)). */
int rlctr_rng_advance(uint64_t* rng_state, uint64_t delta, rlctr_stream_t stream);
int rlctr_linear_fwd(const float* x, int64_t ldx, const float* w, const float* bias, float* y, int64_t batch,
                     int32_t in_dim, int32_t out_dim, int32_t flags, float dropout_p, const uint64_t* rng_state,
                     void* ws, size_t ws_bytes, rlctr_stream_t stream);
/* RLCTR_MLP_RELU: gy <- gy * (y > 0 ? gy_scale : 0) in place first.  RLCTR_MLP_DX_MASK: see above (x is the mask source). */
int rlctr_linear_bwd(const float* x, int64_t ldx, const float* w, const float* y, float* gy, float* dx, float* dw,
                     float* db, int64_t batch, int32_t in_dim, int32_t out_dim, int32_t flags, float gy_scale,
                     float dx_scale, void* ws, size_t ws_bytes, rlctr_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Multi-GPU row sharding (no counterpart in the reference, which is single-device: SURVEY section 8e).
 * owner(id) = id mod world, local_row(id) = id div world.  Groups the n ids of a local batch by
 * owner, stably:
 *   send_local[k]   local row (at its owner) of the k-th element of the send buffer (-1: out of range)
 *   send_slots[k]   position in `ids` of that element
 *   pos_of_slot[i]  position in the send buffer of ids[i]   (the inverse permutation, int64 so it can be
 *                   fed back as the `ids` of rlctr_embed_fwd over the received rows)
 *   bucket_ends[o]  end offset of owner o's bucket in the send buffer, -1 if the bucket is empty
 * The all-to-all exchanges themselves are NCCL calls made by the host on these buffers.
 * ------------------------------------------------------------------------------------ */
size_t rlctr_bucket_ws_bytes(int64_t n, int32_t world);
int rlctr_bucket_by_owner(const int64_t* ids, int64_t n, int32_t world, int64_t n_rows, int64_t* send_local,
                          int64_t* pos_of_slot, uint32_t* send_slots, int64_t* bucket_ends, void* ws,
                          size_t ws_bytes, rlctr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RLCTR_H_ */
