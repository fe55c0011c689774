/* vlnimagine.h - C ABI of libvlnimagine.so: the sm_100a kernels behind the VLN-Imagine
 * navigation hot path (DUET GlocalTextPathNavCMT / HAMT NavCMT).
 *
 * The reference (akhilperincherry/VLN-Imagine) is 100% PyTorch and has no FFI layer; the seam
 * is the nn.Module the agents hold as `self.vln_bert`.  Each entry point below replaces a group
 * of ATen ops that the reference module issues (cited as reference file:line, paths relative to
 * VLN-DUET/map_nav_src/ = D/ and VLN-HAMT/finetune_src/ = H/).  The Python host modules in
 * vln-imagine_b200/ bind these with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (PyTorch); the library never
 *    allocates device memory and borrows pointers only for the asynchronous launch on `stream`;
 *  - activations are row-major [rows, ld] with ld in ELEMENTS; hidden size is 768, 12 heads of 64;
 *  - return value: VI_OK or a negative VI_ERR_*; vi_last_error() gives the thread-local message;
 *    nothing throws or exits across the ABI;
 *  - re-entrant; no global mutable state besides per-process immutable driver entry points.
 */
#ifndef VLNIMAGINE_H_
#define VLNIMAGINE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VI_OK 0
#define VI_ERR_ARG (-1)
#define VI_ERR_CUDA (-2)
#define VI_ERR_UNSUPPORTED (-3)

#define VI_HIDDEN 768
#define VI_HEAD_DIM 64

enum { VI_DT_BF16 = 0, VI_DT_F32 = 1, VI_DT_F16 = 2 };
enum { VI_EPI_NONE = 0, VI_EPI_GELU = 1, VI_EPI_RELU = 2 };
/* key padding: additive (1-m)*-10000 (D/models/ops.py:25-34) or -inf (nn.MultiheadAttention
 * key_padding_mask, D/models/transformer.py:176-177) */
enum { VI_MASK_ADD_NEG10000 = 0, VI_MASK_NEG_INF = 1 };

typedef void* vi_stream_t; /* cudaStream_t */

int vi_version(void);
const char* vi_last_error(void);
/* Select the device, resolve cuTensorMapEncodeTiled, raise the dynamic shared-memory limits. */
int vi_init(int device);

/* ---------------------------------------------------------------------------------------------
 * Dense contractions.  Replaces nn.Linear (aten::addmm) at D/models/vilmodel.py:93-95,147,172,186,
 * 315-317 and H/models/vilmodel_cmt.py (same blocks), plus the fused epilogues that follow them:
 * erf-GELU (:32-38), ReLU (ClsPrediction :1014), residual add (transformer.py:178,181).
 *
 *   Y[r, n] = epi( sum_k X[r,k] * W[g(r)*N + n, k] + bias[g(r)*N + n] ) + residual[r, n]
 *
 * Grouped form: rows are split into n_groups consecutive row ranges ending at group_row_end[g]
 * (HOST array; every group but the last must end on a multiple of 128 rows); group g uses rows
 * [g*N, (g+1)*N) of W / bias.  n_groups == 1 and group_row_end == NULL is the plain GEMM.
 * vi_gemm16   : X, W 16-bit; fp32 accumulation in TMEM (tcgen05.mma fed by TMA).  K % 64 == 0, N % 64 == 0, ldx % 8 == 0.
 *               y_dtype selects a 16-bit (in_dtype) or an fp32 output.
 * vi_gemm_f32 : the fp32 check mode (FFMA, no tensor cores); X, W, Y fp32.
 * bias / residual may be NULL.  residual is fp32 [M, ldr] and requires an fp32 output in vi_gemm16.
 * Operands of either 16-bit format: bf16, or fp16 for tensors whose range the caller has bounded (LayerNorm outputs,
 * probabilities, their projections - same tensor-core rate, 8x smaller rounding error; 16-bit outputs saturate at +-65504
 * instead of overflowing).  Optionally a 16-bit copy of an fp32 output, and LayerNorm folded into the neighbouring
 * contractions so that BertSelfOutput / BertOutput (D/models/vilmodel.py:151-155, 190-194) and norm1 / norm2 of the panorama
 * encoder (D/models/transformer.py:171,179) need no pass of their own:
 *   stats_out  : the producer (dense + residual) writes, for every output row and every 32-column chunk, (mean, M2) of the
 *                chunk: float2 [N / 32][stats_ld].  Its fp32 output is the RAW pre-LayerNorm sum z (plus y16 = z in 16 bits).
 *   VI_LN_FOLD : the consumer computes LayerNorm(z) W^T + b from z itself:  x = z in 16 bits, w = W * gamma (columnwise),
 *                bias = W beta + b, ln_vec_a = row sums of w; the epilogue applies  y = (acc - mu * s_n) / sigma + bias_n
 *                with (mu, sigma) of each row combined from ln_stats (ln_chunks chunks, Chan's formula), then the activation.
 *   VI_LN_RESIDUAL : the residual operand is LayerNorm(z) given as the RAW fp32 rows z: the epilogue adds
 *                (z - mu) / sigma * gamma + beta with ln_vec_a = gamma and bias = beta + b ([n_groups * N], N = 32 * ln_chunks;
 *                no activation).
 * Grouped calls index bias / ln_vec_* as [g * N + n].
 * tile: 0 = the library's own cost model, or the output-tile shape chosen by the caller: width (64, 96, 128, 192, 256)
 * dividing N, optionally | VI_TILE_PAIR for the two-CTA (cta_group::2, 256-row) form, which needs width >= 128 and every
 * group but the last ending on a multiple of 256 rows; any other request is VI_ERR_ARG.  Results do not depend on the tile
 * (the K accumulation order is the same).
 * ------------------------------------------------------------------------------------------- */
#define VI_TILE_PAIR 0x1000
enum { VI_LN_NONE = 0, VI_LN_FOLD = 1, VI_LN_RESIDUAL = 2 };
typedef struct {
  const void* x; int64_t ldx;      /* [M, K] 16-bit */
  const void* w;                   /* [n_groups * N, K] 16-bit, same format as x */
  int in_dtype;                    /* VI_DT_BF16 or VI_DT_F16 */
  const float* bias;               /* [n_groups * N] or NULL */
  const float* residual; int64_t ldr;   /* fp32 [M, ldr] or NULL */
  void* y; int64_t ldy; int y_dtype;    /* primary output: in_dtype or VI_DT_F32 */
  void* y16; int64_t ldy16;        /* optional 16-bit copy (in_dtype) of an fp32 output, or NULL */
  int M, N, K, epilogue;
  int n_groups; const int32_t* group_row_end;   /* HOST array */
  int tile;                        /* 0 (cost model) or width | VI_TILE_PAIR */
  int ln_mode;                     /* VI_LN_* */
  const float* ln_vec_a;
  const float* ln_stats;           /* float2 [ln_chunks][stats_ld] written by the producer of the rows being normalised */
  int ln_chunks; float ln_eps;
  float* stats_out;                /* float2 [N / 32][stats_ld] or NULL */
  int64_t stats_ld;                /* row stride (in float2) of ln_stats and stats_out, >= M */
} vi_gemm_args;
int vi_gemm16(const vi_gemm_args* args, vi_stream_t stream);
int vi_gemm_f32(const float* x, int64_t ldx, const float* w, const float* bias,
                const float* residual, int64_t ldr, float* y, int64_t ldy,
                int M, int N, int K, int epilogue,
                int n_groups, const int32_t* group_row_end, vi_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fused masked multi-head attention (scores never reach HBM).  Replaces
 * matmul/div/add-mask/softmax/matmul at D/models/vilmodel.py:118-134 (BertSelfAttention),
 * :336-349 (BertOutAttention), the GASA bias add at :392-394 and nn.MultiheadAttention in the
 * panorama encoder (D/models/transformer.py:176-177).
 *   q: [B*Lq, ldq], k/v: [B*Lk, ldk/ldv], head h at columns [h*64, h*64+64); o: [B*Lq, ldo].
 *   key_mask [B, Lk] (1 = valid) or NULL; pair_dist [B, Lq, Lk] fp32 or NULL with
 *   bias_affine -> device {w, b}: bias = w*dist + b (sprel_linear, D/models/vilmodel.py:1145-1149).
 *   dtype: VI_DT_BF16 / VI_DT_F16 (tensor-core tiles, fp32 softmax) or VI_DT_F32 (check mode).
 *   lse [B, H, Lq] optional (log-sum-exp per row, kept for the backward pass).
 * ------------------------------------------------------------------------------------------- */
#define VI_ATTN_MAX_PROBLEMS 4
typedef struct {
  const void* q; int64_t ldq;
  const void* k; int64_t ldk;
  const void* v; int64_t ldv;
  void* o; int64_t ldo;
  const uint8_t* key_mask;     /* [B, Lk] or NULL */
  const float* pair_dist;      /* [B, Lq, Lk] or NULL */
  const float* bias_affine;    /* device {w, b} */
  float* lse;                  /* [B, H, Lq] or NULL */
  int32_t B, Lq, Lk;
  float drop_p;                /* attention-probability dropout (training only); 0 = none */
  uint32_t drop_site;          /* dropout site id (see vi_dropout) */
  const uint32_t* drop_seed;   /* device pointer to the dropout seed, or NULL */
} vi_attn_problem;
/* Several independent attention problems (token streams of one row-stacked activation: DUET global | local,
 * HAMT language | vision) in ONE launch; a single problem is n_problems == 1.  16-bit inference shapes (<= 96 keys, no
 * dropout, no lse) run a single-pass kernel; dropout, lse or more keys run the generic mma.sync kernel. */
int vi_attn_fwd_multi(const vi_attn_problem* problems, int n_problems, int H, int dtype, int mask_mode,
                      vi_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Row kernels (one warp per 768-wide row, fp32 statistics, 16-byte accesses).
 * ------------------------------------------------------------------------------------------- */
/* y = LayerNorm(a [+ b]) * gamma + beta.  BertSelfOutput/BertOutput (D/models/vilmodel.py:151-155,
 * 190-194), norm1/norm2/final norm of the panorama encoder (D/models/transformer.py:171,179,86).
 * Writes fp32 (y32) and/or 16-bit (y16: VI_DT_BF16 or VI_DT_F16 per y16_dtype, as everywhere below) copies; either may be
 * NULL.  Grouped form as in vi_gemm_*: rows below group_row_end[g] (HOST array, ascending) use gamma/beta rows g of a
 * [n_groups, 768] stack. */
int vi_add_ln(const float* a, const float* b, const float* gamma, const float* beta, float eps,
              float* y32, void* y16, int y16_dtype, int64_t rows,
              int n_groups, const int32_t* group_row_end, vi_stream_t stream);

/* Input-embedding composer:
 *   y = LN_out( [LN_a](a) + a2 + a3 + LN_f(feat @ feat_w^T + feat_b) + table[idx] + pos_table[row % pos_period]
 *               + const_row + const_row2 )
 * every term optional.  Covers BertEmbeddings (D/models/vilmodel.py:49-78), the panorama /
 * observation embeddings (D/models/vilmodel.py:1091-1121, H/models/vilmodel_cmt.py:521-544),
 * history embeddings (H/...:576-612), gmap/vp input embeddings (D/...:1141-1152) and the
 * imagination type embedding (D/...:562-573). */
typedef struct {
  const float* a;            /* [rows, 768] or NULL */
  const float* a_gamma;      /* LayerNorm over a (NULL: add a as is) */
  const float* a_beta;
  const float* feat;         /* [rows, feat_dim] small geometric features or NULL (feat_dim <= 16) */
  int32_t feat_dim;
  const float* feat_w;       /* [feat_dim, 768]: the TRANSPOSE of nn.Linear(feat_dim, 768).weight (16-byte aligned) */
  const float* feat_b;       /* [768] */
  const float* feat_gamma;   /* LayerNorm over the projected features (NULL: none) */
  const float* feat_beta;
  const int64_t* idx;        /* [rows] row ids into table, or NULL */
  const float* table;        /* [*, 768] */
  const float* pos_table;    /* [>=pos_period, 768] or NULL: adds pos_table[row % pos_period] */
  int32_t pos_period;
  const float* const_row;    /* [768] or NULL */
  const float* const_row2;   /* [768] or NULL */
  const float* out_gamma;    /* final LayerNorm (NULL: none) */
  const float* out_beta;
  float eps;                 /* all LayerNorms here use the same eps (1e-12 in the reference) */
  float* y32;                /* [rows, 768] or NULL */
  void* y16;                 /* 16-bit [rows, 768] or NULL */
  int64_t rows;
  const float* a2;           /* [rows, 768] plain addends (NULL: none); used by the training-mode decomposition */
  const float* a3;
  int32_t y16_dtype;         /* VI_DT_BF16 or VI_DT_F16 */
  const float* ln2_gamma;    /* optional second LayerNorm chained on the result: y32 keeps the first result, y16 = LN2(y32) */
  const float* ln2_beta;     /* (norm1 of the first pre-norm panorama layer, D/models/transformer.py:171) */
  float ln2_eps;
  int64_t zero_rows;         /* rows [rows, rows + zero_rows) of y32 / y16 are zero-filled (the padding up to the next stream of a
                              * row-stacked activation: it flows through the following GEMMs and must stay finite) */
} vi_embed_args;
/* PARAMETER operands (feat_w, feat_b, the LayerNorm vectors, const_row / const_row2) are touched at the top of the kernel,
 * ahead of the programmatic-dependent-launch wait, to have them in L1 when the rows arrive: they must not be outputs of another
 * kernel of THIS library launched just before on the same stream (outputs of any other kernel, or of an earlier synchronised
 * launch, are fine; VI_PDL=0 removes the constraint).  Row operands (a, a2, a3, feat, idx, table, pos_table) have no such rule. */
int vi_embed_compose(const vi_embed_args* args, vi_stream_t stream);

/* out[row] = LayerNorm(h[row]) . w + b   (tail of ClsPrediction / NextActionPrediction:
 * D/models/vilmodel.py:1009-1020, H/models/vilmodel_cmt.py:953-963).  Grouped like vi_add_ln:
 * gamma/beta/w are [n_groups, 768] stacks and b is [n_groups].  gamma == beta == NULL: no LayerNorm, out[row] = h[row] . w + b
 * (the training forward keeps the normalised rows and applies the dot product on its own). */
int vi_ln_dot(const float* h, const float* gamma, const float* beta, float eps,
              const float* w, const float* b, float* out, int64_t rows,
              int n_groups, const int32_t* group_row_end, vi_stream_t stream);

/* y[b*rpb + r] = x[b*x_batch_stride + r*768 ..] * s[b*lds ..]  (ob_embeds * txt_embeds[:, :1],
 * H/models/vilmodel_cmt.py:1191; ob_embeds is the tail slice of every episode's [hist; ob] block, hence the
 * batch stride).  Strides in elements; y rows are dense. */
int vi_mul_bcast(const float* x, int64_t x_batch_stride, const float* s, int64_t lds, float* y32, void* y16, int y16_dtype,
                 int64_t rows, int rows_per_batch, vi_stream_t stream);

/* Action-logit masking and global/local fusion, D/models/vilmodel.py:1182-1217.
 *   fuse = sigmoid(fuse_raw[b]) (0.5 when fuse_raw == NULL: sap_fuse_linear is None);
 *   global = g_raw*fuse, -inf at visited|padded nodes; local = l_raw*(1-fuse), -inf at non-navigable views;
 *   fused = global; fused[b,0] += local[b,0]; for every node j>0 whose id is not in the visited set:
 *   += local[b, v] of the (last) unvisited candidate v>0 with the same id, else += the sum of local[b, v]
 *   over visited candidates v>0 (ascending v).
 * gmap_ids [B,G] / cand_ids [B,P] are the viewpoint-id strings of gmap_vpids / vp_cand_vpids interned to
 * int32 on the host (padding: -1 in gmap_ids, -2 in cand_ids); the visited set is derived on the device
 * from gmap_visited, which replaces the reference's per-sample Python dict look-ups. */
int vi_duet_fuse_logits(const float* g_raw, const float* l_raw, const float* fuse_raw,
                        const uint8_t* gmap_masks, const uint8_t* gmap_visited, const uint8_t* vp_nav_masks,
                        const int32_t* gmap_ids, const int32_t* cand_ids,
                        float* global_logits, float* local_logits, float* fused_logits,
                        int B, int G, int P, vi_stream_t stream);

/* act_logits.masked_fill_(ob_nav_types == 0, -inf)  (H/models/vilmodel_cmt.py:1200) */
int vi_mask_logits_navtype(const float* raw, const int64_t* nav_types, float* out, int64_t n, vi_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Imagination <-> noun-phrase alignment (aux loss), D/models/vilmodel.py:598-655 and 657-779.
 * ------------------------------------------------------------------------------------------- */
/* out[r] = mean over t in [offsets[r], offsets[r+1]) of src[row_idx[t]]  (768-wide rows) */
int vi_gather_mean(const float* src, const int32_t* offsets, const int32_t* row_idx,
                   float* out32, void* out16, int out16_dtype, int R, vi_stream_t stream);
/* dst[dst_rows[r]] = src[r] */
int vi_scatter_rows(const float* src, const int32_t* dst_rows, float* dst, int R, vi_stream_t stream);
/* loss_rows[r] = 1 - cos(proj[r], tgt[r]) (eps 1e-8); *loss_mean = mean_r (0 if R == 0) */
int vi_cosine_loss(const float* proj, const float* tgt, float* loss_rows, float* loss_mean,
                   int R, vi_stream_t stream);
/* InfoNCE: logits_r = cos(proj[r], [tgt[r]; negs[n] for neg_episode[n] != row_episode[r]]) / T,
 * loss_r = -log softmax(logits_r)[0]; *loss_mean = mean_r.  `scratch` must hold
 * R * (n_negs + 2) floats: the similarity matrix first, then the R per-row losses. */
int vi_infonce_loss(const float* proj, const float* tgt, const float* negs,
                    const int32_t* row_episode, const int32_t* neg_episode,
                    float temperature, float* scratch, float* loss_mean,
                    int R, int n_negs, vi_stream_t stream);
/* margin form of the same alignment loss (aux_loss_type 'constrastive-margin', H/models/vilmodel_cmt.py:825-856, 939-942):
 * (1 - cos(p, t)) + mean over the noun-phrase means of OTHER episodes of relu(margin + cos(p, neg) - cos(p, t)); same operands
 * and scratch layout as vi_infonce_loss.  Forward only. */
int vi_margin_loss(const float* proj, const float* tgt, const float* negs, const int32_t* row_episode,
                   const int32_t* neg_episode, float margin, float* loss_rows, float* loss_mean, int R, int n_negs,
                   vi_stream_t stream);

/* Loss rows of the pre-training proxy tasks (VLN-DUET/pretrain_src/model/pretrain_cmt.py:150 MLM, :198-204 MRC):
 *   vi_ce_rows: out[r] = logsumexp(logits[r, 0:n_cols]) - logits[r, labels[r]]            (F.cross_entropy, reduction 'none')
 *   vi_kl_rows: out[r] = sum_c t[r,c] * (log t[r,c] - log_softmax(logits[r])[c]), t == 0 terms dropped  (F.kl_div(...).sum(1))
 * logits / targets are fp32 row-major with leading dimensions ld / ldt >= n_cols (a padded vocabulary GEMM output). */
int vi_ce_rows(const float* logits, int64_t ld, const int64_t* labels, int n_cols, float* out, int64_t rows, vi_stream_t stream);
int vi_kl_rows(const float* logits, int64_t ld, const float* targets, int64_t ldt, int n_cols, float* out, int64_t rows,
               vi_stream_t stream);
/* Backward of vi_ce_rows / vi_kl_rows (what torch autograd gives for the two losses above), vi_xent.cu:
 *   dx[r, c] = dloss[r] * (softmax(logits[r, 0:n_cols])[c] * T[r] - t[r, c])   for c < n_cols
 *   cross-entropy: t = one-hot(labels[r]), T = 1;  KL: t = targets[r], T = sum_c targets[r, c].
 * dloss: device fp32 [rows], the incoming gradient of each row's loss.  Output rows of ld_out >= n_cols elements as fp32 (dx32)
 * and / or 16-bit (dx16, dx16_dtype VI_DT_BF16 / VI_DT_F16: the operand of the gradient GEMMs); columns n_cols <= c < ld_out are
 * written as exact zeros.  A -inf logit has softmax 0.  rows == 0 is a no-op.  Rows of >= 256 columns with ld % 4 == 0,
 * ld_out % 8 == 0 and 16-byte aligned pointers take a CTA per row (16-byte loads and stores); others a warp per row. */
int vi_ce_rows_bwd(const float* logits, int64_t ld, const int64_t* labels, int n_cols, const float* dloss, float* dx32, void* dx16,
                   int dx16_dtype, int64_t ld_out, int64_t rows, vi_stream_t stream);
int vi_kl_rows_bwd(const float* logits, int64_t ld, const float* targets, int64_t ldt, int n_cols, const float* dloss, float* dx32,
                   void* dx16, int dx16_dtype, int64_t ld_out, int64_t rows, vi_stream_t stream);
/* dst[b, r, 0:768] = src[b, r, 0:768] for n_batches x rows_per_batch rows; strides in ELEMENTS.  Writes an
 * fp32 and/or a 16-bit copy.  Builds the cross-attention context cat([txt_embeds, imagine_embeds], 1)
 * (D/models/vilmodel.py:1157, H/models/vilmodel_cmt.py:1110) and gathers the token-0 rows that feed
 * sap_fuse_linear (D/models/vilmodel.py:1185-1187). */
int vi_copy_rows(const float* src, int64_t src_batch_stride, int64_t src_row_stride, float* dst32, void* dst16,
                 int dst16_dtype, int64_t dst_batch_stride, int64_t dst_row_stride, int64_t n_batches, int rows_per_batch,
                 vi_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Backward pass (fine-tuning).  The dense gradients of the 16-bit path:
 *   dX = dY W  (vi_gemm16 with the [K, N] transposed weight shadow),  dW = dY^T X and db = column sums of dY
 *   (vi_wgrad16, no transposes).  The fp32 check mode computes dW with vi_gemm_f32 on vi_transpose'd dY and X and db with
 *   vi_colsum.  The other entry points below are the adjoints of the remaining forward kernels; each mirrors what
 *   torch.autograd computes for the reference ops it cites.
 * ------------------------------------------------------------------------------------------- */
/* dst[c, r] = src[r, c]; dst is [cols, ldd] with columns rows..pad_rows-1 zero-filled (pad_rows <= ldd) */
int vi_transpose(const void* src, int64_t ld, void* dst, int64_t ldd, int rows, int cols, int pad_rows, int dtype,
                 vi_stream_t stream);
/* Weight and bias gradients of a (grouped) dense layer WITHOUT transposes (vi_wgrad.cu):
 *   dw[g] = dY[g]^T X[g]  ([N, K] fp32, groups stacked: dw is [n_groups * N, K]),   db[g] = column sums of dY[g]  (or NULL)
 * dY [rows, N] and X [rows, K] are row-major 16-bit tensors (dtype VI_DT_BF16 / VI_DT_F16), N % 128 == 0, K % 64 == 0; group g
 * covers rows group_row_end[g-1] .. group_row_end[g].  Both operands reach tcgen05.mma as MN-major tiles exactly as they lie in
 * memory; the contraction (over rows) is split over `splits` work units per output tile (0: the library's choice,
 * vi_wgrad16_splits), whose fp32 partials go through `workspace` (vi_wgrad16_workspace floats) and are summed in a fixed order.
 * accumulate != 0: dw / db are added to (gradient accumulation over the steps of an iteration; one writer per element, so the
 * result does not depend on scheduling).
 * What loss.backward() computes for nn.Linear: grad_weight = grad_output^T input, grad_bias = grad_output.sum(0). */
int vi_wgrad16_splits(int N, int K, int n_groups, const int32_t* group_rows);
int64_t vi_wgrad16_workspace(int N, int K, int n_groups, const int32_t* group_rows, int splits);
int vi_wgrad16(const void* dy, int64_t lddy, const void* x, int64_t ldx, int dtype, int N, int K, int n_groups,
               const int32_t* group_row_end, float* dw, float* db, float* workspace, int64_t workspace_floats, int splits,
               int accumulate, vi_stream_t stream);
/* Column reductions over rows run in two deterministic stages (128-row chunks -> a caller-provided fp32 scratch ->
 * fixed-order sum): n_out * ceil(rows / 128) * cols floats for n_out reduced quantities per column. */
/* out[c] = sum_r x[r, c] (fp32 accumulation, fixed order); bias gradients of nn.Linear.  scratch: n_out = 1 */
int vi_colsum(const void* x, int64_t ld, int dtype, float* out, int64_t rows, int cols, float* scratch,
              int64_t scratch_elems, vi_stream_t stream);
/* y = act(x), dx = dy * act'(x); act = VI_EPI_GELU (erf form, D/models/vilmodel.py:32-38) or VI_EPI_RELU.
 * The training forward keeps the pre-activation, so activations run as their own kernels there. */
int vi_act_fwd(const void* x, void* y, int64_t n, int act, int dtype, vi_stream_t stream);
int vi_act_bwd(const void* x, const void* dy, void* dx, int64_t n, int act, int dtype, vi_stream_t stream);
/* LN(dropout(a) + b) and its adjoint: the hidden dropout of BertSelfOutput / BertOutput (D/models/vilmodel.py:151-155,190-194)
 * applied inside the LayerNorm kernels (mask of vi_dropout for a [rows, 768] tensor at `site`).  p == 0: no dropout, and
 * vi_add_ln_drop_bwd is the adjoint of vi_add_ln.
 * Backward: dy = dy32 (+ dy16); dx32 / dx16 = gradient of b (and of a when p == 0); dxa16 (optional, bf16) = dropout(dx) =
 * gradient of a, the operand of the dense layer's gradient GEMMs - no separate dropout or cast pass (p == 0: the 16-bit copy
 * of dx).  dgamma / dbeta [n_groups, 768] (16-byte aligned) are required; accumulate != 0 adds to them instead of overwriting.
 * stats is a [rows, 2] fp32 scratch (mean, rstd).  scratch: at least 2 * ceil(rows / 32) * 768 floats; with
 * 2 * ceil(rows / 8) * 768 the kernel may use chunks of 8 or 16 rows (more CTAs for the short streams of this path; the
 * summation order, hence the last bits of dgamma / dbeta, follows the chunk). */
int vi_add_ln_drop(const float* a, const float* b, const float* gamma, const float* beta, float eps, float* y32, void* y16,
                   int y16_dtype, int64_t rows, int n_groups, const int32_t* group_row_end, float p, const uint32_t* seed,
                   uint32_t site, vi_stream_t stream);
int vi_add_ln_drop_bwd(const float* a, const float* b, const float* gamma, float eps, const float* dy32, const void* dy16,
                       float* dx32, void* dx16, void* dxa16, float* dgamma, float* dbeta, float* stats, int64_t rows,
                       int n_groups, const int32_t* group_row_end, float* scratch, int64_t scratch_elems, int accumulate,
                       float p, const uint32_t* seed, uint32_t site, vi_stream_t stream);
/* small-feature linear of vi_embed_compose: dW[768, feat_dim] = dt^T feat, db[768] = colsum(dt) */
int vi_feat_wgrad(const float* dt, const float* feat, int feat_dim, float* dW, float* db, int64_t rows, float* scratch,
                  int64_t scratch_elems, vi_stream_t stream);
/* dst[idx[r]] += src[r] (idx != NULL) or dst[r % period] += src[r]: embedding / position table adjoints */
int vi_scatter_add_rows(const float* src, const int64_t* idx, int period, float* dst, int64_t rows, vi_stream_t stream);
/* adjoint of the dot-product tail of vi_ln_dot (out[r] = x[r] . w[g] + b[g]) */
int vi_rowdot_bwd(const float* dout, const float* x, const float* w, float* dx, float* dw, float* db_cols, int64_t rows,
                  int n_groups, const int32_t* group_row_end, float* scratch, int64_t scratch_elems, vi_stream_t stream);
/* attention backward for one token stream (same operand conventions as one vi_attn_problem); d_affine -> device {dw, db}
 * of the GASA affine, accumulated (+=); dq / dk / dv have the dtype of q / k / v. */
int vi_attn_bwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                const void* dout, int64_t ldo, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv,
                int dtype, const uint8_t* key_mask, const float* pair_dist, const float* bias_affine, float* d_affine,
                int B, int H, int Lq, int Lk, int mask_mode, float drop_p, uint32_t drop_site, const uint32_t* drop_seed,
                vi_stream_t stream);
/* adjoint of vi_duet_fuse_logits; any of d_global / d_local / d_fused may be NULL (treated as zero) */
int vi_duet_fuse_logits_bwd(const float* g_raw, const float* l_raw, const float* fuse_raw,
                            const uint8_t* gmap_masks, const uint8_t* gmap_visited, const uint8_t* vp_nav_masks,
                            const int32_t* gmap_ids, const int32_t* cand_ids,
                            const float* d_global, const float* d_local, const float* d_fused,
                            float* dg_raw, float* dl_raw, float* dfuse_raw, int B, int G, int P, vi_stream_t stream);
/* adjoint of vi_mul_bcast w.r.t. the broadcast row s: ds[b, :] = sum_r dy[b, r, :] * x[b, r, :] (contiguous [B, rows, 768];
 * the gradient w.r.t. x is vi_mul_bcast(dy, s)).  HAMT act_pred_token 'ob_txt' (H/models/vilmodel_cmt.py:1191). */
int vi_mul_bcast_bwd_s(const float* dy, const float* x, float* ds, int64_t n_batches, int rows_per_batch, vi_stream_t stream);
/* adjoint of vi_cosine_loss: dloss is the device scalar gradient of the mean; dproj / dtgt may be NULL */
int vi_cosine_loss_bwd(const float* proj, const float* tgt, const float* dloss, float* dproj, float* dtgt, int R,
                       vi_stream_t stream);
/* adjoint of vi_infonce_loss w.r.t. proj (the noun-phrase means are constants under fix_lang_inside_cosine_model,
 * D/models/vilmodel.py:1249-1255); `sims` = the first R * (n_negs + 1) floats the forward call left in its loss_rows scratch */
int vi_infonce_loss_bwd(const float* proj, const float* tgt, const float* negs, const int32_t* row_episode,
                        const int32_t* neg_episode, float temperature, const float* sims, const float* dloss,
                        float* dproj, int R, int n_negs, vi_stream_t stream);
/* adjoint of vi_margin_loss w.r.t. proj (H/models/vilmodel_cmt.py:825-856); `sims` = the cosines the forward call left in its
 * loss_rows scratch */
int vi_margin_loss_bwd(const float* proj, const float* tgt, const float* negs, const int32_t* row_episode,
                       const int32_t* neg_episode, float margin, const float* sims, const float* dloss,
                       float* dproj, int R, int n_negs, vi_stream_t stream);

/* Dropout (training only): y = x * keep / (1 - p) with keep(i) = hash(i, *seed, site) >= p * 2^32; the backward pass is the
 * same call on the gradient.  `seed` is a device pointer (the host module advances it once per optimiser step, also inside
 * replayed CUDA graphs); `site` distinguishes the dropout layers of one iteration.  nn.Dropout of BertEmbeddings /
 * BertSelfOutput / BertOutput (D/models/vilmodel.py:77,153,192), ImageEmbeddings (:1124), the panorama encoder layers
 * (D/models/transformer.py:178-181), MLPProjectionHead (:585) and VLNBert.drop_env (D/models/model.py:27). */
int vi_dropout(const void* x, void* y, int64_t n, float p, const uint32_t* seed, uint32_t site, int dtype, vi_stream_t stream);

/* fp32 -> bf16 or fp16 (saturating at +-65504): 16-bit shadow copies of weights and activations */
int vi_cast_h16(const float* src, void* dst, int dst_dtype, int64_t n, vi_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Per-step graph glue of a DUET rollout (SURVEY.md section 8(f), rows N1 / N2).  Replaces the Python GraphMap /
 * FloydGraph objects (D/models/graph_utils.py:42-148) and the agent's per-step collate loops
 * (D/r2r/agent.py:98-207, 466-479) by dense per-episode arrays in HBM, caller-owned:
 *   pos f64 [B,N,3]   dis f64 [B,N,N] (95959595 = never reached, graph_utils.py:44)   point i32 [B,N,N] (-1 = direct edge)
 *   visited u8 [B,N]  esum f32 [B,N,H]   ecnt f32 [B,N]
 * Node indices are the order in which viewpoints entered GraphMap.node_positions (the host interns the id strings);
 * -1 marks the [stop] slot / padding.  fp64 state: distances, path lengths and the distance features are bit-identical
 * to the reference's Python-float arithmetic; sin / cos of the fp32-cast angles agree to 1 ulp. */
int vi_graph_init(double* dis, int32_t* point, uint8_t* visited, float* ecnt, int B, int N, vi_stream_t stream);
/* GraphMap.update_graph (graph_utils.py:109-115): positions, add_edge (:53-58) to every candidate of the current
 * viewpoint, FloydGraph.update(k) (:60-70).  cur_node[b] = -1 leaves episode b untouched (ended, agent.py:601-603);
 * n_nodes[b] = nodes known after this update; cand_node [B,C] padded with -1. */
int vi_graph_update(double* pos, double* dis, int32_t* point, uint8_t* visited, int B, int N, const int32_t* cur_node,
                    const double* cur_pos, const int32_t* cand_node, const double* cand_pos, int C,
                    const int32_t* n_nodes, vi_stream_t stream);
/* agent.py:466-479: masked mean of pano_embeds [B,V,H] rewrites the current node, each UNVISITED candidate view j < C
 * adds pano_embeds[b,j] to its node (GraphMap.update_node_embed, graph_utils.py:117-126); then (agent.py:125-129,
 * 176-178) gmap_img_embeds[b,g] = esum / ecnt of gmap_node[b,g] (zeros for -1) and vp_img_embeds = [0 ; pano_embeds]
 * ([B,V+1,H]); either output may be NULL.  cur_node[b] = -1 skips the update of an ended episode. */
int vi_graph_embed_step(const float* pano_embeds, const uint8_t* pano_masks, int B, int V, int H, const int32_t* cur_node,
                        const int32_t* cand_node, int C, const uint8_t* visited, float* esum, float* ecnt, int N,
                        const int32_t* gmap_node, int G, float* gmap_img_embeds, float* vp_img_embeds, vi_stream_t stream);
/* GraphMap.get_pos_fts (graph_utils.py:14-40,131-148) for the gmap slots ([B,G,7], zero beyond gmap_lens[b]) and the
 * candidate views (vp_pos_fts [B,P,14] = start-viewpoint features | candidate features in rows 1..C, agent.py:182-196);
 * gmap_pair_dists [B,G,G] raw metres with zero row / column 0 and diagonal (agent.py:137-141).  Outputs may be NULL. */
int vi_graph_features(const double* pos, const double* dis, const int32_t* point, int B, int N, const int32_t* cur_node,
                      const double* heading, const double* elevation, const int32_t* gmap_node, const int32_t* gmap_lens,
                      int G, float* gmap_pos_fts, float* gmap_pair_dists, const int32_t* cand_node, int C,
                      const int32_t* start_node, int P, float* vp_pos_fts, vi_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VLNIMAGINE_H_ */
