/* clipk - C ABI of the B200 (sm_100a) fused contrastive-loss library.
 *
 * This is the drop-in boundary for the ClipLoss / gather_features hot path of chen-yy20/Megatron-CLIP.
 * The reference has no native interface for this path: it is a chain of PyTorch library calls made from
 * open_CLIP/src/open_clip/loss.py.  Each entry point below names the reference lines it replaces; the host
 * side that keeps the reference's Python signatures lives in megatron-clip_b200/clipk/loss.py and binds these
 * symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (PyTorch's caching allocator); the library
 *    allocates nothing persistent and never synchronises the device;
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it;
 *  - return value: 0 = ok, < 0 = CLIPK_E* below, > 0 = a cudaError_t; clipk_last_error() gives a
 *    thread-local description.  The library never throws and never aborts;
 *  - there is no CPU path and no other GPU architecture: on anything but compute capability 10.x every
 *    compute entry returns CLIPK_EARCH.
 *  - matrices are row-major with a leading dimension in ELEMENTS; dtype is the element type of X and Y.
 *
 * Math.  For a block of `rows` local rows X [rows, d] against `cols` columns Y [cols, d],
 *   S = logit_scale * X * Y^T   (never stored),  the positive of row i is column diag_offset + i.
 */
#ifndef CLIPK_H_
#define CLIPK_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CLIPK_VERSION 2

#define CLIPK_OK 0
#define CLIPK_EINVAL (-1)       /* bad argument (null pointer, non-positive size, misaligned pointer or ld) */
#define CLIPK_EUNSUPPORTED (-2) /* shape or dtype the kernels do not handle (d % 8 != 0, ...) */
#define CLIPK_EARCH (-3)        /* current device is not compute capability 10.x */
#define CLIPK_EWORKSPACE (-4)   /* workspace smaller than clipk_*_workspace_bytes() */
#define CLIPK_EDRIVER (-5)      /* cuTensorMapEncodeTiled unavailable or failed */

#define CLIPK_BF16 0  /* bf16 [rows, d] */
#define CLIPK_F32 1   /* fp32; only a source type of clipk_to_f16 and a destination type of clipk_cast */
#define CLIPK_F16 3   /* scaled fp16, one plane  [rows, round_up(d, 64)], zero padded: value = stored * inv_scale */
#define CLIPK_F16X2 4 /* scaled fp16, two planes [rows, 2 * round_up(d, 64)] = [hi | lo]: value = (hi + lo) * inv_scale.
                         The kernels contract the three plane pairs lo.hi, hi.lo, hi.hi, which reproduces an fp32
                         product to ~2^-22 on the 16-bit tensor pipe. */

int clipk_version(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
long long clipk_launch_count(void);
const char* clipk_last_error(void);

/* 0 when the current CUDA device can run the kernels (CC 10.x), CLIPK_EARCH otherwise. */
int clipk_check_device(void);

/* [rows, d] bf16 or fp32 (src_dtype, ld_src) -> CLIPK_F16 (planes = 1) or CLIPK_F16X2 (planes = 2) in dst, with
 * ld_dst == planes * round_up(d, 64).  The power-of-two scale maps max|x| into [2^13, 2^14).  scale_io is two device
 * floats: [0] scratch, [1] receives inv_scale.  bf16 -> one fp16 plane is exact (8 significant bits fit in 11); it
 * feeds the gradient GEMMs, whose other operand (the softmax gradient G) needs more mantissa than bf16 has.
 * fp32 -> two planes replaces the fp32 matmul of loss.py:112-119 when autocast is off. */
int clipk_to_f16(const void* src, int src_dtype, long long rows, long long d, long long ld_src, void* dst, int planes,
                 long long ld_dst, float* scale_io, void* stream);
/* same with max |x| already known (a device float, finite and from the same data) */
int clipk_to_f16_amax(const void* src, int src_dtype, long long rows, long long d, long long ld_src, void* dst, int planes,
                      long long ld_dst, float* scale_io, const float* amax, void* stream);

/* ---- forward ------------------------------------------------------------------------------------------
 * clipk_fwd_stats replaces, for one direction, the logits GEMM and the log-softmax reduction of
 *   loss.py:112-113 / 115-116 / 118-119 (logit_scale * a @ b.T) and loss.py:135-138 (F.cross_entropy)
 * without materialising the [rows, cols] logits: it returns, per row i,
 *   row_max[i] = max_j S_ij,
 *   row_sum[i] = sum_j exp(S_ij - row_max[i]),
 *   row_dot[i] = sum_j exp(S_ij - row_max[i]) * S_ij      (gives dloss/dlogit_scale without a backward pass over S)
 *   pos_logit[i] = S[i, diag_offset + i]   (written only when that column exists; may be NULL).
 * Calling it with X and Y swapped gives the statistics of the other direction (logits_per_text).
 * dtype: CLIPK_BF16, CLIPK_F16 or CLIPK_F16X2 for both operands; x/y_inv_scale are device scalars (NULL = 1).
 */
size_t clipk_fwd_workspace_bytes(int rows, int cols, int d, int dtype);
int clipk_fwd_stats(const void* X, const void* Y, int rows, int cols, int d, long long ldx, long long ldy, int dtype,
                    const float* x_inv_scale, const float* y_inv_scale, const float* logit_scale,
                    long long diag_offset, float* row_max, float* row_sum, float* row_dot, float* pos_logit,
                    void* workspace, size_t workspace_bytes, void* stream);

/* clipk_fwd_both: the statistics of BOTH directions of the same block - what two clipk_fwd_stats calls (X against Y,
 * then Y against X) return - as row_stats [3][rows] and col_stats [3][cols] (max, sum, dot planes, natural-log units).
 * For bf16 operands whose logits are provably bounded (logit_scale * max|x_i| * max|y_j| <= ~66, checked on the device
 * from the row norms) this is ONE sweep over the tiles: every tile feeds the row and the column sums (for d <= 512 with
 * the rows of X resident in shared memory).  Otherwise the library runs the exact two-sweep form by itself (same
 * results, the cost of two clipk_fwd_stats calls).  pos_logit may be NULL.  amax_xy (may be NULL) receives max |x| of
 * X and of Y when the single-sweep path computed them on its way (NaN otherwise): clipk_to_f16_amax takes them, so the
 * backward need not read the features again just to find its fp16 scale.  exact != 0 forces the two-sweep form, whose
 * `max` planes are the true row / column maxima (the single sweep reports its global reference there; max + log(sum)
 * is the log-sum-exp either way) - callers that want top-1 accuracy (pos_logit >= max) ask for it. */
size_t clipk_fwd_both_workspace_bytes(int rows, int cols, int d, int dtype);
int clipk_fwd_both(const void* X, const void* Y, int rows, int cols, int d, long long ldx, long long ldy, int dtype,
                   const float* x_inv_scale, const float* y_inv_scale, const float* logit_scale, long long diag_offset,
                   float* row_stats, float* pos_logit, float* col_stats, float* amax_xy, int exact, void* workspace,
                   size_t workspace_bytes, void* stream);

/* clipk_finalize merges statistics into log-sum-exps, the two cross-entropy sums (loss.py:135-138) and the two
 * sums that make up dloss/dlogit_scale:
 *   lse_row[i] = row_max[i] + log(row_sum[i])                                  i < rows
 *   lse_col[j] = logsumexp over the nparts (max, sum) pairs of column j        j < cols
 *   sums[0] = sum_i (lse_row[i] - pos_logit[i])            sums[1] = sum_i (lse_col[diag_offset + i] - pos_logit[i])
 *   sums[2] = sum_i (E_row[i] - pos_logit[i])              sums[3] = sum_i (E_col[diag_offset + i] - pos_logit[i])
 * where E is the expected logit under the row / column softmax (dot / sum), so that
 *   dloss/dlogit_scale = (sums[2] + sums[3]) / (2 * num_logits * logit_scale).
 * col_*_parts hold nparts parts, part p of column j at [p * part_stride + j]: one part per data-parallel rank
 * after the all-gather of the column statistics (the exchange that replaces materialising logits_per_text on every rank).
 */
int clipk_finalize(const float* row_max, const float* row_sum, const float* row_dot, const float* pos_logit, int rows,
                   const float* col_max_parts, const float* col_sum_parts, const float* col_dot_parts, int nparts,
                   long long part_stride, int cols, long long diag_offset, float* lse_row, float* lse_col, float* sums,
                   void* stream);

/* ---- backward -----------------------------------------------------------------------------------------
 * clipk_bwd replaces autograd's backward of the same lines (softmax - onehot and the four gradient GEMMs).  It
 * recomputes S tile by tile from X, Y (dtype as in the forward), forms
 *   G = alpha * (P_row - Id) + beta * (P_col - Id),
 *   P_row = exp(S - lse_row[:, None]),  P_col = exp(S - lse_col[None, :]),
 * holds it as fp16 (x 2^14; two planes when g_dtype == CLIPK_F16X2) in an L2-sized panel of the workspace (about
 * 4736 x 4736 at a time), and accumulates in fp32, with Xg / Yg the CLIPK_F16 or CLIPK_F16X2 copies of the features:
 *   dX_acc [rows, d] = logit_scale * gscale * G * Yg          (NULL to skip)
 *   dY_acc [cols, d] = logit_scale * gscale * G^T * Xg        (NULL to skip; the caller reduce-scatters it)
 * Per panel: one launch recomputes and writes G, one launch runs the dX tiles and the dY tiles together.
 * gscale is a device scalar = grad_output / (2 * num_logits).  dX_acc and dY_acc are overwritten.
 * split_row_col = 1: dX is built from alpha (P_row - Id) alone and dY from beta (P_col - Id) alone, from ONE recompute
 * that writes the two parts as two planes of the panel - the gradients of local_loss=True, gather_with_grad=False
 * (loss.py:53-56: the gathered tensors carry no gradient, so dI sees only the image->text softmax and dT only the
 * text->image one).  One-plane (CLIPK_F16) gradient operands only.
 */
size_t clipk_bwd_workspace_bytes(int rows, int cols, int d, int g_dtype);
int clipk_bwd(const void* X, const void* Y, int rows, int cols, int d, long long ldx, long long ldy, int dtype,
              const float* x_inv_scale, const float* y_inv_scale, const void* Xg, const void* Yg, long long ldxg,
              long long ldyg, int g_dtype, const float* xg_inv_scale, const float* yg_inv_scale,
              const float* logit_scale, long long diag_offset, const float* lse_row, const float* lse_col,
              float alpha, float beta, int split_row_col, const float* gscale, float* dX_acc, float* dY_acc,
              void* workspace, size_t workspace_bytes, void* stream);

/* ---- the whole loss step in two calls ---------------------------------------------------------------------------------
 * clipk_step_forward / clipk_step_backward run everything ClipLoss.forward (loss.py:123-140) and its autograd do on one
 * rank - including, between the ranks of one NVLink domain, gather_features (loss.py:20-64) and the backward of its
 * all-gather - as ONE enqueue each: no host work, allocation or synchronisation between the kernels.
 *
 *   forward   prep (one pass over the local rows: optional L2 normalisation + cast to the bf16 operands, operand
 *             statistics; the text rows land in the buffer the peers pull from)
 *             -> all-gather of the text rows and the statistics by pulling from peer memory (world > 1)
 *             -> single-sweep tcgen05 forward (row AND column statistics of the [rows, cols] block), merge
 *             -> all-gather of the [3, cols] column statistics (world > 1) -> finalize: lse_row, lse_col, loss.
 *   backward  fp16 copies of both operands -> per panel: recompute G, gradient GEMMs (the text-gradient tiles go
 *             straight into their owners' memory over NVLink when world > 1) -> barrier -> finish: sum of the slots,
 *             Jacobian of the normalisation, cast, dlogit_scale.
 *
 * Operands are bf16 (src_dtype CLIPK_BF16, or CLIPK_F32 inputs cast on the way - what autocast does to the reference's
 * matmul); d % 64 == 0; world == 1 or 2..8 ranks with rows % 128 == 0.  Everything else takes the individual entries
 * above.  All pointers are device pointers except `peer` (host struct) and peer->err (pinned host memory).
 */
#define CLIPK_MAX_PEERS 8
#define CLIPK_STAT_WORDS 8
typedef struct clipk_peer {
    int world, rank;
    /* index = rank that OWNS the memory; entries of other ranks are their peer-mapped addresses */
    void* text_src[CLIPK_MAX_PEERS];    /* [rows, d] bf16: the rank's text operand rows for this call                  */
    void* stats_src[CLIPK_MAX_PEERS];   /* CLIPK_STAT_WORDS floats: the rank's operand statistics                      */
    void* col_src[CLIPK_MAX_PEERS];     /* [3, cols] fp32: column statistics of the rank's block                       */
    void* grad_slot[CLIPK_MAX_PEERS];   /* [rows, d] fp32: THIS rank's slot of the text gradient in the owner's memory */
    void* flags_gather[CLIPK_MAX_PEERS];/* unsigned[CLIPK_MAX_PEERS] per purpose, zero at start                        */
    void* flags_stats[CLIPK_MAX_PEERS];
    void* flags_grad[CLIPK_MAX_PEERS];
    unsigned int epoch_gather, epoch_stats, epoch_grad;   /* grow by one per call, same on all ranks                  */
    const float* my_slots;              /* [world][rows, d] fp32: the slots this rank owns (slot w written by rank w)  */
    int* err;                           /* pinned host word: non-zero after a peer wait timed out                      */
} clipk_peer;

typedef struct clipk_step {
    int rows, cols, d;                  /* local rows b, global columns N = world * b, embedding width                 */
    int src_dtype;                      /* CLIPK_BF16 or CLIPK_F32: dtype of image / text                              */
    int normalize;                      /* 1: rows are L2-normalised first (F.normalize, open_clip/model.py:216,231)   */
    float eps;
    const void* image; const void* text;            /* this rank's [rows, d] inputs                                   */
    long long ld_image, ld_text;
    const float* logit_scale;           /* device scalar                                                               */
    float loss_div;                     /* loss = (CE sums) / loss_div: 2b (single, local) or 2N (global, then summed  */
                                        /* over the ranks by the caller)                                               */
    float grad_coef;                    /* feature gradients = grad_out * grad_coef * d(CE sums): 1/2b or 1/2N         */
    int grad_split;                     /* 1: local_loss without gather_with_grad - dI from the row softmax only, dT   */
                                        /* from the column softmax only (see clipk_bwd's split_row_col)               */
    /* buffers that live from the forward to the backward (caller-allocated, one set per call) */
    void* x_op;                         /* [rows, d] bf16 image operand; == image when nothing has to be produced      */
    void* y_all;                        /* [cols, d] bf16 gathered text operand; == text under the same condition      */
    float* inv_x; float* inv_y;         /* [rows] 1 / max(|row|, eps)  (normalize only)                                */
    float* stats;                       /* [world][CLIPK_STAT_WORDS]                                                   */
    float* lse_row; float* lse_col;     /* [rows], [cols]                                                              */
    float* scal;                        /* 16 floats: [0..3] CE / dscale sums, [4] loss, [5] s * dloss/ds, [8..9] LSE   */
                                        /* min / max (ints)                                                            */
    void* g16;                          /* [rows + cols, d] fp16 + 64 floats: the operands' fp16 copies for the gradient */
                                        /* GEMMs.  world > 1: made by the forward while it waits for the peers' column  */
                                        /* statistics (NULL: the backward makes them in its workspace)                  */
    /* backward only */
    const float* grad_out;              /* device scalar                                                               */
    void* d_image; void* d_text;        /* [rows, d] in out_dtype (NULL = not wanted)                                  */
    float* d_scale;                     /* device scalar (NULL = not wanted)                                           */
    int out_dtype;                      /* CLIPK_BF16 or CLIPK_F32                                                     */
    const clipk_peer* peer;             /* NULL when world == 1                                                        */
    void* workspace; size_t workspace_bytes;        /* scratch, may be shared by all calls of one shape on one stream; */
                                                    /* its first 256 bytes must be ZERO when it is created (a ticket   */
                                                    /* that every forward returns to zero)                             */
    void* stream;
} clipk_step;
size_t clipk_step_workspace_bytes(const clipk_step* step);
int clipk_step_forward(const clipk_step* step);
int clipk_step_backward(const clipk_step* step);

/* ---- SigLipLoss: the pairwise sigmoid loss (open_clip >= 2.21, loss.py SigLipLoss) in two calls -----------------------
 * For the b local rows x_i of rank r against all N = world * b text rows y_j (rank-major), with s = logit_scale (already
 * exponentiated) and t = logit_bias:
 *   l_ij = s x_i.y_j + t,  z_ij = +1 if j == diag_offset + i else -1,  loss = (1/b) sum_ij softplus(-z_ij l_ij),
 *   g_ij = sigma(l_ij) - [j == diag_offset + i],
 *   d_x = go (s/b) G Y [rows, d],  d_y = go (s/b) G^T X [cols, d] (the caller reduce-scatters it over the ranks),
 *   d_scale = go (1/b) sum_ij g_ij x_i.y_j,  d_bias = go (1/b) sum_ij g_ij      (per rank, not reduced).
 * The [rows, cols] logits are never stored.
 *   clipk_siglip_forward   one A-resident tcgen05 sweep over the tiles (per row: sum of softplus, largest negative logit,
 *                          positive logit) and two small merge kernels -> loss, gmax = largest |g_ij| of the block
 *   clipk_siglip_backward  fp16 copies of X and Y; per panel of G: recompute sweep that writes fp16(g * 2^e), with 2^e
 *                          chosen on the device from gmax so that the largest entry lands in [2^13, 2^14), and its row
 *                          sums of g and g x.y; the two gradient GEMMs (gemm_pair_kernel); then d_scale, d_bias.
 * Every sum is merged in a fixed order: two calls on the same inputs give bit-identical results.  bf16 operands,
 * d % 64 == 0, rows 16-byte aligned.  The library allocates nothing and never synchronises. */
#define CLIPK_SIGLIP_STATE_WORDS 8
typedef struct clipk_siglip {
    int rows, cols, d;                  /* local rows b, columns N (all ranks' text rows), embedding width (d % 64 == 0) */
    const void* x; long long ldx;       /* [rows, d] bf16 image features, leading dimension in elements                */
    const void* y; long long ldy;       /* [cols, d] bf16 text features of all ranks, rank-major                        */
    const float* logit_scale;           /* device scalar s                                                              */
    const float* logit_bias;            /* device scalar t (NULL = 0)                                                   */
    long long diag_offset;              /* the positive of row i is column diag_offset + i (rank * rows)                */
    float* state;                       /* CLIPK_SIGLIP_STATE_WORDS floats, written by the forward, read and extended   */
                                        /* by the backward: [0] loss, [1] gmax, [2] largest negative logit, [3]         */
                                        /* smallest positive logit, [4] 2^e of the G panel, [5] go * s / (b * 2^e)      */
    /* backward only */
    const float* grad_out;              /* device scalar go                                                             */
    float* d_x;                         /* [rows, d] fp32, overwritten (NULL = not wanted)                              */
    float* d_y;                         /* [cols, d] fp32, overwritten (NULL = not wanted)                              */
    float* d_scale; float* d_bias;      /* device scalars (NULL = not wanted)                                           */
    void* workspace; size_t workspace_bytes;        /* scratch of clipk_siglip_workspace_bytes(), 256-byte aligned;   */
                                                    /* nothing in it lives from one call to the next                   */
    void* stream;
} clipk_siglip;
size_t clipk_siglip_workspace_bytes(const clipk_siglip* p);
int clipk_siglip_forward(const clipk_siglip* p);
int clipk_siglip_backward(const clipk_siglip* p);

/* ---- opt-in: the L2 normalisation in front of the loss (SURVEY section 8 f-1) ---------------------------------------
 * The reference normalises in the model, not in the loss (F.normalize, open_clip/model.py:216,231,277,281); these two
 * entries let a caller hand RAW embeddings to clipk.fused_normalize_clip_loss and get gradients with respect to them.
 *   clipk_normalize_fwd: y[r, :] = x[r, :] / max(|x[r, :]|, eps),  inv_norm[r] = 1 / max(|x[r, :]|, eps)
 *   clipk_normalize_bwd: dx = (g - y (y . g)) * inv_norm   (the Jacobian of the normalisation; a plain scaling where
 *                        |x| < eps)
 * dtype CLIPK_BF16 or CLIPK_F32 for x, y, g, dx alike; d % 8 == 0; eps as in F.normalize (1e-12). */
int clipk_normalize_fwd(const void* x, int dtype, long long rows, long long d, long long ldx, void* y, long long ldy,
                        float* inv_norm, float eps, void* stream);
int clipk_normalize_bwd(const void* g, long long ldg, const void* y, long long ldy, const float* inv_norm, int dtype,
                        long long rows, long long d, void* dx, long long ldd, float eps, void* stream);

/* dst[i] = (dtype) src[i]; the fp32 gradient accumulators are returned in the dtype of the inputs. */
int clipk_cast(const float* src, void* dst, long long n, int dtype, void* stream);

/* Measurement hooks (bench.py).  clipk_bwd_panel: extents of the softmax-gradient panel clipk_bwd uses for this block
 * (one recompute launch + one gradient-GEMM launch per panel).  clipk_profile_begin / _end: while a profile runs every
 * kernel launch of this library is followed by an event on its stream; _end synchronises and writes
 * "kernel:launches:milliseconds;" per kernel name into `out` (time between consecutive events = the kernel launched in
 * between, on one stream).  Not thread-safe; leave it off in production. */
int clipk_bwd_panel(int rows, int cols, int d, long long* panel_rows, long long* panel_cols);
int clipk_profile_begin(void* stream);
int clipk_profile_end(char* out, size_t out_bytes);

/* Test hook: dumps the register <-> (lane, column) mapping of tcgen05.ld.16x256b, which the single-sweep forward relies
 * on: out (8 * 32 * 16 ints) receives, for warp w, 16-lane half h, thread t, register k, the value lane * 1000 + column
 * at index ((w * 2 + h) * 32 + t) * 16 + k. */
int clipk_debug_tmem_layout(int* out, void* stream);

/* ---- dense logits tiles (evaluation side; also the test hook of the tensor-core mainloop) -----------------------------
 * clipk_gemm16: D[M, N] (fp32, ldd) (+)= A * B^T with 16-bit operands on the same tcgen05/TMA mainloop as the loss
 *   (bf16 when f16 == 0, fp16 when f16 == 1; both operands share the format - the hardware rejects a mix).
 *   a_mn = 0: A is [M, K] row-major (K contiguous);  a_mn = 1: A is stored [K, M] row-major (M contiguous).
 *   b_mn likewise for B ([N, K] or [K, N]).  N % 4 == 0, ldd % 4 == 0; rows of B past its extent read as zero.
 * It materialises a panel of logits for the callers that rank instead of reduce: get_clip_metrics
 * (training/train.py:631-648: logit_scale * image_features @ text_features.t(), argsort) and the zero-shot classifier
 * (training/zero_shot.py:54-57: 100 * image_features @ classifier, topk).
 */
int clipk_gemm16(const void* A, const void* B, float* D, int M, int N, int K, long long lda, long long ldb,
                 long long ldd, int a_mn, int b_mn, int f16, int accumulate, void* stream);

/* clipk_rank_count: position of the target column in each row of such a panel, without sorting it.  S holds `rows` rows
 * of `cols` logits (fp32, ld % 4 == 0, 16-byte aligned); the panel's first row is global row row0.  The target of global
 * row g is target[g] (device int64, indexed by GLOBAL row) or, with target == NULL, column diag_offset + g.
 *   greater[g]     = #{ j : S[g, j] >  S[g, t] }              (-1 when t is not a column of the panel)
 *   ties_before[g] = #{ j < t : S[g, j] == S[g, t] }          (may be NULL)
 * greater + ties_before is the index of the target in a stable descending sort of the row: what
 * torch.where(torch.argsort(logits, descending=True) == ground_truth) yields (train.py:640-641), and `rank < k` is the
 * top-k test of zero_shot.py:36-39.  Both outputs are indexed by global row. */
int clipk_rank_count(const float* S, int rows, int cols, long long ld, const long long* target, long long diag_offset,
                     long long row0, int* greater, int* ties_before, void* stream);

/* ---- distillation term of DistillClipLoss (loss.py:187-216) on logits panels ----------------------------------------
 * dist_loss(teacher, student) = mean_i [ lse(S_i) - sum_j softmax(T_i)(j) * S_ij ] per direction.  The LSEs of both
 * models come from clipk_fwd_both + clipk_finalize; the cross term needs student and teacher logits of the same
 * element, so it is taken from a pair of panels made by clipk_gemm16 (S = student, T = teacher raw products of the same
 * [rows, cols] block, fp32, leading dimension ld; logits = S * (*s_mul), T * (*t_mul), device scalars that carry
 * logit_scale and the operands' power-of-two scales).  The panel holds ALL columns of its rows; its first row is global
 * row row0, and vectors indexed by row are indexed by GLOBAL row.
 *   clipk_distill_cross: row_cross[g] = sum_j exp(T_gj - t_lse_row[g]) * S_gj                (complete per call)
 *                        col_part[j]  = sum_{rows of the panel} exp(T_gj - t_lse_col[j]) * S_gj   (the caller adds panels)
 *   clipk_distill_grad : G[r, j] = fp16( 2^14 * ( exp(S - s_lse_row[g]) - exp(T - t_lse_row[g])
 *                                               + exp(S - s_lse_col[j]) - exp(T - t_lse_col[j]) ) ),  G is [rows, ldg]:
 *                        the derivative of both directions' terms with respect to the student's logits times 2 n,
 *                        in the operand format of the gradient GEMMs (clipk_gemm16 with f16 = 1).
 * rows <= 65535 per call.  STATUS: validated on a B200 (tests/test_distill_gpu.py) and on the CPU emulation; the
 * default path of clipk/distill.py for the shapes it accepts (CLIPK_FUSED_DISTILL=0 switches it off). */
int clipk_distill_cross(const float* S, const float* T, int rows, int cols, long long ld, const float* s_mul,
                        const float* t_mul, const float* t_lse_row, const float* t_lse_col, long long row0,
                        float* row_cross, float* col_part, void* stream);
int clipk_distill_grad(const float* S, const float* T, int rows, int cols, long long ld, const float* s_mul,
                       const float* t_mul, const float* s_lse_row, const float* t_lse_row, const float* s_lse_col,
                       const float* t_lse_col, long long row0, void* G, long long ldg, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLIPK_H_ */
