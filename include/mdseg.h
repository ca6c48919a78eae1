/*
 * mdseg.h — C ABI of libmdseg_b200.so
 *
 * B200 (sm_100a) implementation of the per-pixel multi-dataset label-space hot
 * path of Mrhonor/Mul-Datasets-Semantic-Segmentation.  The reference has no
 * FFI of its own (it is pure Python on ATen); every entry point below cites the
 * reference lines whose work it replaces.  SURVEY.md §8(b) is the contract.
 *
 * Conventions
 *   - plain C: pointers, sizes, enums.  No torch / C++ types cross this ABI.
 *   - every pointer is a DEVICE pointer unless the parameter says "host".
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *   - the library never allocates or frees device memory and never
 *     synchronises the host; the caller owns every buffer.
 *   - return value: 0 = OK, non-zero = error; text via mdseg_last_error().
 *   - data errors found on the device (labels outside [0,C) ∪ {ignore}) set
 *     bits in a caller-owned int32 `err_flag` (may be NULL) — the reference
 *     would hit a device assert inside nll_loss / a reshape error in bincount.
 */
#ifndef MDSEG_H_
#define MDSEG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDSEG_VERSION 100 /* 0.1.0 */

/* element types */
enum {
  MDSEG_F32 = 0,
  MDSEG_BF16 = 1,
  MDSEG_F16 = 2,
  MDSEG_U8 = 10,
  MDSEG_I32 = 11,
  MDSEG_I64 = 12
};

/* layouts of logits and features */
enum { MDSEG_NCHW = 0, MDSEG_NHWC = 1 };

/* err_flag bits */
enum {
  MDSEG_ERR_LABEL_RANGE = 1, /* label not in [0,C) and != ignore          */
  MDSEG_ERR_PRED_RANGE = 2,  /* prediction not in [0,Cb)                  */
  MDSEG_ERR_TOPK_RANGE = 4,  /* n_min larger than the number of loss px   */
  MDSEG_ERR_DATASET_ID = 8,  /* dataset id outside [0,n_datasets)         */
  MDSEG_ERR_GRAPH_KIND = 16  /* a graph declared column-one-hot 0/1 is not */
};

#define MDSEG_MAX_DATASETS 32

/*
 * OHEM selection state of one "segment" (= one call of the reference's
 * OhemCELoss / MdsOhemCELoss).  Lives in device memory, caller-allocated,
 * 128 bytes.  Zeroed by mdseg_ohem_begin; filled by the *_fwd kernels;
 * completed by mdseg_ohem_select; consumed by the *_bwd kernels.  The layout is
 * public so tests can read it back.
 */
typedef struct mdseg_ohem_state {
  unsigned long long n_valid; /* #{label != ignore}             (ohem_ce_loss.py:25,52) */
  unsigned long long n_hard;  /* #{loss > thresh}               (ohem_ce_loss.py:30,74) */
  unsigned long long n_px;    /* number of loss entries of this segment               */
  unsigned long long n_min;   /* n_valid / 16                                          */
  unsigned long long n_sel;   /* |S| : number of selected entries                      */
  unsigned long long n_gt;    /* top-k mode: #{loss > kth}                             */
  double sum_hard;            /* Σ loss over {loss > thresh}                           */
  double sum_sel;             /* Σ loss over S                                         */
  float thresh;               /* τ = -log(thresh_prob)                                 */
  float kth;                  /* top-k mode: the n_min-th largest loss                 */
  float inv_n_sel;            /* 1/|S| (0 if S empty)                                  */
  float loss;                 /* mean over S (NaN if S empty, like torch.mean([]))     */
  unsigned int mode;          /* 0 = threshold set, 1 = top-k fallback                 */
  unsigned int tie_quota;     /* top-k mode: how many entries == kth belong to S       */
  unsigned int tie_taken;     /* select: ties examined so far (first-come hand-out)    */
  unsigned int n_ties;        /* top-k mode: #{loss == kth}                            */
  unsigned int reserved[8];
} mdseg_ohem_state;

/*
 * Where the low-resolution logits of image b live, for the fused
 * upsample+CE kernels.  Passed BY VALUE from the host.  Image b of dataset
 * d = dataset_ids[b] (d = 0 when dataset_ids == NULL) reads
 *     base[d] + b * image_stride[d]          (elements, layout [C[d], h, w])
 * - main multi-dataset loss: every base[d] is the projected-logit buffer
 *   (loss_cross_datasets.py:1006), C[d] = n_cats of dataset d;
 * - aux heads: base[d] = aux_logits[d] ([ΣB, C_d, h, w], all images;
 *   loss_cross_datasets.py:1051).
 * seg_per_dataset != 0 -> OHEM segment of image b is d (aux heads: one
 * selection per dataset, :1053-1056), else segment 0 (MdsOhemCELoss: one
 * selection over the whole batch, ohem_ce_loss.py:70-88).
 */
typedef struct mdseg_src_table {
  const void* base[MDSEG_MAX_DATASETS];
  long long image_stride[MDSEG_MAX_DATASETS];
  int C[MDSEG_MAX_DATASETS];
  int C_alloc[MDSEG_MAX_DATASETS]; /* channels allocated per image (>= C; 0 means C) */
  int n_datasets;
  int dtype;           /* MDSEG_F32 / BF16 / F16 */
  int seg_per_dataset; /* 0 / 1 */
  int cmax_ready;      /* cmax already holds the per-pixel channel maximum of the sources */
  float* cmax;         /* optional workspace, fp32 [n_images, h, w]: max_c src[b, c, y, x].  When
                          non-NULL (and dtype F32, w % 4 == 0, up-sampling factor <= 5) the
                          TMA-pipelined kernels are used; mdseg_up_ce_fwd fills it first unless
                          cmax_ready (mdseg_proj_fwd can produce it for free). */
} mdseg_src_table;

/*
 * Sparse bipartite / remap matrix G [C_ds, C_uni] of one dataset in CSR (rows
 * = dataset classes) and CSC (columns = unified classes) form, device
 * resident.  vals may be NULL (all ones: the 0/1 graphs of the SEG stage and
 * ClassRemap.getRemapMatrix, class_remap.py:176-183).
 */
typedef struct mdseg_sparse_graph {
  const int* csr_ptr;    /* [C_ds + 1]  */
  const int* csr_col;    /* [nnz] unified ids, ascending within a row */
  const float* csr_val;  /* [nnz] or NULL */
  const int* csc_ptr;    /* [C_uni + 1] */
  const int* csc_row;    /* [nnz] dataset classes, ascending within a column */
  const float* csc_val;  /* [nnz] or NULL */
  const float* dense;    /* [C_ds, C_uni] row-major or NULL; when non-NULL the
                            dense kernels are used (GNN stage) */
  int C_ds;
  int nnz;
  int col_onehot;        /* every column has at most one entry (UOT / pretrain graphs,
                            ltbgnn_direct_learn.py:426-439,689-692) */
  int reserved;
  /* optional (may be NULL): the CSR rows padded to a multiple of 4 entries by repeating the
   * last entry of the row; csr4_ptr[n] is the row start in QUADS.  Lets mdseg_mds_bwd fetch four
   * unified ids per shared-memory load when it broadcasts a dataset-class gradient. */
  const int* csr4_ptr;   /* [C_ds + 1]  */
  const int* csr4_col;   /* [4 * csr4_ptr[C_ds]] */
} mdseg_sparse_graph;

typedef struct mdseg_graph_table {
  mdseg_sparse_graph g[MDSEG_MAX_DATASETS];
  int n_datasets;
  int C_uni;
} mdseg_graph_table;

/* ---- library ---------------------------------------------------------- */
int mdseg_version(void);
/* thread-local, valid until the next failing call on this thread */
const char* mdseg_last_error(void);
/* number of SMs of the current device (cached) — grids are sized from it */
int mdseg_sm_count(void);

/* ---- a1 / a2: LUT remap -------------------------------------------------
 * out[p] = lut[in[p]];  values outside [0,255] (int inputs) map to `oob`.
 * Replaces `label = self.lb_map[label]` (lib/base_dataset.py:81-82) and the
 * per-class masked writes of ClassRemap.SingleSegRemapping / SegRemapping /
 * ReverseSegRemap (lib/class_remap.py:34-66,189-203), which are 256-entry
 * LUTs.  in_dtype / out_dtype ∈ {U8, I32, I64}. */
int mdseg_lut_remap(const void* in, int in_dtype, void* out, int out_dtype,
                    const uint8_t* lut256, int oob, int64_t n, void* stream);

/* ---- a4: multi-hot label remap ---------------------------------------------
 * out[p, u] = table[labels[p], u] (bytes 0 / 1; labels outside [0,255] give a zero
 * row).  table: uint8 [256, C_uni], out: uint8 / bool [n_px, C_uni], 16-byte aligned.
 * Replaces ClassRemapOneHotLabel.SegRemapping / SingleSegRemappingOneHot
 * (lib/class_remap.py:239-276): one compare + masked scatter per dataset class. */
int mdseg_multihot_remap(const void* labels, int label_dtype, const uint8_t* table,
                         int C_uni, int64_t n_px, uint8_t* out, void* stream);

/* ---- a12: confusion matrix ----------------------------------------------
 * hist[l*Cb + q] += 1 for every p with l = (lut ? lut[label[p]] : label[p])
 * != ignore, q = pred[p].  hist is int64 [Ca*Cb], accumulated into.
 * Replaces evaluate.py:89-93,174-181 (np.bincount(label[keep]*C+pred[keep]))
 * and the rectangular variants evaluate.py:631-634,1738-1741. */
int mdseg_confusion(const void* label, int label_dtype, const void* pred,
                    int pred_dtype, const uint8_t* lut256, int64_t* hist,
                    int Ca, int Cb, int ignore, int64_t n, int32_t* err_flag,
                    void* stream);

/* ---- a1 + a12 for a whole multi-dataset batch in one launch each -----------------------------
 * The trainers' batch holds images of several datasets (tools/train_ltbgnn_all_datasets_snp.py:708-750,
 * lib/MultiSetReader.py:26-34); the reference remaps / evaluates them dataset by dataset.  Here image
 * b uses table / class count / histogram of dataset dataset_ids[b] (NULL: dataset 0). */
typedef struct mdseg_hist_table {
  int n_datasets;
  int C[MDSEG_MAX_DATASETS];             /* classes of dataset d: its histogram is C[d] x C[d] */
  long long offset[MDSEG_MAX_DATASETS];  /* element offset of that histogram inside `hist`      */
} mdseg_hist_table;
/* out[b, p] = luts[lut_ids[b]][in[b, p]]; luts: device uint8 [n_luts][256] */
int mdseg_lut_remap_images(const void* in, int in_dtype, void* out, int out_dtype, const uint8_t* luts, int n_luts,
                           const int32_t* lut_ids, int oob, int n_images, int64_t px_per_image, int32_t* err_flag,
                           void* stream);
/* hist_d[l*C_d + q] += 1 over the images of dataset d, for every dataset; luts (optional, device
 * uint8 [n_datasets][256]) are applied to the labels first.  Images are px_per_image % 16 == 0. */
int mdseg_confusion_images(const void* label, int label_dtype, const void* pred, int pred_dtype,
                           const uint8_t* luts, const int32_t* dataset_ids, int n_images, int64_t px_per_image,
                           int64_t* hist, const mdseg_hist_table* tab /*host*/, int ignore, int32_t* err_flag,
                           void* stream);
/* iou[d*iou_stride + c], miou[d] for every dataset (evaluate.py:94-98) */
int mdseg_miou_images(const int64_t* hist, const mdseg_hist_table* tab /*host*/, float* iou, int iou_stride,
                      float* miou, void* stream);

/* ---- a13: IoU from the histogram (device, no sync) ------------------------
 * iou[c] = h[c,c] / (Σ_r h[r,c] + Σ_q h[c,q] - h[c,c]) (NaN when 0/0) and
 * miou = nanmean(iou).  evaluate.py:94-98. */
int mdseg_miou(const int64_t* hist, int C, float* iou, float* miou,
               void* stream);

/* ---- a8: OHEM state -------------------------------------------------------*/
size_t mdseg_ohem_state_bytes(void);
/* workspace for mdseg_ohem_select, per segment */
size_t mdseg_select_workspace_bytes(int n_segments);
/* zero n_segments states and set their threshold τ = -log(thresh_prob) given
 * as the already-computed float `thresh` (ohem_ce_loss.py:17,42). */
int mdseg_ohem_begin(mdseg_ohem_state* states, int n_segments, float thresh,
                     void* stream);

/* ---- a7 + first half of a8: full-resolution CE forward --------------------
 * loss_px[p] = logsumexp_c(z[p,:]) - z[p,label[p]]   (0 where label == ignore)
 * lse_px[p]  = logsumexp (natural log), kept for the backward.
 * Accumulates n_valid / n_hard / sum_hard / n_px into states[0].
 * Replaces nn.CrossEntropyLoss(ignore_index=255, reduction='none') and the
 * `loss > thresh` compare of lib/loss/ohem_ce_loss.py:25-30. */
int mdseg_ohem_ce_fwd(const void* logits, int dtype, int layout,
                      const void* labels, int label_dtype, int N, int C, int H,
                      int W, int ignore, float* loss_px, float* lse_px,
                      mdseg_ohem_state* state, int32_t* err_flag, void* stream);

/* ---- second half of a8: selection ------------------------------------------
 * For each segment: n_min = n_valid/16; S = {loss > τ}; if |S| < n_min, S =
 * the n_min largest entries (radix select over the fp32 bit pattern, no
 * sort); loss_out[seg] = mean over S.  image_seg (device int32 [n_images]) maps
 * an image to its segment (NULL: all images belong to segment 0; entries < 0
 * or >= n_segments are skipped).  In top-k mode the entries equal to the k-th
 * value that do not fit into S are overwritten in loss_px with the next
 * smaller float, so that the backward kernels can test `loss >= kth`.
 * Replaces ohem_ce_loss.py:30-34 / :74-90. */
int mdseg_ohem_select(float* loss_px, int n_images, int64_t px_per_image,
                      const int32_t* image_seg, mdseg_ohem_state* states,
                      int n_segments, void* workspace, float* loss_out,
                      int32_t* err_flag, void* stream);

/* ---- a9: full-resolution CE backward ----------------------------------------
 * dlogits[p,c] = grad_out * w_p * (softmax(z[p,:])_c - [c == label_p]),
 * w_p = 1/|S| for p in S else 0.  grad_out: device float scalar (AMP scale).
 * dlogits has the dtype / layout of logits and is fully overwritten. */
int mdseg_ohem_ce_bwd(const void* logits, int dtype, int layout,
                      const void* labels, int label_dtype, int N, int C, int H,
                      int W, int ignore, const float* loss_px,
                      const float* lse_px, mdseg_ohem_state* state,
                      const float* grad_out, float grad_scale, void* dlogits,
                      void* stream);

/* ---- a5: bipartite projection (sparse 0/1 or weighted graphs) ----------------
 * y[b, n, :, :] = Σ_c G_d[n, c] * x[b, c, :, :], d = dataset_ids[b].
 * x: [n_images, C_uni, h, w] (dtype), y: fp32 [n_images, y_cmax, h, w] (only
 * the first C_ds(d) channels of image b are written).
 * Replaces torch.einsum('bchw,nc->bnhw', logits[dataset_ids==i], bi_graphs[i])
 * (lib/loss/loss_cross_datasets.py:1006; lib/models/semseg.py:344). */
int mdseg_proj_fwd(const void* x, int dtype, const mdseg_graph_table* graphs /*host*/,
                   const int32_t* dataset_ids, int n_images, int h, int w,
                   float* y, int y_cmax, float* cmax_out /* optional fp32 [n_images,h,w]: max_n y */,
                   int32_t* err_flag, void* stream);

/* The same projection with the DENSE graphs (GNN stage: soft adjacency with grad,
 * loss_cross_datasets.py:997-1006) on the tcgen05 tensor cores: a [128 px, C_uni] x
 * [C_uni, C_ds] tile per CTA, fp32 accumulators in TMEM.  fp32 inputs are split into
 * three bf16 terms per operand (six products, relative error ~2^-21); bf16 / fp16
 * inputs take one product in their own type with G rounded to it (what autocast does
 * to the reference einsum).  Datasets with a sparse graph, or a dense one outside the
 * envelope (C_ds < 8, C_ds > 256, C_uni < 32), go through the kernels of
 * mdseg_proj_fwd inside the same call.  `workspace` (caller-owned, device) receives the
 * converted graphs; it is rewritten on every call, so graphs may change between calls. */
size_t mdseg_proj_fwd_tc_workspace_bytes(const mdseg_graph_table* graphs /*host*/, int dtype);
int mdseg_proj_fwd_tc(const void* x, int dtype, const mdseg_graph_table* graphs /*host*/,
                      const int32_t* dataset_ids, int n_images, int h, int w,
                      float* y, int y_cmax, float* cmax_out, void* workspace,
                      size_t workspace_bytes, int32_t* err_flag, void* stream);

/* dx[b, c, :, :] = Σ_n G_d[n, c] * (dyA[b, n] + dyB[b, n]); dyB may be NULL.
 * dx has dtype of x and is fully overwritten (zeros for images whose dataset
 * id is out of range). */
int mdseg_proj_bwd(const float* dyA, const float* dyB, int y_cmax,
                   const mdseg_graph_table* graphs /*host*/,
                   const int32_t* dataset_ids, int n_images, int h, int w,
                   void* dx, int dtype, void* stream);

/* The same adjoint with the dense graphs on the tcgen05 tensor cores (K = C_ds, the unified
 * channels tiled by at most 128 per CTA); precision and envelope as mdseg_proj_fwd_tc, the
 * remaining datasets and the zero fill go through the kernels of mdseg_proj_bwd. */
size_t mdseg_proj_bwd_tc_workspace_bytes(const mdseg_graph_table* graphs /*host*/, int dtype);
int mdseg_proj_bwd_tc(const float* dyA, const float* dyB, int y_cmax,
                      const mdseg_graph_table* graphs /*host*/, const int32_t* dataset_ids,
                      int n_images, int h, int w, void* dx, int dtype, void* workspace,
                      size_t workspace_bytes, void* stream);

/* d bi_graph (GNN stage): dG_d[n, c] += Σ_{b in d} Σ_px (dyA+dyB)[b,n,px] * x[b,c,px]
 * dG: fp32 [n_datasets][dg_stride] with row-major [C_ds, C_uni] inside, must be
 * zeroed by the caller. */
int mdseg_proj_bwd_graph(const void* x, int dtype, const float* dyA,
                         const float* dyB, int y_cmax,
                         const mdseg_graph_table* graphs /*host*/,
                         const int32_t* dataset_ids, int n_images, int h, int w,
                         float* dG, long long dg_stride, void* stream);

/* The same with the dense graphs on the tcgen05 tensor cores: K = the pixels of an image slab
 * (both operands are K-major in HBM), one 128-class M tile and all of C_uni (<= 512) per CTA,
 * per-CTA partial sums in `workspace`, then a fixed-order reduction into dG (deterministic;
 * the FFMA route uses atomics).  Precision as mdseg_proj_fwd_tc. */
size_t mdseg_proj_bwd_graph_tc_workspace_bytes(const mdseg_graph_table* graphs /*host*/,
                                               int n_images, int h, int w);
int mdseg_proj_bwd_graph_tc(const void* x, int dtype, const float* dyA, const float* dyB,
                            int y_cmax, const mdseg_graph_table* graphs /*host*/,
                            const int32_t* dataset_ids, int n_images, int h, int w,
                            float* dG, long long dg_stride, void* workspace,
                            size_t workspace_bytes, void* stream);

/* ---- a5 for channels_last (NHWC) unified logits -------------------------------
 * The projection of mdseg_proj_fwd with x [n_images, h, w, C_uni] pixel-major (what a model run with
 * memory_format=torch.channels_last produces); y and cmax_out are the same NCHW outputs, bit-identical to
 * mdseg_proj_fwd on the NCHW copy of x.  Sparse graphs only (dense graphs take mdseg_proj_fwd_tc on NCHW),
 * C_uni <= MDSEG_NHWC_MAX_CUNI and every C_ds <= MDSEG_NHWC_MAX_CDS. */
#define MDSEG_NHWC_MAX_CUNI 1536
#define MDSEG_NHWC_MAX_CDS 768
int mdseg_proj_fwd_nhwc(const void* x, int dtype, const mdseg_graph_table* graphs /*host*/,
                        const int32_t* dataset_ids, int n_images, int h, int w,
                        float* y, int y_cmax, float* cmax_out, int32_t* err_flag, void* stream);

/* The adjoint of mdseg_proj_bwd written pixel-major: dx [n_images, h, w, C_uni] in `dtype`, fully overwritten
 * (zeros for images whose dataset id is out of range), bit-identical to mdseg_proj_bwd given the same dy.
 * Same graph limits as mdseg_proj_fwd_nhwc. */
int mdseg_proj_bwd_nhwc(const float* dyA, const float* dyB, int y_cmax,
                        const mdseg_graph_table* graphs /*host*/,
                        const int32_t* dataset_ids, int n_images, int h, int w,
                        void* dx, int dtype, void* stream);

/* Layout moves of the aux heads' channels_last sources.  `nhwc` lists the heads as [n_images, h, w, C_d]
 * (image_stride in elements); `planar` lists where image b's rows go as [C_d, h, w] planes at
 * base[d] + b * image_stride[d] (one shared buffer [n_images, max C_d, h, w] or one per head), same dtype.
 * mdseg_nhwc_to_planar copies the rows of each image's own head d = dataset_ids[b] (0 when NULL).
 * mdseg_planar_to_nhwc writes every head's NHWC tensor: the planar rows for the image's own head, zeros for
 * every other head. */
int mdseg_nhwc_to_planar(const mdseg_src_table* nhwc /*host*/, const int32_t* dataset_ids, int n_images, int h,
                         int w, const mdseg_src_table* planar /*host*/, void* stream);
int mdseg_planar_to_nhwc(const mdseg_src_table* planar /*host*/, const int32_t* dataset_ids, int n_images, int h,
                         int w, const mdseg_src_table* nhwc /*host*/, void* stream);

/* ---- a6 + a7 (+ a10): fused bilinear upsample (align_corners=True) + CE -------
 * For every label pixel (Y,X) of image b: interpolate the C low-res logits of
 * the image's source (see mdseg_src_table) to (Y,X) exactly as
 * F.interpolate(mode='bilinear', align_corners=True) does
 * (loss_cross_datasets.py:1007), then per-pixel CE as in mdseg_ohem_ce_fwd.
 * The [B,C,H,W] upsampled tensor is never materialised.
 * labels: [n_images, H, W]; loss_px / lse_px: fp32 [n_images*H*W]. */
int mdseg_up_ce_fwd(const mdseg_src_table* src /*host*/, const int32_t* dataset_ids,
                    const void* labels, int label_dtype, int n_images, int h,
                    int w, int H, int W, int ignore, float* loss_px,
                    float* lse_px, mdseg_ohem_state* states, int32_t* err_flag,
                    void* stream);

/* Adjoint: gradient w.r.t. the low-res logits.  Written as two fp32 planes with
 * the layout of the source (base/stride/C taken from `dst`, dtype must be F32):
 * plane A holds the contributions through the upper interpolation row, plane B
 * through the lower one; their sum is the gradient (mdseg_proj_bwd and
 * mdseg_add_planes consume them).  Both planes are fully overwritten for every
 * image whose dataset id is valid.  grad_out (device, may be NULL = 1) holds one
 * float per OHEM segment: grad_out[d] when src->seg_per_dataset, else grad_out[0]. */
int mdseg_up_ce_bwd(const mdseg_src_table* src /*host*/, const int32_t* dataset_ids,
                    const void* labels, int label_dtype, int n_images, int h,
                    int w, int H, int W, int ignore, const float* loss_px,
                    const float* lse_px, mdseg_ohem_state* states,
                    const float* grad_out, float grad_scale,
                    const mdseg_src_table* dstA /*host*/,
                    const mdseg_src_table* dstB /*host*/, void* stream);

/* ---- a9 of the multi-dataset loss in one call --------------------------------------
 * dx[b, c, :, :] = d loss / d logits_uni for loss = MdsOhemCELoss(upsample(einsum(logits_uni, G_d)))
 * (autograd replay of lib/loss/loss_cross_datasets.py:1006-1007,1074 + lib/loss/ohem_ce_loss.py:61-90).
 * `src` describes the PROJECTED low-res logits kept by the forward (fp32 [n_images, C_alloc, h, w]).
 * Fused route (fp32 sources, column-one-hot sparse graphs, up-sampling factor in [1,5] per axis):
 * one kernel recomputes the softmax, applies the adjoint of the bilinear interpolation and
 * broadcasts through G^T into dx; a small fix-up kernel finishes the rows on segment
 * boundaries.  Otherwise: mdseg_up_ce_bwd into two planes of the workspace + mdseg_proj_bwd.
 * dx ([n_images, C_uni, h, w], dx_dtype) is fully overwritten.  The workspace is caller-owned
 * scratch of at least mdseg_mds_bwd_workspace_bytes(...) bytes. */
size_t mdseg_mds_bwd_workspace_bytes(const mdseg_src_table* src /*host*/, const mdseg_graph_table* graphs /*host*/,
                                     int n_images, int h, int w, int H, int W);
int mdseg_mds_bwd(const mdseg_src_table* src /*host*/, const mdseg_graph_table* graphs /*host*/,
                  const int32_t* dataset_ids, const void* labels, int label_dtype, int n_images, int h, int w,
                  int H, int W, int ignore, const float* loss_px, const float* lse_px, mdseg_ohem_state* states,
                  const float* grad_out, float grad_scale, void* dx, int dx_dtype, void* workspace,
                  size_t workspace_bytes, void* stream);

/* The same backward without a projection (aux heads, loss_cross_datasets.py:1044-1056): the gradient w.r.t.
 * the low-res sources, written into `dst` (base / image_stride / C per dataset as in `src`, any float
 * dtype).  Only the images of dataset d are written in dst->base[d]; the caller zero-initialises the rest
 * (the reference row-selects aux_logits[i][dataset_ids == i], so those rows get no gradient).
 * Sources must be fp32 on the fused route; other cases take the two-plane route inside the workspace. */
size_t mdseg_up_ce_bwd_direct_workspace_bytes(const mdseg_src_table* src /*host*/, int n_images, int h, int w, int H,
                                              int W);
/* 1 when mdseg_up_ce_bwd_direct takes the fused single-pass kernel for this source table and geometry (fp32
 * sources, aligned rows, up-sampling factor <= 5): destinations may then have any image stride. */
int mdseg_up_ce_bwd_direct_is_fused(const mdseg_src_table* src /*host*/, int h, int w, int H, int W);
int mdseg_up_ce_bwd_direct(const mdseg_src_table* src /*host*/, const int32_t* dataset_ids, const void* labels,
                           int label_dtype, int n_images, int h, int w, int H, int W, int ignore,
                           const float* loss_px, const float* lse_px, mdseg_ohem_state* states,
                           const float* grad_out, float grad_scale, const mdseg_src_table* dst /*host*/,
                           void* workspace, size_t workspace_bytes, void* stream);

/* out = a + b converted to out_dtype (aux heads: dlogits_aux = A + B) */
int mdseg_add_planes(const float* a, const float* b, void* out, int out_dtype,
                     int64_t n, void* stream);

/* ---- a11: eval probability accumulation ---------------------------------------
 * probs[c, Y, X] (+)= softmax_c(upsample(logits)[., Y, X]); `first` != 0
 * overwrites instead of accumulating; `flip` != 0 mirrors the low-res logits
 * along W first (evaluate.py:165-171).  h==H && w==W is the ori_scales=False
 * case (no interpolation, evaluate.py:156-164).  One image per call. */
int mdseg_eval_accum(const void* logits, int dtype, int C, int h, int w,
                     float* probs, int H, int W, int flip, int first,
                     void* stream);

/* ---- a11 + a12 fused over all passes of one image (SURVEY §8 f1) ------------------
 * pred[p] = argmax_c Σ_s softmax_c(upsample(logits_s (mirrored along W if flip_s))[., p]),
 * hist[label[p] * C + pred[p]] += 1 for label != ignore — evaluate.py:136-181 for one
 * image with every (scale, flip) pass at hand, without the [C, H, W] probability tensor:
 * the per-pass soft-max statistics (8 bytes per pixel and pass) go to `workspace`, the
 * class accumulators live in registers.  The sums are bit-identical to mdseg_eval_accum
 * pass by pass followed by mdseg_argmax_hist.  pred (int64 [H*W]) and hist (int64 [C*C],
 * accumulated into) are each optional. */
#define MDSEG_MAX_EVAL_PASSES 16
typedef struct mdseg_eval_pass {
  const void* logits; /* device, [C, h, w] */
  int h, w;
  int flip;
  int reserved;
} mdseg_eval_pass;
typedef struct mdseg_eval_passes {
  mdseg_eval_pass p[MDSEG_MAX_EVAL_PASSES];
  int n_passes;
  int dtype; /* MDSEG_F32 / BF16 / F16, common to all passes */
} mdseg_eval_passes;
size_t mdseg_eval_fused_workspace_bytes(int n_passes, int H, int W);
int mdseg_eval_fused(const mdseg_eval_passes* passes /*host*/, int C, int H, int W,
                     int64_t* pred, const void* label, int label_dtype,
                     const uint8_t* lut256, int64_t* hist, int ignore,
                     void* workspace, size_t workspace_bytes,
                     int32_t* err_flag, void* stream);

/* pred[p] = argmax_c probs[c, p] (first maximal index, like torch.argmax on
 * distinct values); optionally fused with the confusion matrix update
 * (label/hist may be NULL).  evaluate.py:172-181. */
int mdseg_argmax_hist(const float* probs, int C, int64_t n_px, int64_t* pred,
                      const void* label, int label_dtype, const uint8_t* lut256,
                      int64_t* hist, int ignore, int32_t* err_flag,
                      void* stream);

/* legacy 'nearest' resize of a label map (evaluate.py:156-157):
 * src = min(floor(dst * (in/out)), in-1), scale in fp32. */
int mdseg_label_nearest(const void* in, int dtype, int Hin, int Win, void* out,
                        int Hout, int Wout, int n_images, void* stream);

/*
 * Label branch of the training data pipeline as ONE gather (SURVEY.md §8 f3).  Replaces, per sample and on a
 * DataLoader worker in the reference:  label = lb_map[label] (lib/base_dataset.py:81-82) ->
 * cv2.resize(lb, (im_w, im_h), INTER_NEAREST) (lib/transform_cv2.py:43) -> np.pad(..., 255) (:52-53) ->
 * crop (:57-61) -> horizontal flip (:71-77) -> int64 tensor (:300).
 * One view per output image, in DEVICE memory (array of n_images structs); the host fills in the integers the
 * reference's random draws produce.  Output pixels that fall into the padding get `pad_value` (255), which is NOT
 * passed through the LUT (the reference pads after the LUT).  Source index rule of OpenCV's INTER_NEAREST:
 * s = min(floor(d * (1. / ((double)dst / src))), src - 1).
 */
typedef struct mdseg_label_view {
  const uint8_t* src;       /* raw label image, uint8 [src_h, src_w], device memory */
  long long src_row_stride; /* bytes between source rows */
  int src_h, src_w;
  int im_h, im_w;           /* size after the resize */
  int pad_top, pad_left;    /* rows / columns of padding in front of the resized image */
  int crop_y, crop_x;       /* crop origin inside the padded image */
  int flip;                 /* != 0: columns reversed after the crop */
  int lut;                  /* row of `luts` applied to the source bytes; < 0: identity */
} mdseg_label_view;

/* out: [n_images, out_h, out_w] uint8 or int64; out_w % 16 == 0.  luts: [n_luts][256] uint8 or NULL. */
int mdseg_label_pipeline(const mdseg_label_view* views /*device*/, int n_images, const uint8_t* luts, int n_luts,
                         void* out, int out_dtype, int out_h, int out_w, int pad_value, void* stream);

/*
 * Image branch of the same training transforms as ONE gather (SURVEY.md §8 f3).  Replaces, per sample and on a
 * DataLoader worker in the reference, after cv2.imread(p)[:, :, ::-1]:  cv2.resize(im, (im_w, im_h)) (INTER_LINEAR,
 * uint8) -> np.pad(..., 0) -> crop -> horizontal flip -> ColorJitter(brightness, contrast, saturation) ->
 * ToTensor(mean, std), fp32.  The crop / pad / flip integers are those of mdseg_label_view for the same sample.
 * Out-of-image pixels are colour (0, 0, 0) and then go through the jitter and the table, as in the reference.
 * Brightness and contrast are one composed byte table (`lut`), saturation multiplies by the matrix with `sat_diag` on
 * the diagonal and `sat_off` elsewhere (fp32 FMA chain in input-channel order, / 3, clip, truncate), and ToTensor is a
 * float table per channel and byte.  The INTER_LINEAR arithmetic is OpenCV's fixed-point one, bit for bit.
 */
typedef struct mdseg_image_view {
  const uint8_t* src;       /* decoded image, uint8 [src_h, src_w, 3] interleaved (pixel stride 3), device memory */
  long long src_row_stride; /* bytes between source rows */
  int src_h, src_w;
  int im_h, im_w;           /* size after the resize */
  int pad_top, pad_left;    /* rows / columns of padding in front of the resized image */
  int crop_y, crop_x;       /* crop origin inside the padded image */
  int flip;                 /* != 0: columns reversed after the crop */
  int swap_rb;              /* != 0: the source is BGR (cv2.imread), output channel c reads source channel 2 - c */
  int norm;                 /* row of `norm`; a value outside [0, n_norm) reads row 0 */
  int saturate;             /* != 0: apply the saturation matrix after `lut` */
  float sat_diag, sat_off;  /* float32(1 + 2r), float32(1 - r) */
  uint8_t lut[256];         /* brightness then contrast, composed; identity when jitter is off */
} mdseg_image_view;

/* out: fp32, [n_images, 3, out_h, out_w] (MDSEG_NCHW) or [n_images, out_h, out_w, 3] (MDSEG_NHWC, the storage of a
 * channels_last tensor), 16-byte aligned; out_w % 16 == 0.  norm: [n_norm][3][256] fp32, n_norm >= 1. */
int mdseg_image_pipeline(const mdseg_image_view* views /*device*/, int n_images, const float* norm, int n_norm,
                         float* out, int out_layout, int out_h, int out_w, void* stream);

/* ---- f4: NLLPlus loss (soft-max in the unified space, projection of PROBABILITIES, up-sampling, -log) ----------
 * Replaces AdjNLLPlusLoss.forward (lib/loss/loss_helper.py:647-668) as driven by MdsOhemNLLPlusLoss
 * (lib/loss/ohem_ce_loss.py:92-146):
 *     pred  = softmax(x, dim=1)                                   mdseg_softmax_nchw
 *     probs = einsum('bchw,nc->bnhw', pred, Adj)                  mdseg_proj_fwd on `pred`
 *     probs = F.interpolate(probs, label size, bilinear, align_corners=True);  loss = -log(probs)[label]
 *                                                                 mdseg_up_nll_fwd (no [B,C,H,W] tensor)
 * then mdseg_ohem_select on loss_px, and backward:
 *     d loss / d probs_low                                        mdseg_up_nll_bwd (tent gather, no atomics)
 *     d loss / d pred = Adj^T (.)                                 mdseg_proj_bwd
 *     d loss / d x    = pred * (dpred - sum_c pred_c dpred_c)     mdseg_softmax_bwd_nchw */
/* pred[b, c, p] = softmax_c x[b, :, p];  x: [n_images, C, hw] of `dtype`, pred fp32 */
int mdseg_softmax_nchw(const void* x, int dtype, int n_images, int C, int64_t hw, float* pred, void* stream);
/* dx[b, c, p] = pred * (dpred - sum_c pred * dpred);  dx of dx_dtype, may alias dpred when fp32 */
int mdseg_softmax_bwd_nchw(const float* pred, const float* dpred, int n_images, int C, int64_t hw, void* dx,
                           int dx_dtype, void* stream);
/* loss_px[b, Y, X] = -log(bilinear_ac(src[d][b, label])(Y, X)), 0 for ignored pixels, -1 for images of no dataset;
 * OHEM counters (n_valid, n_hard, sum_hard, n_px) are accumulated into the image's segment as mdseg_up_ce_fwd does.
 * src: fp32 projected probabilities (layout as mdseg_src_table). */
int mdseg_up_nll_fwd(const mdseg_src_table* src /*host*/, const int32_t* dataset_ids, const void* labels,
                     int label_dtype, int n_images, int h, int w, int H, int W, int ignore, float* loss_px,
                     mdseg_ohem_state* states, int32_t* err_flag, void* stream);
/* dst[d][b, n, y, x] += sum over selected label pixels of class n under the tent of (y, x) of -w * tent / prob;
 * dst: fp32 planes shaped like src, ZERO-INITIALISED by the caller; w = grad_out[seg] * grad_scale / |S|. */
int mdseg_up_nll_bwd(const mdseg_src_table* src /*host*/, const int32_t* dataset_ids, const void* labels,
                     int label_dtype, int n_images, int h, int w, int H, int W, int ignore, const float* loss_px,
                     const mdseg_ohem_state* states, const float* grad_out, float grad_scale,
                     const mdseg_src_table* dst /*host*/, void* stream);

/* ---- a5: index lists of a column-one-hot 0/1 bi_graph, built on the device ---------------------------------
 * The SEG stage's graphs (lib/models/ltbgnn_direct_learn.py:426-439, ClassRemap.getRemapMatrix lib/class_remap.py:
 * 176-183) are walked as CSR / CSC lists by mdseg_proj_* and mdseg_mds_bwd.  A caller that knows the kind declares it
 * and gets the lists without a device -> host copy of the matrix: G fp32 [C_ds, C_uni] row-major; buf:
 * mdseg_graph_build_onehot_ints(C_ds, C_uni) ints holding, each rounded up to a multiple of 4 ints and in this order,
 * csr_ptr [C_ds + 1], csc_ptr [C_uni + 1], csr4_ptr [C_ds + 1], csr_col [C_uni], csc_row [C_uni],
 * csr4_col [C_uni + 3 C_ds], scratch [C_uni] (the field meanings of mdseg_sparse_graph).  A matrix with a value other
 * than 0 / 1 or with two entries in a column sets MDSEG_ERR_GRAPH_KIND in err_flag. */
size_t mdseg_graph_build_onehot_ints(int C_ds, int C_uni);
int mdseg_graph_build_onehot(const float* G, int C_ds, int C_uni, int* buf, int32_t* err_flag, void* stream);

/* ---- f2: the prototype head and the dense projection for 16-bit operands on TMA + tcgen05 ------------------------
 * y[b, n, p] = sum_c G_d[n, c] x[b, c, p], d = dataset_ids[b], and its two adjoints.  With one operand and
 * dataset_ids = NULL this is the prototype head torch.einsum('bchw,nc->bnhw', feats, unify_prototype)
 * (lib/models/semseg.py:325-333,342-343; lib/loss/loss_cross_datasets.py:950,961,971) under amp.autocast, the
 * prototypes in the role of G; with one operand per dataset it is the DENSE bipartite projection of 16-bit unified
 * logits (GNN stage, loss_cross_datasets.py:997-1006); with folded prototypes (bi_graph @ unify_prototype in the role of
 * G, the features in the role of x) it is both at once.
 * x: bf16 / fp16, hw % 8 == 0, 16-byte aligned, in `layout`: MDSEG_NCHW [n_images, C_uni, hw] (read by TMA as an
 * MN-major UMMA operand — no thread touches it) or MDSEG_NHWC [n_images, hw, C_uni] (channels_last; C_uni % 8 == 0, the
 * 16-byte TMA pixel stride).  y and dy16 are planar in either layout.  Every output for MDSEG_NHWC is bit-identical to
 * the one for MDSEG_NCHW on x made NCHW-contiguous (same products, same K order, same reduction order).
 * graphs_t / graphs_tt: host arrays of n_datasets device pointers; operand d in the dtype of x, row-major
 * [n_tiles * NT, ldb] with NT = mdseg_head_tc16_tile(rows) (ldb % 8 == 0, rows and columns past the matrix zero);
 * a NULL entry skips the dataset. */
int mdseg_head_tc16_tile(int N);
/* graphs_t[d] = G_d [C_ds[d], C_uni] (ldb >= C_uni).  y: fp32 [n_images, y_cmax, hw]; rows of images whose dataset is
 * skipped are untouched. */
int mdseg_proj_fwd_tc16(const void* x, int dtype, int layout, int n_images, int C_uni, int64_t hw,
                        const void* const* graphs_t, int ldb, const int* C_ds /*host*/, int n_datasets,
                        const int32_t* dataset_ids, float* y, int y_cmax, void* stream);
/* The two adjoints (autograd replay of the einsums under amp.autocast).
 * dy16: [n_images, y_cmax, hw] in the dtype of x, planes >= C_ds[dataset] of an image ZERO.
 * mdseg_proj_bwd_tc16: dx[b, c, p] = sum_n G_d[n, c] dy16[b, n, p].  graphs_tt[d] = G_d transposed, [C_uni, C_ds[d]]
 * (ldb >= y_cmax).  dx: fp32 or the dtype of dy16, in `layout`, fully written (zeros for images whose dataset id is out
 * of range).
 * mdseg_proj_bwd_graph_tc16: dG[d][n, c] = sum over the images b of dataset d and pixels p of dy16[b, n, p] x[b, c, p]:
 * split-K over pixel slabs, fixed-order reduction per dataset of the per-slab partials in `workspace` (deterministic).
 * dG: fp32 [n_datasets, y_cmax, C_uni], fully overwritten (zeros for a dataset without images).  dataset_ids = NULL
 * with n_datasets = 1 sums over every image (d prototype of the head). */
int mdseg_proj_bwd_tc16(const void* dy16, int dtype, int layout, int n_images, int y_cmax, int64_t hw,
                        const void* const* graphs_tt, int ldb, int C_uni, int n_datasets, const int32_t* dataset_ids,
                        void* dx, int dx_dtype, void* stream);
size_t mdseg_proj_bwd_graph_tc16_workspace_bytes(int n_images, int C_uni, int64_t hw, int y_cmax);
int mdseg_proj_bwd_graph_tc16(const void* dy16, const void* x, int dtype, int layout, int n_images, int C_uni, int64_t hw,
                              int y_cmax, const int32_t* dataset_ids, int n_datasets, float* dG, void* workspace,
                              size_t workspace_bytes, void* stream);

/* ---- MscEvalCrop (evaluate.py:650-753): sliding-window evaluation ------------------------------------------
 * probs[c, y0 + y, x0 + x] += g(softmax_c(logits)[c, y, x] (+ softmax_c(logits_flip)[c, y, cw - 1 - x])) for one chip
 * [C, ch, cw] inside the scale-level map probs [C, PH, PW] (fp32).  logits_flip may be NULL; exp_after != 0 applies
 * exp() to the summed probabilities, as the reference does when flip is on (evaluate.py:689). */
int mdseg_eval_chip_accum(const void* logits, const void* logits_flip, int dtype, int C, int ch, int cw, float* probs,
                          int PH, int PW, int y0, int x0, int exp_after, void* stream);
/* dst[c] (+)= F.interpolate(src[c, y0:y0+sh, x0:x0+sw], (H, W), bilinear, align_corners=True)  (evaluate.py:722-724);
 * first != 0 overwrites dst. */
int mdseg_prob_resize_accum(const float* src, int C, int PH, int PW, int y0, int x0, int sh, int sw, float* dst, int H,
                            int W, int first, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MDSEG_H_ */
