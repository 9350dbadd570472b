/*
 * pnce.h -- C ABI of libpnce.so, the B200 (sm_100a) PatchNCE hot path.
 *
 * The reference (Cameronr11/GAN-Variant-Research) has no FFI: its seam is two Python symbols in
 * GAN_Variant1/losses/patchnce_cut.py (SURVEY.md section 8b).  These entry points are what a
 * binding for that seam calls; each one cites the reference lines it replaces.  The Python host
 * (gan_variant_research_b200/patchnce.py) binds them with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions (all entry points):
 *   - every pointer named dev_* / inside pnce_layer_t is a DEVICE pointer owned by the caller
 *     (torch tensors in practice); the library allocates nothing persistent on the device path;
 *   - every call is asynchronous on `stream` (a cudaStream_t / CUstream passed as void*), performs
 *     no host synchronisation and is CUDA-graph capturable;
 *   - return value: 0 on success, a negative pnce_status_t otherwise; nothing throws;
 *   - thread-safe per (workspace, stream) pair.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     PNCE_ERR_CUDA.
 *   - kernels are launched with programmatic dependent launch allowed (every kernel waits for its
 *     prerequisite grids before its first global access, so stream order is what the caller sees);
 *     the environment variable PNCE_PDL=0, read once per process, launches them the ordinary way.
 */
#ifndef PNCE_H_
#define PNCE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PNCE_ABI_VERSION 10
#define PNCE_MAX_LAYERS 8      /* nce_layers per call (reference config uses 5 ids -> 4 maps)   */
#define PNCE_MAX_PATCHES 4096  /* P = min(num_patches, H*W)  patchnce_cut.py:60; argument check only: the
                                * kernels take P <= 1024 (tensor cores, C <= 256) or P <= 1280 (fp32 CUDA cores),
                                * PNCE_ERR_UNSUPPORTED beyond                                                  */
#define PNCE_MAX_CHANNELS 1024

typedef enum {
  PNCE_OK = 0,
  PNCE_ERR_ARG = -1,        /* NULL pointer, bad shape, too many layers ...                      */
  PNCE_ERR_UNSUPPORTED = -2,/* shape outside the compiled limits                                 */
  PNCE_ERR_WORKSPACE = -3,  /* workspace too small / misaligned                                  */
  PNCE_ERR_CUDA = -4,       /* a CUDA runtime call failed (see pnce_last_cuda_error)             */
  PNCE_ERR_ALIGN = -5       /* a tensor base pointer is not element-aligned                      */
} pnce_status_t;

typedef enum { PNCE_F32 = 0, PNCE_F16 = 1, PNCE_BF16 = 2 } pnce_dtype_t;

/* How the per-image logits / dQ contractions are evaluated.
 *   PNCE_MATH_SIMT_F32 : fp32 FFMA, bit-for-bit the reference's fp32 op order up to summation order
 *   PNCE_MATH_TC_BF16X3: tcgen05 bf16 tensor cores, operands split hi+lo (3 MMAs), fp32 accumulate
 *   PNCE_MATH_TC_BF16  : tcgen05 bf16 single pass (the AMP regime of the reference: fp16 GEMM)    */
typedef enum { PNCE_MATH_SIMT_F32 = 0, PNCE_MATH_TC_BF16X3 = 1, PNCE_MATH_TC_BF16 = 2 } pnce_math_t;

/* One nce layer: a pair of contiguous NCHW feature maps and the ids sampled on it.
 * Replaces the (src_feat, tgt_feat) pair zipped at patchnce_cut.py:36 plus patch_ids of :63.   */
typedef struct pnce_layer {
  const void*    src;   /* (B,C,H,W) source features, no gradient          patchnce_cut.py:142 */
  const void*    tgt;   /* (B,C,H,W) target features                       patchnce_cut.py:145 */
  void*          dtgt;  /* (B,C,H,W) dense d loss / d tgt, same dtype; written by pnce_bwd only  */
  const int64_t* ids;   /* (P,) int64 in [0,H*W), with replacement, shared by the batch     :63 */
  int32_t C, H, W, P;
} pnce_layer_t;

int         pnce_abi_version(void);
const char* pnce_status_string(int status);
const char* pnce_last_cuda_error(void);

/* Bytes of device scratch pnce_fwd/pnce_bwd need for this problem (ids order, normalised rows,
 * d rows, id bitmap ...).  Contents need no initialisation.                                    */
int pnce_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch, size_t* bytes);

/* Forward of PatchNCELoss.forward for all layers in one pass        patchnce_cut.py:25-110
 *   gather (:66-74) -> L2 normalise (:77-78) -> per-image logits/tau, clamp (:85-88)
 *   -> diagonal CE (:91-94) -> non-finite guards (:97-108) -> batch mean, layer mean (:103,:40)
 * and, fused, the backward of all of that up to the per-patch gradient rows (unit upstream
 * gradient), kept in the workspace for pnce_bwd.  Logits never reach HBM.
 *   dev_loss_out : float[1 + n_layers]  -> [0] total loss, [1+l] layer losses
 *   dev_nonfinite: int[2]               -> [0] number of (layer,image) pairs whose loss was replaced
 *                                          by 0 (the reference prints a warning for each, :98);
 *                                          [1] internal kernel-protocol timeout flag (must read 0; when it is
 *                                          raised dev_loss_out[0] is NaN as well, so the failure is visible in-band) */
int pnce_fwd(const pnce_layer_t* layers, int n_layers, int batch, int dtype, float temperature,
             int math_mode, void* dev_workspace, size_t workspace_bytes, float* dev_loss_out,
             int* dev_nonfinite, void* stream);

/* The id bookkeeping (sorted ids, ranks, per-tile slot ranges) as a step of its own: pnce_plan_ids sorts the
 * ids of every layer into a caller-owned buffer of pnce_plan_bytes bytes (only layers[l].ids, C, H, W, P are
 * read); pnce_fwd_planned / pnce_bwd_planned then take it instead of sorting themselves.  The ids
 * (patchnce_cut.py:63) depend on nothing but the generator state, so a caller can draw AND sort them on a
 * side stream while the GPU is still busy with whatever precedes the loss -- 10 us less at the head of the
 * step.  Tensor-core math modes only (PNCE_ERR_UNSUPPORTED otherwise).                               */
int pnce_plan_bytes(const pnce_layer_t* layers, int n_layers, size_t* bytes);
int pnce_plan_ids(const pnce_layer_t* layers, int n_layers, void* dev_plan, size_t plan_bytes, void* stream);
int pnce_fwd_planned(const pnce_layer_t* layers, int n_layers, int batch, int dtype, float temperature,
                     int math_mode, void* dev_workspace, size_t workspace_bytes, void* dev_plan,
                     size_t plan_bytes, float* dev_loss_out, int* dev_nonfinite, void* stream);
int pnce_bwd_planned(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int math_mode,
                     void* dev_workspace, size_t workspace_bytes, void* dev_plan, size_t plan_bytes,
                     const float* dev_grad_out, void* stream);

/* The id draw of patchnce_cut.py:60-63 done BY THE LIBRARY, inside the id-sort launch: layers[l].ids must point to
 * WRITABLE int64[P] buffers and receives, for l = 0, 1, ..., exactly what l-th call of
 *     torch.randint(0, H*W, (P,), device='cuda')
 * returns when the CUDA generator's Philox state is (philox_seed, philox_offset): ATen's random_from_to kernel gives
 * element i the first 32-bit word of Philox4x32-10(key = seed, subsequence = i, counter = offset / 4) modulo H*W, and
 * every call advances the offset by 4 -- so layer l draws at philox_offset + 4 l and the CALLER advances its generator
 * by 4 * n_layers (torch: gen.set_offset(gen.get_offset() + 4 * n)) to keep the RNG stream aligned with the reference's
 * training step.  Saves the n_layers randint launches (and their host time) per step; the Python host validates the
 * law against torch.randint once per process and falls back to calling torch.randint if it ever stops holding.
 *   pnce_fwd_draw      : pnce_fwd with the draw (tensor-core math modes; PNCE_ERR_UNSUPPORTED otherwise)
 *   pnce_plan_ids_draw : pnce_plan_ids with the draw (then pnce_fwd_planned / pnce_bwd_planned)
 *   pnce_draw_ids      : the draw alone (only layers[l].ids, H, W, P are read)                                */
int pnce_fwd_draw(const pnce_layer_t* layers, int n_layers, int batch, int dtype, float temperature,
                  int math_mode, void* dev_workspace, size_t workspace_bytes, unsigned long long philox_seed,
                  unsigned long long philox_offset, float* dev_loss_out, int* dev_nonfinite, void* stream);
int pnce_plan_ids_draw(const pnce_layer_t* layers, int n_layers, unsigned long long philox_seed,
                       unsigned long long philox_offset, void* dev_plan, size_t plan_bytes, void* stream);
int pnce_draw_ids(const pnce_layer_t* layers, int n_layers, unsigned long long philox_seed,
                  unsigned long long philox_offset, void* stream);

/* Backward: writes every layers[l].dtgt densely (zero off the sampled positions, duplicate ids
 * accumulated) scaled by the upstream gradient *dev_grad_out (NULL = 1.0).  `math_mode` and the
 * workspace must be the ones given to the matching pnce_fwd.  Replaces the autograd
 * chain of SURVEY.md section 8 row a11 (index_put_ / select_backward / zeros + adds).           */
int pnce_bwd(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int math_mode,
             void* dev_workspace, size_t workspace_bytes, const float* dev_grad_out, void* stream);

/* ---- channels-last maps (an extension: the reference's `feat.view(B, C, -1)`, patchnce_cut.py:56, only takes
 * contiguous NCHW) ------------------------------------------------------------------------------------------------
 * With layout = PNCE_LAYOUT_NHWC every layers[l].src / tgt / dtgt is the storage of a torch.channels_last tensor:
 * logical shape (B, C, H, W), memory order (B, H, W, C) -- a sampled patch is then C CONTIGUOUS values instead of C
 * values in C different DRAM lines, and the gather reads exactly the bytes it uses (DESIGN.md 4.7).  Ids, loss and
 * gradient values obey the same law as the NCHW entry points (the oracle on the permuted data).  Tensor-core math
 * modes and their shape envelope only (PNCE_ERR_UNSUPPORTED otherwise).
 *   pnce_fwd_ex = pnce_fwd (plan == NULL, philox == NULL), pnce_fwd_draw (philox = {seed, offset}) or
 *                 pnce_fwd_planned (plan != NULL, from pnce_plan_ids / pnce_plan_ids_draw) with a layout;
 *   pnce_bwd_ex = pnce_bwd / pnce_bwd_planned with a layout.  PNCE_LAYOUT_NCHW makes them the calls above.        */
typedef enum { PNCE_LAYOUT_NCHW = 0, PNCE_LAYOUT_NHWC = 1 } pnce_layout_t;
int pnce_fwd_ex(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int layout, float temperature,
                int math_mode, void* dev_workspace, size_t workspace_bytes, void* dev_plan, size_t plan_bytes,
                const unsigned long long* philox_seed_offset, float* dev_loss_out, int* dev_nonfinite, void* stream);
int pnce_bwd_ex(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int layout, int math_mode,
                void* dev_workspace, size_t workspace_bytes, void* dev_plan, size_t plan_bytes,
                const float* dev_grad_out, void* stream);

/* ---- minibatch negatives: upstream CUT's nce_includes_all_negatives_from_minibatch (ABI 6) --------------------------
 * The reference's configs/train_gan_cutpp.yaml:80 declares patchnce.nce_includes_all_negatives_from_minibatch; upstream
 * CUT implements it as batch_dim_for_bmm = 1, i.e. the loss of patchnce_cut.py:42-110 applied to ONE "image" whose rows
 * are the whole batch.  Per layer, with N = B * P rows in image-major order:
 *   Q, K = normalize(tgt / src patches of every image) (:77-78), Z = clamp(Q K^T / tau, -50, 50) (N x N, :85-88),
 *   loss_l = mean over the N rows of CE(Z_i, i) (:91-94), the image guard of :97-99 applied to that single group (a
 *   non-finite group contributes 0 and its rows get a zero upstream gradient), total = sum_l loss_l / n_layers (:40).
 * d loss / d tgt keeps the factor 1 / (P B n_layers); keys carry no gradient (:142).  The N x N logits never leave the
 * SM (k_loss_tc_mb).  Under data parallelism the negatives are those of the caller's shard (as upstream CUT under DDP);
 * the pnce_mb_shard_* calls below contrast with every rank's keys instead.
 * Tensor-core math modes only; P <= 1024, C <= 256 and B * round_up(P, 128) <= 65536 per layer (PNCE_ERR_UNSUPPORTED
 * otherwise).
 *   pnce_mb_workspace_bytes : bytes of the workspace pnce_mb_fwd needs
 *   pnce_mb_fwd             : the arguments of pnce_fwd_ex (layout, id plan or Philox draw -- same ids, same generator
 *                             advance as pnce_fwd_ex); dev_nonfinite[0] counts the LAYERS whose loss was replaced by 0.
 *                             The backward is pnce_bwd_ex on the same workspace, layout and math mode.            */
int pnce_mb_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch, size_t* bytes);
int pnce_mb_fwd(const pnce_layer_t* layers, int n_layers, int batch, int dtype, int layout, float temperature,
                int math_mode, void* dev_workspace, size_t workspace_bytes, void* dev_plan, size_t plan_bytes,
                const unsigned long long* philox_seed_offset, float* dev_loss_out, int* dev_nonfinite, void* stream);

/* ---- global negatives: minibatch negatives across data-parallel ranks (ABI 7) ---------------------------------------
 * configs/train_gan_cutpp.yaml:80 (nce_includes_all_negatives_from_minibatch) with the batch sharded over `world` ranks,
 * rank r holding global images r * batch_local ... r * batch_local + batch_local - 1, every rank using the same ids.
 * Per layer, rank r's batch_local * P query rows are contrasted with the keys of ALL world * batch_local images
 * (patchnce_cut.py:42-110 on the group of world * batch_local * P rows, row i's positive = the key of the same global
 * (image, patch)); rank r's loss is the mean row CE over its own rows, so the mean of the ranks' losses is the one-GPU
 * minibatch loss of the global batch, and d loss_r / d tgt_r divided by world is the one-GPU gradient of shard r.  The
 * guard is global: a non-finite query row on any rank, or a non-finite key, zeroes the layer on every rank
 * (dev_nonfinite[0] counts guarded layers).  The envelope is pnce_mb_fwd's, applied to the global batch.  The library
 * has no collective of its own; the caller exchanges the slots:
 *   pnce_mb_shard_workspace_bytes : total bytes, and where the `world` slots start (slot_offset, always
 *                                   pnce_mb_workspace_bytes(batch_local)) and their stride (slot_bytes, 256-aligned)
 *   pnce_mb_shard_keys            : the id prep (plan or Philox draw as in pnce_fwd_ex) and the gather; fills slot `rank`
 *                                   with this rank's keys and its "a query row is non-finite" flags
 *   -- the caller all-gathers the slot region [slot_offset, slot_offset + world * slot_bytes) in place --
 *   pnce_mb_shard_loss            : logits, CE and d loss / d q over every slot's keys (k_loss_tc_mb_gn); the backward is
 *                                   pnce_bwd_ex(batch_local) on the same workspace
 * Keys carry no gradient (:142), so the backward needs no exchange.  world < 1, rank outside [0, world), dtype or layout
 * out of range: PNCE_ERR_ARG; simt_f32 or a global batch outside the envelope: PNCE_ERR_UNSUPPORTED; NULL or short
 * workspace: PNCE_ERR_WORKSPACE -- all before any CUDA call.                                                          */
int pnce_mb_shard_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch_local, int world, size_t* bytes,
                                  size_t* slot_offset, size_t* slot_bytes);
int pnce_mb_shard_keys(const pnce_layer_t* layers, int n_layers, int batch_local, int dtype, int layout, int world,
                       int rank, int math_mode, void* dev_workspace, size_t workspace_bytes, void* dev_plan,
                       size_t plan_bytes, const unsigned long long* philox_seed_offset, void* stream);
int pnce_mb_shard_loss(const pnce_layer_t* layers, int n_layers, int batch_local, int dtype, int layout, int world,
                       int rank, float temperature, int math_mode, void* dev_workspace, size_t workspace_bytes,
                       void* dev_plan, size_t plan_bytes, float* dev_loss_out, int* dev_nonfinite, void* stream);

/* ---- north-star module split (SURVEY.md section 8b / row a13) ------------------------------ */

/* PatchSampleF(use_mlp=False) forward for one map: rows_out (B*P, C) fp32 = L2-normalised patches
 * in ids order, inv_out (B*P) = 1/||x|| (negative -1/eps when ||x|| < eps, NaN for a non-finite
 * row).  inv_out == NULL selects the RAW gather (no normalisation) that feeds the netF head.
 *                                                                         patchnce_cut.py:53-78 */
int pnce_sample_fwd(const void* dev_feat, int dtype, int batch, int C, int H, int W,
                    const int64_t* dev_ids, int P, float* dev_rows_out, float* dev_inv_out,
                    void* stream);

/* Backward of pnce_sample_fwd: d rows (B*P, C) fp32 -> dense d feat (B,C,H,W) in `dtype`.
 * dev_rows == dev_inv == NULL: backward of the raw gather (pure scatter, duplicates accumulated). */
int pnce_sample_bwd_workspace_bytes(int batch, int C, int H, int W, int P, size_t* bytes);
int pnce_sample_bwd(const float* dev_drows, const float* dev_rows, const float* dev_inv, int dtype,
                    int batch, int C, int H, int W, const int64_t* dev_ids, int P,
                    void* dev_workspace, size_t workspace_bytes, void* dev_dfeat, void* stream);

/* PatchNCELoss(feat_q, feat_k) on already-normalised rows (B*P, D) fp32, rows grouped per image:
 * loss_out[0] = mean_b mean_i CE_i (:83-103); dq_out = d loss / d feat_q for unit upstream;
 * dk_out optional (NULL when feat_k is detached, as in the reference :142).                     */
int pnce_rows_loss_workspace_bytes(int batch, int P, int D, size_t* bytes);
int pnce_rows_loss_fwd_bwd(const float* dev_q, const float* dev_k, int batch, int P, int D,
                           float temperature, int math_mode, void* dev_workspace,
                           size_t workspace_bytes, float* dev_loss_out, int* dev_nonfinite,
                           float* dev_dq_out, float* dev_dk_out, void* stream);

/* The same loss for EVERY layer of a PatchSampleF output in one call (upstream CUT loops `crit(f_q, f_k)` over the
 * layers and averages: one pack launch + one tcgen05 loss launch instead of one pair per layer, and the light layers
 * fill the SMs the heavy ones leave idle).  loss_out[0] = mean over layers, loss_out[1 + l] = layer l;
 * rows[l].dq = d loss_out[0] / d q_l for unit upstream (the 1/n_layers factor included).  Tensor-core modes only,
 * P <= 256 and D <= 256 for every layer (PNCE_ERR_UNSUPPORTED otherwise: call the per-layer entry).   patchnce_cut.py:36-40, :83-103 */
typedef struct pnce_rows {
  const float* q;     /* (B*P, D) fp32 rows, grouped per image, already L2-normalised */
  const float* k;     /* (B*P, D) fp32 keys (no gradient: the reference detaches them, :142) */
  float*       dq;    /* (B*P, D) fp32, written */
  int32_t      P, D;
} pnce_rows_t;
int pnce_rows_loss_multi_workspace_bytes(const pnce_rows_t* rows, int n_layers, int batch, size_t* bytes);
int pnce_rows_loss_multi_fwd_bwd(const pnce_rows_t* rows, int n_layers, int batch, float temperature, int math_mode,
                                 void* dev_workspace, size_t workspace_bytes, float* dev_loss_out, int* dev_nonfinite,
                                 void* stream);
/* pnce_rows_loss_multi_fwd_bwd with minibatch negatives (see pnce_mb_fwd): per layer, every row of feat_q is contrasted
 * with the B * P rows of feat_k, label = its own row (upstream CUT's PatchNCELoss with batch_dim_for_bmm = 1 on the
 * PatchSampleF output, patchnce_cut.py:83-103 on one group).  P <= 256, D <= 256, B * round_up(P, 128) <= 65536 per
 * layer; rows[l].dq 32-byte aligned (PNCE_ERR_ALIGN otherwise); dev_nonfinite[0] counts guarded layers.            */
int pnce_rows_mb_workspace_bytes(const pnce_rows_t* rows, int n_layers, int batch, size_t* bytes);
int pnce_rows_mb_fwd_bwd(const pnce_rows_t* rows, int n_layers, int batch, float temperature, int math_mode,
                         void* dev_workspace, size_t workspace_bytes, float* dev_loss_out, int* dev_nonfinite,
                         void* stream);
/* ---- row route with global negatives: minibatch negatives across data-parallel ranks (ABI 10) -----------------------
 * The law of pnce_mb_shard_* on rows used as given.  `world` ranks each hold batch_local images, rank r global images
 * r * batch_local ... r * batch_local + batch_local - 1, every rank with the same ids; rows[l].q / .k are the rank's
 * (batch_local * P, D) rows of layer l, grouped per image and already L2-normalised (PatchSampleF's output).  Per layer,
 * rank r's query rows are contrasted with the key rows of ALL world * batch_local images in global (image, patch) order;
 * row i's positive is the key of the same global row; Z = clamp(q k^T / tau, -50, 50).  Rank r's loss is the mean row
 * CE over its own rows, then the mean over layers, so the mean of the ranks' losses is pnce_rows_mb_fwd_bwd's loss on
 * the global rows and rows[l].dq / world is that call's d loss / d q restricted to shard r.  The guard is global: a
 * non-finite query row on any rank, or a non-finite key, zeroes the layer on every rank (its dq rows are 0, as one GPU
 * writes them); dev_nonfinite[0] counts guarded layers.  The envelope is pnce_rows_mb_fwd_bwd's applied to the global
 * batch: tensor-core math, P <= 256, D <= 256, world * batch_local * round_up(P, 128) <= 65536 per layer.
 *   pnce_rows_mb_shard_workspace_bytes : total bytes, where the `world` slots start (slot_offset, always
 *                                        pnce_rows_mb_workspace_bytes(batch_local)) and their stride (slot_bytes,
 *                                        256-aligned; the slot format of pnce_mb_shard_workspace_bytes with C = D)
 *   pnce_rows_mb_shard_keys            : the row pack (k_rows_pack): queries into the prefix, keys straight into slot
 *                                        `rank`, with this rank's "a query row is non-finite" flags (reads q, k)
 *   -- the caller all-gathers the slot region [slot_offset, slot_offset + world * slot_bytes) in place --
 *   pnce_rows_mb_shard_loss            : logits, CE and d loss / d q over every slot's keys (k_loss_tc_mb_gn); writes
 *                                        rows[l].dq row-major (32-byte aligned: PNCE_ERR_ALIGN otherwise)
 * Keys carry no gradient, so nothing is exchanged for the backward.  world < 1, rank outside [0, world), math mode out of
 * range, NULL rows / loss or a bad shape: PNCE_ERR_ARG; simt_f32 or a global batch outside the envelope:
 * PNCE_ERR_UNSUPPORTED; NULL, misaligned or short workspace: PNCE_ERR_WORKSPACE -- all before any CUDA call.           */
int pnce_rows_mb_shard_workspace_bytes(const pnce_rows_t* rows, int n_layers, int batch_local, int world, size_t* bytes,
                                       size_t* slot_offset, size_t* slot_bytes);
int pnce_rows_mb_shard_keys(const pnce_rows_t* rows, int n_layers, int batch_local, int world, int rank, int math_mode,
                            void* dev_workspace, size_t workspace_bytes, void* stream);
int pnce_rows_mb_shard_loss(const pnce_rows_t* rows, int n_layers, int batch_local, int world, int rank,
                            float temperature, int math_mode, void* dev_workspace, size_t workspace_bytes,
                            float* dev_loss_out, int* dev_nonfinite, void* stream);

/* All maps of one PatchSampleF call in ONE launch each way (the per-map entry points above cost a launch per
 * layer and leave the GPU half empty on the small layers): forward reads feat / ids and writes rows (and inv,
 * NULL for all layers = raw patches); backward reads drows / rows / inv / ids and writes dfeat densely.   */
typedef struct pnce_sample {
  const void*    feat;   /* (B,C,H,W), dtype of the call                        forward  */
  const int64_t* ids;    /* (P) positions in [0, H*W)                           both     */
  float*         rows;   /* (B*P, C) fp32: written by forward, read by backward (NULL there = raw) */
  float*         inv;    /* (B*P) norm bookkeeping of the forward, or NULL (raw patches)           */
  const float*   drows;  /* (B*P, C) incoming gradient                          backward */
  void*          dfeat;  /* (B,C,H,W) dense gradient, dtype of the call         backward */
  int32_t        C, H, W, P;
} pnce_sample_t;
int pnce_sample_multi_fwd(const pnce_sample_t* maps, int n_maps, int batch, int dtype, void* stream);
int pnce_sample_multi_bwd_workspace_bytes(const pnce_sample_t* maps, int n_maps, int batch, size_t* bytes);
int pnce_sample_multi_bwd(const pnce_sample_t* maps, int n_maps, int batch, int dtype, void* dev_workspace,
                          size_t workspace_bytes, void* stream);

/* ---- netF head, fused (north-star pieces 3-5; absent from the reference: SURVEY.md 8 row a13) ---
 * PatchSampleF(use_mlp=True): raw gather -> Linear(C_l, nc) -> ReLU -> Linear(nc, nc) -> L2 normalise for the
 * src (k, no gradient) and tgt (q) patches of every layer, then the same logits / diagonal CE as
 * pnce_fwd on the head's output; all contractions on tcgen05 (math_mode TC_BF16X3 or TC_BF16).
 * Supported: nc = 128 or 256, P <= 1024, C <= 256.  Weights are fp32, nn.Linear layout (out, in).     */
typedef struct pnce_head {
  const float* w1;  /* (nc, C)  */
  const float* b1;  /* (nc)     */
  const float* w2;  /* (nc, nc) */
  const float* b2;  /* (nc)     */
  float* dw1;       /* outputs of pnce_head_bwd, same shapes, overwritten; may be NULL for pnce_head_fwd */
  float* db1;
  float* dw2;
  float* db2;
} pnce_head_t;

int pnce_head_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch, int nc, size_t* bytes);
int pnce_head_fwd(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype,
                  int nc, float temperature, int math_mode, void* dev_workspace, size_t workspace_bytes,
                  float* dev_loss_out, int* dev_nonfinite, void* stream);
/* Writes every layers[l].dtgt densely and every heads[l].d*, all scaled by *dev_grad_out (NULL = 1). */
int pnce_head_bwd(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype,
                  int nc, int math_mode, void* dev_workspace, size_t workspace_bytes,
                  const float* dev_grad_out, void* stream);
/* The same backward in two calls, for data-parallel callers: _params writes every heads[l].d* (layers[l].dtgt
 * may be NULL), _dense then writes every layers[l].dtgt.  Between the two the caller can start the all-reduce
 * of the head gradients on another stream, so that the only collective of the path (SURVEY.md section 8e)
 * runs under the HBM-bound dense kernel instead of after it.  Same workspace and arguments for both.      */
int pnce_head_bwd_params(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype,
                         int nc, int math_mode, void* dev_workspace, size_t workspace_bytes,
                         const float* dev_grad_out, void* stream);
int pnce_head_bwd_dense(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype,
                        int nc, int math_mode, void* dev_workspace, size_t workspace_bytes,
                        const float* dev_grad_out, void* stream);

/* The fused head on channels-last maps (layout as in pnce_fwd_ex); phases: 1 = pnce_head_bwd_params, 2 = pnce_head_bwd_dense,
 * 3 = pnce_head_bwd.                                                                                              */
int pnce_head_fwd_ex(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype, int layout,
                     int nc, float temperature, int math_mode, void* dev_workspace, size_t workspace_bytes,
                     float* dev_loss_out, int* dev_nonfinite, void* stream);
int pnce_head_bwd_ex(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype, int layout,
                     int phases, int nc, int math_mode, void* dev_workspace, size_t workspace_bytes,
                     const float* dev_grad_out, void* stream);

/* ---- netF head with minibatch negatives (ABI 8) -----------------------------------------------------------------------
 * The law of pnce_mb_fwd on the head's output: per layer, with N = B * P rows in image-major order and the ids shared by
 * the batch, q = normalize(netF(raw tgt patches)), k = normalize(netF(raw src patches)) (no gradient),
 * Z = clamp(q k^T / tau, -50, 50) (N x N), loss_l = mean over the N rows of CE(Z_i, i), total = sum_l loss_l / n_layers.
 * A non-finite layer contributes 0 and its rows get a zero upstream gradient (so that layer's head gradients are 0);
 * dev_nonfinite[0] counts the guarded LAYERS.  d loss / d tgt keeps the factor 1 / (B P n_layers); the head learns
 * through q only.  At B = 1 this is pnce_head_fwd_ex's loss.
 *   pnce_head_mb_workspace_bytes : bytes of the workspace; PNCE_ERR_UNSUPPORTED outside the head envelope (nc = 128 or
 *                                  256, P <= 1024, C <= 256) or the minibatch one (B * round_up(P, 128) <= 65536)
 *   pnce_head_mb_fwd             : the arguments of pnce_head_fwd_ex; the same prep, weight blobs, gather and head
 *                                  GEMMs, then the minibatch loss kernel (k_loss_tc_mb).  simt_f32 and shapes outside
 *                                  the envelope: PNCE_ERR_UNSUPPORTED before any CUDA call.
 * A sampled patch (either side) holding a NaN / Inf makes its layer non-finite, as in torch, where ReLU keeps the NaN.
 * The backward is pnce_head_bwd_ex (any phases) on the same workspace, layout and math mode; the workspace is
 * pnce_head_workspace_bytes' layout followed by the raw patches' sums of squares.                                     */
int pnce_head_mb_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch, int nc, size_t* bytes);
int pnce_head_mb_fwd(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch, int dtype, int layout,
                     int nc, float temperature, int math_mode, void* dev_workspace, size_t workspace_bytes,
                     float* dev_loss_out, int* dev_nonfinite, void* stream);

/* ---- netF head with global negatives: minibatch negatives across data-parallel ranks (ABI 9) ------------------------
 * The law of pnce_mb_shard_* on the head's output.  `world` ranks each hold batch_local images, rank r global images
 * r * batch_local ... r * batch_local + batch_local - 1, every rank with the same ids and head parameters.  Per layer,
 * rank r's query rows q = normalize(netF(raw tgt patches)) are contrasted with the keys
 * k = normalize(netF(raw src patches)) (no gradient) of ALL world * batch_local images; row i's positive is the key of
 * the same global (image, patch).  Rank r's loss is the mean row CE over its own rows, so the mean of the ranks' losses
 * is pnce_head_mb_fwd's loss on the global batch, d loss_r / d tgt_r divided by world is the one-GPU gradient of shard
 * r, and the rank-mean of the head gradients is the one-GPU head gradient.  The guard is global: a layer is guarded on
 * every rank exactly when pnce_head_mb_fwd on the global batch guards it (dev_nonfinite[0] counts guarded layers).  The
 * envelope is pnce_head_mb_fwd's, applied to the global batch.  The caller exchanges the slots:
 *   pnce_head_mb_shard_workspace_bytes : total bytes, where the `world` slots start (slot_offset, always
 *                                        pnce_head_mb_workspace_bytes(batch_local)) and their stride (slot_bytes,
 *                                        256-aligned; the slot format of pnce_mb_shard_workspace_bytes with C = nc)
 *   pnce_head_mb_shard_keys            : prep, weight blobs, gather and both head GEMMs; the keys go straight into slot
 *                                        `rank`, with this rank's "a query row is non-finite" flags
 *   -- the caller all-gathers the slot region [slot_offset, slot_offset + world * slot_bytes) in place --
 *   pnce_head_mb_shard_loss            : logits, CE and d loss / d (head output) over every slot's keys
 *                                        (k_loss_tc_mb_gn); the backward is pnce_head_bwd_ex(batch_local, any phases) on
 *                                        the same workspace, layout and math mode
 * Keys carry no gradient, so the backward needs no exchange.  world < 1, rank outside [0, world), dtype, layout or math
 * mode out of range, NULL heads or weights: PNCE_ERR_ARG; simt_f32, nc not 128 / 256 or a global batch outside the
 * envelope: PNCE_ERR_UNSUPPORTED; NULL, misaligned or short workspace: PNCE_ERR_WORKSPACE -- all before any CUDA call.
 * dev_nonfinite may be NULL; when given, [1] receives the tensor-core protocol-timeout flag as in pnce_head_fwd_ex.   */
int pnce_head_mb_shard_workspace_bytes(const pnce_layer_t* layers, int n_layers, int batch_local, int world, int nc,
                                       size_t* bytes, size_t* slot_offset, size_t* slot_bytes);
int pnce_head_mb_shard_keys(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch_local,
                            int dtype, int layout, int nc, int world, int rank, int math_mode, void* dev_workspace,
                            size_t workspace_bytes, int* dev_nonfinite, void* stream);
int pnce_head_mb_shard_loss(const pnce_layer_t* layers, const pnce_head_t* heads, int n_layers, int batch_local,
                            int dtype, int layout, int nc, int world, int rank, float temperature, int math_mode,
                            void* dev_workspace, size_t workspace_bytes, float* dev_loss_out, int* dev_nonfinite,
                            void* stream);

/* ---- PatchSampleF(use_mlp=True).forward(feats, num_patches, patch_ids) as a module of its own (north_star's netF
 * signature; absent from the reference, SURVEY.md section 8 row a13): for every map, raw gather -> Linear(C_l, nc) ->
 * ReLU -> Linear(nc, nc) -> x / max(||x||, 1e-6), all contractions on tcgen05, and its backward.
 *   forward : reads maps[l].feat / ids, writes maps[l].rows (B*P, nc) fp32 -- normalised, row b*P + p <-> ids[p], the
 *             order upstream CUT's PatchSampleF returns -- and maps[l].inv (B*P), the norm bookkeeping of pnce_sample_fwd;
 *   backward: reads maps[l].drows (gradient w.r.t. rows), rows and inv of the forward and the SAME workspace (it holds
 *             the gathered patches, the hidden activations and the sorted ids); writes every heads[l].d* and, unless
 *             every maps[l].dfeat is NULL (maps without gradient), the dense maps[l].dfeat.
 * nc = 128 or 256, P <= 1024, C <= 256; math_mode TC_BF16X3 or TC_BF16; layout as in pnce_fwd_ex.
 * dev_status: int[1], set to 1 on a kernel-protocol timeout (may be NULL).                                        */
int pnce_netf_workspace_bytes(const pnce_sample_t* maps, int n_maps, int batch, int nc, size_t* bytes);
int pnce_netf_fwd(const pnce_sample_t* maps, const pnce_head_t* heads, int n_maps, int batch, int dtype, int layout,
                  int nc, int math_mode, void* dev_workspace, size_t workspace_bytes, int* dev_status, void* stream);
int pnce_netf_bwd(const pnce_sample_t* maps, const pnce_head_t* heads, int n_maps, int batch, int dtype, int layout,
                  int nc, int math_mode, void* dev_workspace, size_t workspace_bytes, int* dev_status, void* stream);

/* ---- "next" row 3 (SURVEY.md section 8f): optimiser-side multi-tensor ops ------------------------------------
 * One launch over a list of fp32 tensors described by device-resident tables (built once by the caller: parameter
 * storage does not move during training): chunk c covers elements [chunk_start[c], chunk_start[c] +
 * pnce_multi_chunk_elems()) of tensor chunk_tensor[c].
 *   mode 0: dst = a * src + b * dst, both products and the sum rounded separately -- EMA.update(), utils/io_ckpt.py:23-29,
 *           with a = 1 - decay, b = decay, dst = shadow, src = param (bit-identical to the reference's expression);
 *   mode 1: dst = src                                   -- EMA.apply_shadow() / restore(), :31-43                 */
int pnce_multi_chunk_elems(void);
int pnce_multi_axpby(float* const* dev_dst, const float* const* dev_src, const long long* dev_numel,
                     const int* dev_chunk_tensor, const long long* dev_chunk_start, int n_chunks, float a, float b,
                     int mode, void* stream);

/* AMPContext.step_optimizer(optimizer, max_grad_norm) of the reference (utils/amp_utils.py:29-41) for an optim.Adam
 * (training/sched_optim.py:20-25): GradScaler.unscale_, clip_grad_norm_, the skip-on-non-finite optimizer.step() and
 * GradScaler.update(), as three launches over the same chunk tables as above (one entry per parameter that has a
 * gradient) and with no host sync: the skip decision, the per-tensor step counters (dev_step[t]: one float each,
 * torch's "capturable" layout) and the loss scale stay on the device.
 *   dev_scale / dev_growth_tracker : GradScaler._scale (float) and ._growth_tracker (int32) device scalars, or both
 *                                    NULL = no scaler (gradients used as they are, never skipped)
 *   max_grad_norm < 0              : no clipping
 *   dev_scratch                    : pnce_amp_adam_scratch_floats(n_chunks) floats, zeroed ONCE by the caller; after
 *                                    the call [1] holds the total gradient norm (before clipping, after unscaling)
 * Arithmetic = ATen's foreach Adam (lerp_, mul_, addcmul_, sqrt, div_, add_, addcdiv_), bias corrections in double:
 * bit-identical to torch whenever the clip coefficient clamps to 1; otherwise the total norm is summed in another
 * order than torch's (norm of per-tensor norms) and values agree to fp32 rounding.  Gradients are left unscaled and
 * clipped, as the reference leaves them; amsgrad / maximize are not supported.                                  */
size_t pnce_amp_adam_scratch_floats(int n_chunks);
int pnce_amp_adam_step(float* const* dev_param, float* const* dev_grad, float* const* dev_exp_avg,
                       float* const* dev_exp_avg_sq, float* const* dev_step, const long long* dev_numel,
                       const int* dev_chunk_tensor, const long long* dev_chunk_start, int n_chunks, int n_tensors,
                       float* dev_scale, int* dev_growth_tracker, float growth_factor, float backoff_factor,
                       int growth_interval, float max_grad_norm, double lr, double beta1, double beta2, double eps,
                       double weight_decay, float* dev_scratch, void* stream);

/* ---- "next" row 4 (SURVEY.md section 8f): D-side elementwise work -----------------------------------------------
 * DiffAugment (training/diffaugment.py:6-60, policy color -> translation -> cutout, any of the three left out) as one
 * pass over the images -- two launches with 'color' (contrast needs the per-image mean first), one without.  The
 * random draws are the CALLER's: the same torch.rand / torch.randint calls as the reference, in the same order, so the
 * parameters and the RNG stream are bit-identical; NULL pointers / zero cut sizes switch a stage off.
 *   dev_rb/rs/rc : rand(B) in the image dtype (:8, :15, :22);  dev_tx/ty : randint(-shift, shift+1, (B,)) int64 (:28-29)
 *   dev_ox/oy    : randint(0, H + (1 - cut_h % 2), (B,)) / same for W, int64 (:46-47);  cut_h/cut_w : int(H*ratio+.5) (:45)
 *   backward = 0 : dev_out = augment(dev_in);   backward = 1 : dev_out = d loss / d input given dev_in = d loss / d output
 *                  (the op is affine in the image, so the backward needs the parameters only)
 *   dev_scratch  : pnce_diffaug_scratch_floats(B, H, W) floats (needed with 'color')                              */
size_t pnce_diffaug_scratch_floats(int B, int H, int W);
int pnce_diffaug(const void* dev_in, void* dev_out, int dtype, int B, int C, int H, int W, const void* dev_rb,
                 const void* dev_rs, const void* dev_rc, const long long* dev_tx, const long long* dev_ty,
                 const long long* dev_ox, const long long* dev_oy, int cut_h, int cut_w, float* dev_scratch,
                 int backward, void* stream);
/* Hinge losses over the list of discriminator outputs (losses/adv_hinge.py:6-62), one launch per direction.
 *   mode 0: discriminator_hinge_loss(real_preds, fake_preds) (:6-32);  mode 1: generator_hinge_loss(fake_preds) (:35-62)
 * real / fake / dreal / dfake are HOST arrays of `scales` device pointers (dreal / dfake entries may be NULL);
 * numel[s] = elements of scale s; the loss leaves as one fp32 device scalar.                                      */
int pnce_hinge_fwd(const void* const* real, const void* const* fake, const long long* numel, int scales, int mode,
                   int dtype, float* dev_loss, void* stream);
int pnce_hinge_bwd(const void* const* real, const void* const* fake, void* const* dreal, void* const* dfake,
                   const long long* numel, int scales, int mode, int dtype, const float* dev_grad_out, void* stream);

/* ---- compressible device memory for the dense gradients (B200 L2 / HBM compute-data compression) ---------------
 * d tgt_feat (row a11: the `zeros` + `index_put_` autograd materialises, patchnce_cut.py:66-74 backward) is a zero fill
 * with a sampled float in a few per cent of its lines; in memory created with CU_MEM_ALLOCATION_COMP_GENERIC the dense
 * kernels write it ~12 % faster and the generator's backward reads it ~40 % faster.  pnce_comp_alloc / pnce_comp_free
 * have the signature torch.cuda.memory.CUDAPluggableAllocator binds (alloc(size, device, stream) -> ptr or NULL;
 * free(ptr, size, device, stream)); a caller without torch maps them onto its own allocator hooks.  Memory comes from
 * cuMemCreate / cuMemMap (plain VMM memory when the device refuses compression); every pointer handed out must come
 * back through pnce_comp_free.                                                                                      */
int   pnce_comp_supported(int device);
void* pnce_comp_alloc(ptrdiff_t size, int device, void* stream);
void  pnce_comp_free(void* ptr, ptrdiff_t size, int device, void* stream);
int   pnce_comp_is_compressed(const void* ptr);

/* Library self-test of the tcgen05 building blocks (bulk copy -> smem, tcgen05.mma with a K-major
 * or MN-major B operand, commit, tcgen05.ld): D(128 x n) = A(128 x k) * B on pre-tiled bf16 operand
 * blobs with host-supplied descriptor strides.  *dev_err is set to 1 on a protocol timeout.       */
int pnce_selftest_umma(const void* dev_a_blob, size_t a_bytes, const void* dev_b_blob, size_t b_bytes,
                       unsigned a_lbo, unsigned a_sbo, unsigned a_kstep, unsigned b_lbo, unsigned b_sbo,
                       unsigned b_kstep, int n, int k, int b_mn_major, float* dev_d_out, int* dev_err,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PNCE_H_ */
