/* libcmtcoop_b200 -- C ABI of the B200-native CMT / CMTCoop token-fusion hot path.
 *
 * Every entry point replaces one piece of the reference's Python/PyTorch path
 * (suren3141/CMT-Cooperative-Perception, paths below are relative to
 * projects/mmdet3d_plugin/).  Conventions:
 *   - the caller (PyTorch) owns every buffer, workspace included; the library never
 *     allocates, frees or synchronises device memory;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = ok, negative = error (cmt_last_error_string() explains);
 *     no exception crosses this boundary;
 *   - sm_100a only: on any other device every launch entry returns CMT_ERR_ARCH.
 *     There is no CPU or generic-CUDA fallback.
 *   - dtype codes: CMT_F32 / CMT_BF16 / CMT_F16.  Three compute precisions: bf16 and fp16 run the tensor-core
 *     kernels (same rate; fp16 has 3 more mantissa bits, bf16 the fp32 exponent range), fp32 the CUDA-core
 *     verification kernels.
 */
#ifndef CMTCOOP_B200_H_
#define CMTCOOP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CMT_OK 0
#define CMT_ERR_BAD_ARG (-1)
#define CMT_ERR_CUDA (-2)
#define CMT_ERR_ARCH (-3)
#define CMT_ERR_WORKSPACE (-4)

#define CMT_F32 0
#define CMT_BF16 1
#define CMT_F16 2       /* fp16: a compute dtype of every entry below that takes one (never of the task-head chain:
                           cmt_split3_bf16 / cmt_gemm_segmented / cmt_task_head_tail), and a feature-map dtype */
#define CMT_BF16_SIMT 3 /* cmt_cross_attn_fwd only: bf16 operands through the fp32 CUDA-core kernel (comparator) */

/* flags of cmt_gemm_bias_act */
#define CMT_GEMM_RELU 1          /* out = max(out, 0)                                  */
#define CMT_GEMM_BIAS_PER_ROW 2  /* bias indexed by output row (default: by column)    */
#define CMT_GEMM_FORCE_SIMT 4    /* fp32 CUDA-core kernel even for bf16 operands (not fp16) */
#define CMT_GEMM_TRANSPOSE_OUT 8 /* store C^T inside each column block (16-bit tensor-core path only) */

/* flags of cmt_add_layernorm */
#define CMT_LN_X_ROW_BROADCAST 1 /* x is ONE row [C] shared by all M rows (decoder layer 0: see cmt_add_layernorm) */

int cmt_version(void);
const char* cmt_last_error_string(void);
/* 0 when device `dev` is sm_100 (B200), CMT_ERR_ARCH otherwise. */
int cmt_check_device(int dev);

/* ---- K1: camera-ray 3D position-encoding lift --------------------------------------
 * Replaces the eager meshgrid/einsum/normalise block of CmtHead._rv_pe
 * (models/dense_heads/cmt_head.py:417-432, same code cmt_head_coop.py:283-298).
 * img2lidar: [n_cam,4,4] fp32 row-major = float32(inv_float64(lidar2img)) (cmt_head.py:428-429).
 * out:       [n_cam,H,W,D*3] (feature index 3*k+c, cmt_head.py:433), fp32, bf16 or fp16.
 * pc_range:  6 host floats.  Token index inside a frame is cam*H*W + i*W + j. */
int cmt_ray_pe(const float* img2lidar, void* out, int n_cam, int H, int W, int D, float pad_h,
               float pad_w, const float* pc_range_host, int out_dtype, void* stream);

/* ---- K1b: reference-point re-projection for the query embedding ---------------------
 * Replaces CmtHead._rv_query_embed up to the rv_embedding MLP (cmt_head.py:439-464).
 * ref:       [B,Nq,3] fp32 in [0,1] (already inverse_sigmoid(...).sigmoid()'ed, :470)
 * lidar2img: [B,V,4,4] fp32, img2lidar: [B,V,4,4] fp32
 * out:       [B,V,Nq,D*3] (fp32|bf16|fp16), mask: [B,V,Nq] fp32 (1.0 inside image & z>0).
 *            Where mask is 0 the features are written as 0: the view sum ignores them, and their true values
 *            overflow fp16 for points near the camera plane. */
int cmt_ray_query_pe(const float* ref, const float* lidar2img, const float* img2lidar, void* out,
                     float* mask, int B, int V, int Nq, int D, float pad_h, float pad_w,
                     const float* pc_range_host, int out_dtype, void* stream);

/* out[b,n,:] = base[b,n,:] + sum_v mask[b,v,n] * emb[b,v,n,:]  (cmt_head.py:466 and the `bev + rv` of :492).
 * emb fp32|bf16|fp16, out fp32; base (nullable) fp32 at base + b*base_bstride + n*C (base_bstride = 0: one [Nq,C]
 * embedding shared by every frame -- in eval the BEV query embedding depends on the weights only).
 * view_valid (nullable DEVICE array, since version 103): uint8 [V, B], entry [v][b] != 0 when camera v delivered frame b.
 * An absent view is left out of the sum (its emb and mask are not read, so NaN there changes nothing); the present
 * views are summed in the same order as without the mask.  NULL: every view is present. */
int cmt_masked_view_sum(const void* emb, const float* mask, const float* base, int64_t base_bstride, float* out,
                        int B, int V, int Nq, int C, int emb_dtype, void* stream, const uint8_t* view_valid);

/* ---- sine/cosine BEV embedding ------------------------------------------------------
 * pos2embed (cmt_head.py:40-50) including its `dim_t = 2*(i//2)/F + 1` divisor.
 * pos: [N,pos_stride] fp32 (only columns 0 (x) and 1 (y) are read); out: [N,2F] = cat(emb(y), emb(x)),
 * fp32|bf16|fp16. */
int cmt_pos2embed(const float* pos, void* out, int N, int pos_stride, int F, int out_dtype,
                  void* stream);

/* ---- K4: token gather / transpose / concat / pos-add / cast -------------------------
 * Replaces the rearrange + cat + repeat of CmtTransformer.forward
 * (models/utils/cmt_transformer.py:105-110) fused with `key = key + key_pos`
 * (models/utils/petr_transformer.py:296-299).
 * x_bev:   [B,C,n_bev] NCHW-flattened, or NULL (n_bev = 0: no BEV tokens; n_bev > 0: rows [0,n_bev) of xk / xv are
 *          produced by cmt_shared_conv_tokens and only the image tokens are gathered, at row offset n_bev)
 * x_img:   [B*V,C,n_img] or NULL (V = 0)
 *          both in feat_dtype = CMT_F32 | CMT_BF16 | CMT_F16 (what the neck / backbone hands over; every feature
 *          is rounded to out_dtype on arrival, so 16-bit features change no bit of the bf16 path)
 * bev_pos: [n_bev,C] fp32 (batch-invariant), rv_pos: [B*V*n_img,C] fp32
 * xk = mem + pos, xv = mem, token-major, order BEV tokens then image tokens view-major,
 * N_kv = n_bev + V*n_img.  Only tokens [tok_begin, tok_end) are produced: xk, xv are
 * [B, tok_end - tok_begin, C] (0, N_kv = everything; a sub-range = this rank's share of a KV-token
 * split).  rv_rows > 0: rv_pos holds only rows [rv_tok0, rv_tok0 + rv_rows) of every frame's V*n_img image tokens,
 * [B, rv_rows, C] (the rank computed the rv-PE MLP for its own tokens only); rv_rows = 0: all of them.
 * out dtype fp32|bf16|fp16.
 * sensor_valid (nullable DEVICE array, since version 103): uint8 [S, B], one row per sensor in token order -- row 0 the
 * BEV map when n_bev > 0, then the V cameras -- entry [s][b] != 0 when sensor s delivered frame b.  Every token of an
 * absent (sensor, frame) is written as a zero row of xk and of xv; its features and position encoding are not read
 * (they may hold anything, NaN included).  NULL: every sensor is present. */
int cmt_gather_tokens(const void* x_bev, const void* x_img, const float* bev_pos,
                      const float* rv_pos, void* xk, void* xv, int B, int C, int n_bev, int V,
                      int n_img, int tok_begin, int tok_end, int rv_tok0, int rv_rows, int feat_dtype, int out_dtype,
                      void* stream, const uint8_t* sensor_valid);

/* Key-keep bytes of cmt_cross_attn_fwd from the sensor mask of cmt_gather_tokens (since version 103):
 * key_keep [B, n_bev + V*n_img] uint8 (DEVICE), entry [b][t] = 1 when the sensor of token t delivered frame b, else 0
 * (sensor_valid [S, B] as there, S = (n_bev > 0) + V). */
int cmt_sensor_key_keep(const uint8_t* sensor_valid, uint8_t* key_keep, int B, int n_bev, int V, int n_img, void* stream);

/* ---- K2: projection / MLP GEMM ------------------------------------------------------
 * C = act((A * B^T + bias) * alpha); A:[M,K] (lda), B:[N,K] (ldb), both row-major, K contiguous.
 * Replaces F.linear in _in_projection_packed / out_proj (models/utils/attention.py:21-27,138)
 * and the nn.Linear+ReLU pairs of rv_embedding / bev_embedding (cmt_head.py:292-301).
 * Batched: `batch` problems, element strides strideA/strideB (0 = shared operand)/strideC.
 * Output addressing ("column blocks"): element (m,n) of batch z is stored at
 *     C + z*strideC + (n / cb)*cb_stride + m*ldc + (n % cb)
 * cb >= N gives a plain row-major matrix; cb = 32 with ldc = 32 gives the per-head
 * [.., H, tokens, 32] layout the attention kernel reads.  With CMT_GEMM_TRANSPOSE_OUT the block is
 * written transposed,
 *     C + z*strideC + (n / cb)*cb_stride + (n % cb)*ldc + m
 * which with cb = 32, ldc = ld gives the token-contiguous V^T layout [.., H, 32, ld] (16-bit operands and
 * output, cb % 32 == 0, N % 32 == 0, N <= 1984).
 * norm2_max (16-bit path, or NULL): [batch][N/32] fp32, zero-initialised by the caller; the epilogue raises
 * entry (z, n/32) to the largest squared norm of a row's 32-column block (one attention head of one
 * query/key).  cmt_cross_attn_fwd turns the two maxima into a bound on every score (see there).
 * in_dtype bf16 or fp16 -> TMA + tcgen05 kernel (fp32 accumulate in TMEM); in_dtype fp32 -> fp32
 * CUDA-core kernel (verification mode).  out_dtype: fp32 or the 16-bit dtype of the operands (fp32 operands: fp32 or
 * bf16).  Requirements for 16-bit operands: K % 8 == 0, lda/ldb % 8 == 0, 16-byte aligned bases, and
 * (cb >= N or cb % 32 == 0). */
int cmt_gemm_bias_act(const void* A, const void* B, const float* bias, void* C, int M, int N,
                      int K, int64_t lda, int64_t ldb, int64_t ldc, int64_t cb, int64_t cb_stride,
                      int batch, int64_t strideA, int64_t strideB, int64_t strideC, float alpha,
                      int flags, int in_dtype, int out_dtype, float* norm2_max, void* stream);

/* Segmented-K form of cmt_gemm_bias_act (bf16 operands, tensor-core path, plain row-major output):
 *     C[z][m][n] = act((sum_s sum_k A_z[m + a_row_off + row_shift[s]][acol[s] + k] * B_zb[n][s*seg_k + k] + bias[n]) * alpha)
 * for s < n_seg <= 18, k < seg_k (a multiple of 64), zb = z / b_batch_div.  A_z is the [a_rows, a_cols] matrix at
 * A + z*strideA (row stride lda); rows outside [0, a_rows) read as zero.  One mechanism, two uses: implicit convolutions
 * (a filter tap = a row shift of a channel-last operand: the k = 3 task-head convolutions over the query axis,
 * cmt_head.py:116-150, and the 3x3 shared_conv below) and split-precision products (A = [hi | mid | lo] bf16 terms of an
 * fp32 operand, segments pairing them with the matching terms of the weights: fp32-grade task-head logits on the tensor
 * cores).  seg_acol / seg_row_shift are HOST arrays of n_seg ints. */
int cmt_gemm_segmented(const void* A, const void* B, const float* bias, void* C, int M, int N, int n_seg, int seg_k,
                       const int* seg_acol_host, const int* seg_row_shift_host, int a_row_off, int64_t a_rows,
                       int a_cols, int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA, int64_t strideB,
                       int b_batch_div, int64_t strideC, float alpha, int flags, int out_dtype, void* stream);

/* ---- shared_conv: 3x3 conv 512->256 + BatchNorm(eval) + ReLU as an implicit GEMM writing BEV tokens ----------------
 * Replaces ConvModule(conv3x3 no bias, BN2d, ReLU) of CmtHead (models/dense_heads/cmt_head.py:280-287, applied :481,
 * coop: cmt_head_coop.py:343) TOGETHER with the BEV half of the token rearrange / pos add
 * (models/utils/cmt_transformer.py:105-110, petr_transformer.py:296-299): the NCHW fp32 map never exists.
 * dtype (out_dtype / dtype, the trailing argument of both entries): CMT_BF16 or CMT_F16, the operand and token dtype.
 * Step 1, cmt_nchw_to_padded_nhwc: x [B,C,H,W] (fp32|bf16|fp16) -> out (dtype) [B][2*guard_rows + (H+2)*(W+2)][C], pixel
 *   (y,x) in row guard_rows + (y+1)*(W+2) + (x+1); only interior rows are written (the caller zero-fills `out` once),
 *   guard_rows >= W + 3.
 * Step 2, cmt_shared_conv_tokens: w (dtype) [Cout][9*Cin], tap-major (w[o][(ky*3+kx)*Cin + c] = conv.weight[o][c][ky][kx] *
 *   bn_scale[o]), bias fp32 [Cout] = bn.bias - bn.running_mean * bn_scale, bev_pos fp32 [H*W, Cout];
 *   for every frame b and token t = y*W + x in [tok_begin, tok_end):
 *     v = ReLU(conv(x)[b,:,y,x] + bias);  xv[b][t - tok_begin][:] = dtype(v);  xk[b][t - tok_begin][:] = dtype(v + bev_pos[t])
 *   with out_frame_stride elements between frames (N_kv * Cout: the image tokens follow, cmt_gather_tokens with
 *   x_bev = NULL).  Cin % 64 == 0, Cout % 32 == 0, Cout <= 1984.
 * frame_valid (cmt_nchw_to_padded_nhwc, nullable DEVICE array, since version 103): uint8 [B]; the interior rows of a
 *   frame b with frame_valid[b] == 0 are written as zeros and its input is not read, so step 2 produces finite rows
 *   ReLU(bias) (+ bev_pos) for it.  NULL: every frame is present. */
int cmt_nchw_to_padded_nhwc(const void* x, void* out, int B, int C, int H, int W, int guard_rows, int in_dtype,
                            void* stream, int out_dtype, const uint8_t* frame_valid);
int cmt_shared_conv_tokens(const void* xp, const void* w, const float* bias, const float* bev_pos, void* xk, void* xv,
                           int B, int Cin, int Cout, int H, int W, int guard_rows, int64_t out_frame_stride,
                           int tok_begin, int tok_end, void* stream, int dtype);

/* ---- K3: flash cross-attention ------------------------------------------------------
 * Replaces flash_attn_unpadded_kvpacked_func as called by FlashAttention.forward
 * (models/utils/attention.py:46-92; softmax(Q K^T / sqrt(d)) V, non-causal, no dropout).
 * q:   [B,Nq,H*32] row-major (row stride q_ld), ALREADY multiplied by log2(e)/sqrt(32)
 * k:   per (b,h) a [N_kv,32] matrix (row stride 32) at k + b*k_bstride + h*k_hstride
 * vt:  per (b,h) a [32,N_kv] matrix (row stride v_ld) at vt + b*v_bstride + h*v_hstride
 * Only tokens [kv_begin,kv_end) are attended (multi-GPU / split-KV partials).
 * o:   [B,Nq,H*32] (o_dtype, row stride H*32), normalised over the attended tokens
 * key_keep: [B,N_kv] bytes, 1 = attend, 0 = padded key, or NULL.  This is the key_padding_mask branch of
 *      FlashAttention.forward (attention.py:76-90: unpad_input + cu_seqlens_k); dropping a key from the packed
 *      sequence and giving it weight zero are the same softmax.  A query with no attended key gets o = 0.
 * q_norm2_max [B*H], k_norm2_max (entry (b,h) at b*kn_bstride + h), both or neither NULL: upper bounds of
 *      |q|^2 and |k|^2 per (frame, head) as written by cmt_gemm_bias_act(norm2_max).  |q.k| <= |q||k| bounds
 *      every score of the (frame, head); when that bound is <= 60 (bf16) or <= 14 (fp16; log2 units) the
 *      tensor-core kernel uses it as a fixed softmax shift and skips the running row maximum and the accumulator
 *      rescale (same result: the softmax is shift-invariant, and all weights stay normal numbers of the dtype);
 *      larger bounds and NULL use the online softmax.
 * lse: [B,H,Nq] fp32 natural-log sum-exp of the scaled scores over the attended tokens, or NULL
 * dtype bf16 or fp16 (q, k, vt and the softmax weights P) -> tcgen05 kernel, work split over all SMs along the KV
 * axis with partials in `workspace` (cmt_cross_attn_workspace_bytes) merged by a second kernel; dtype fp32 -> fp32
 * CUDA-core kernel.  o_dtype: fp32 or the operand dtype (fp16 only with fp16 operands).  Head dim is fixed at 32
 * (256/8, the only value the reference configs use). */
size_t cmt_cross_attn_workspace_bytes(int B, int H, int Nq, int n_kv_tokens);
int cmt_cross_attn_fwd(const void* q, const void* k, const void* vt, void* o, float* lse, int B,
                       int H, int Nq, int N_kv, int kv_begin, int kv_end, int64_t q_ld,
                       int64_t k_bstride, int64_t k_hstride, int64_t v_bstride, int64_t v_hstride,
                       int64_t v_ld, const unsigned char* key_keep, const float* q_norm2_max,
                       const float* k_norm2_max, int64_t kn_bstride, int dtype, int o_dtype,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Log-sum-exp merge of G partial attention results (KV-token split across GPUs or streams):
 * part g: o [B,Nq,H*32] fp32 at o_parts + g*o_gstride, lse [B,H,Nq] fp32 (natural log) at lse_parts + g*lse_gstride
 * (strides in elements; 0 = densely stacked [G,...] arrays) -> o [B,Nq,H*32] (o_dtype fp32|bf16|fp16), lse (nullable).  With
 * o_gstride = lse_gstride = B*Nq*H*32 + B*H*Nq and lse_parts = o_parts + B*Nq*H*32 the parts are the packed
 * (O | LSE) records of ONE all-gather per decoder layer. */
int cmt_lse_merge(const float* o_parts, const float* lse_parts, void* o, float* lse, int G, int B,
                  int H, int Nq, int64_t o_gstride, int64_t lse_gstride, int o_dtype, void* stream);

/* The same merge fused with its exchange over peer memory (NVLink / NVSwitch), replacing the NCCL all-gather of the
 * KV-token split.  records[g] / ctx[g] / arrive[g] are HOST arrays of G <= 8 device pointers, all into memory mapped
 * into every rank of the group (the caller maps it, e.g. torch symmetric memory): rank g's packed (O | LSE) record of
 * this exchange -- o [B,Nq,H*32] fp32 followed by lse [B,H,Nq] fp32 --, rank g's context buffer [B,Nq,H*32] (o_dtype)
 * (fp32|bf16|fp16) and rank g's block of 16 uint32 counters; `state` points at two uint32 {exchange number, finished blocks} in LOCAL
 * memory; counters and state are zero before the first exchange.  The kernel announces the local record to all ranks,
 * waits for theirs, merges this rank's 1/G of the rows straight from the G records (remote ones read through NVLink),
 * stores them into EVERY rank's context buffer, and returns once all ranks' rows have landed in ctx[rank]
 * (scatter = 1: NVLink carries (G-1)/G of a record in and of a context out per rank; two handshakes).  scatter = 0: every
 * rank merges ALL rows from the G records into ctx[rank] only (G - 1 records in, one handshake); scatter < 0 picks by
 * group size (0 for G <= 2).  Every rank must pass the same mode.
 * Collective: every rank of the group calls it once per exchange, in the same order; two consecutive exchanges must
 * use different record buffers; a context buffer may be reused by the next exchange once its local reader is ahead of
 * this call in the stream.  A rank that does not arrive within ~30 s traps. */
int cmt_lse_merge_peer(const void* const* records, void* const* ctx, void* const* arrive, void* state, int rank, int G,
                       int B, int H, int Nq, int o_dtype, int scatter, void* stream);

/* ---- decoder small ops: fused residual add + LayerNorm --------------------------------
 * One launch for `query = norm(identity + attn_out)` of mmcv BaseTransformerLayer (post-norm order
 * self_attn, norm, cross_attn, norm, ffn, norm) plus PETRTransformerDecoder's shared post_norm
 * (models/utils/petr_transformer.py:363-371) and the casts / `query + query_pos` (:294-295) the
 * next projection needs.  x, r (nullable), add (nullable): [M,C] fp32; C must be 256.
 *   y    = LN(x + r; gamma, beta, eps)            fp32, required
 *   y2   = LN(y; gamma2, beta2, eps)              fp32, optional (NULL)
 *   ylp  = cast(y), yadd = cast(y + add)          lp_dtype (fp32|bf16|fp16), each optional (NULL)
 * flags & CMT_LN_X_ROW_BROADCAST: x is a single row [C] used for every output row.  Decoder layer 0 runs on the zero
 * target (cmt_transformer.py:114), so its self-attention attends over values that are all equal to the value bias and
 * returns out_proj(b_v) for every query whatever the weights of the softmax: that one row is the whole `x + attn_out`. */
int cmt_add_layernorm(const float* x, const float* r, const float* gamma, const float* beta, float eps,
                      int M, int C, float* y, const float* gamma2, const float* beta2, float* y2,
                      const float* add, void* ylp, void* yadd, int lp_dtype, int flags, void* stream);

/* ---- task heads -------------------------------------------------------------------------
 * SeparateTaskHead (models/dense_heads/cmt_head.py:97-203 with GroupLayerNorm1d :53-94) for all output heads at once,
 * final_kernel k = 1 (fusion / camera configs) or 3 (LiDAR configs: the convolutions run over the QUERY axis), fp32-grade
 * arithmetic throughout (these logits feed the top-k, multi_task_bbox_coder.py:61-64).  Three launches:
 *
 * 1. cmt_split3_bf16: a (and optionally b) [Z, Nq, 256] fp32 -> out bf16 [Z, Nq + 2, 768] = [x1 | x2 | x3] per row with
 *    x = nan_to_num(a) (cmt_head.py:499), or max(nan_to_num(a), nan_to_num(b)) for the cooperative heads
 *    (cmt_head_coop.py:358,383-389), x1 = bf16(x), x2 = bf16(x - x1), x3 = bf16(x - x1 - x2); rows 0 and Nq + 1 of every
 *    z are zero (convolution padding).  Z = decoder layers * frames.  `merged` (nullable): fp32 copy of x, [Z, Nq, 256].
 *    frames > 0: the inputs are strided -- row q of z = (layer, frame) sits at row layer*layer_stride_rows + frame*Nq + q
 *    (both nodes' frames stacked in one decoder pass: a = the stack, b = a + frames*Nq*256, layer_stride_rows =
 *    2*frames*Nq); frames = 0: dense [Z, Nq, 256].
 *    node_valid (nullable DEVICE array, since version 102): uint8 [2, frames], entry [n][f] != 0 when node n (0: the node
 *    in `a`, 1: the node in `b`) delivered frame f.  Needs b and frames > 0 (for the dense layout pass frames = B and
 *    layer_stride_rows = B*Nq).  Frame f then takes max(nan_to_num(a), nan_to_num(b)) with both nodes, nan_to_num of the
 *    present node's rows with one, and zero rows with none; `merged` follows the same rule, and an absent node's rows
 *    are not read (they may hold anything).  NULL: every node is present.
 * 2. cmt_gemm_segmented with 6 segments per tap (x1w1, x1w2, x2w1, x1w3, x2w2, x3w1; the weights split the same way):
 *    the first grouped convolution as a tensor-core GEMM that reproduces the fp32 product to ~2^-22.
 * 3. cmt_task_head_tail: group-LN + ReLU + second convolution (+ optional reference-point decode):
 *   h:     [L, M, NH, HC] fp32   first-conv output, L = decoder layers (conv groups), M = frames*Nq rows,
 *                                NH = output heads (center, height, dim, rot, vel, cls_logits), HC = 64
 *   gamma, beta: [L, NH, HC]     GroupLayerNorm1d affine;  eps: its epsilon (1e-6)
 *   w2:    [L, NH, CMAX, ksize, HC], b2: [L, NH, CMAX]   second conv, zero-padded to CMAX <= 32 outputs per head
 *   out:   [L, M, NH, CMAX] fp32 = sum_t ReLU(LN(h[q + t - ksize/2]) * gamma + beta) . w2[:, t] + b2
 *          (rows outside a frame's [0, Nq) contribute zero: Conv1d zero padding of the hidden activations)
 *   ref_logit (nullable): [M, 3] fp32 inverse_sigmoid(reference points); with it, output (head, o) whose
 *          dec_comp[head*CMAX + o] = c >= 0 becomes sigmoid(out + ref_logit[row][c]) * dec_scale[..] + dec_offset[..]
 *          (cmt_head.py:501-513: center and height to metric coordinates); dec_* are DEVICE arrays of NH*CMAX entries.
 *   head_off_host / head_cout_host (nullable HOST arrays of NH entries, NH <= 8): instead of the padded layout, head i is
 *          written as its own contiguous [L, M, cout[i]] tensor starting at out + off[i] (elements). */
int cmt_split3_bf16(const float* a, const float* b, void* out, float* merged, int64_t Z, int Nq, int C, int frames,
                    int64_t layer_stride_rows, void* stream, const uint8_t* node_valid);
int cmt_task_head_tail(const float* h, const float* gamma, const float* beta, const float* w2,
                       const float* b2, float* out, int L, int M, int NH, int HC, int CMAX, float eps,
                       int ksize, int Nq, const float* ref_logit, const int* dec_comp, const float* dec_scale,
                       const float* dec_offset, const int64_t* head_off_host, const int* head_cout_host, void* stream);

/* ---- cooperative V2I merge ----------------------------------------------------------
 * out = max(nan_to_num(a), nan_to_num(b)) element-wise (cmt_head_coop.py:358,383-389). */
int cmt_coop_max(const float* a, const float* b, float* out, int64_t n, void* stream);

/* ---- box decode ------------------------------------------------------------------------
 * MultiTaskBBoxCoder.decode_single for every frame of a batch in one launch, with no host synchronisation (graph
 * capturable): replaces the per-frame sigmoid / top-k / gather / denormalize_bbox / mask loop of
 * MultiTaskBBoxCoder.decode (core/bbox/coders/multi_task_bbox_coder.py:46-141, core/bbox/util.py:37-68) and, with
 * bottom_center, the z shift of CmtHead.get_bboxes (models/dense_heads/cmt_head.py:912).
 *   task_ptrs_host: HOST array of 6*T device pointers, per task t < T <= CMT_BOX_DECODE_MAX_TASKS the last decoder
 *       layer's contiguous fp32 outputs {cls_logits [B,Nq,C_t], center [B,Nq,2], height [B,Nq,1], dim [B,Nq,3],
 *       rot [B,Nq,2], vel [B,Nq,2]};  task_classes_host: HOST array of the T class counts C_t.
 *   num_classes must equal sum C_t; the flat candidate index is q*num_classes + c, c running over the tasks' classes in
 *   concatenation order (torch.cat(cls_logits, -1)).  Per frame:
 *     score = 1 / (1 + expf(-logit)); the K = max_num largest scores in descending order, ties by ascending flat index
 *     (torch.sort(descending=True, stable=True)[:K]; NaN ranks above +inf);
 *     label = idx % num_classes, q = idx / num_classes; box = [cx, cy, cz, exp(w), exp(l), exp(h), atan2(rot0, rot1),
 *     vx, vy] from the task that owns the label; kept when post_center_range_host[0..2] <= (cx, cy, cz) <=
 *     post_center_range_host[3..5] and, if use_score_threshold, score > score_threshold;  bottom_center: z -= h * 0.5.
 *   Outputs (caller-owned, fixed shape): boxes [B,K,9] fp32, scores [B,K] fp32, labels [B,K] int64 -- the kept slots
 *     first, in score order, then zeros with label -1;  count [B] int32 kept slots;  topk_index [B,K] int64 every
 *     selected flat index before the mask.
 *   node_valid (nullable DEVICE array, since version 102): uint8 [n_nodes, B]; frame b is decoded when any entry
 *     [n][b] != 0.  Otherwise its head outputs are not read and the frame gets count 0, zero boxes and scores, and
 *     labels and topk_index -1 in every slot.  NULL: every frame is decoded (n_nodes is then ignored).
 *   Limits (CMT_ERR_BAD_ARG otherwise): 1 <= K <= min(CMT_BOX_DECODE_MAX_K, Nq*num_classes), and
 *     Nq*num_classes <= CMT_BOX_DECODE_MAX_CANDIDATES (one CTA per frame keeps every score in shared memory; nuScenes
 *     is 900 x 10 = 9000). */
#define CMT_BOX_DECODE_MAX_TASKS 8
#define CMT_BOX_DECODE_MAX_K 1024
#define CMT_BOX_DECODE_MAX_CANDIDATES 49152
int cmt_bbox_topk_decode(const float* const* task_ptrs_host, const int* task_classes_host, int T, int B, int Nq,
                         int num_classes, int max_num, const float* post_center_range_host, float score_threshold,
                         int use_score_threshold, int bottom_center, float* boxes, float* scores, int64_t* labels,
                         int32_t* count, int64_t* topk_index, void* stream, const uint8_t* node_valid, int n_nodes);

/* ---- diagnostics -----------------------------------------------------------------------
 * Cycle accounting of the tcgen05 attention kernel on the CURRENT device.  dev_buf: device buffer of
 * 3*96*16 + 148 int64 (or NULL to switch the hook off again).  While set, every CTA of every following
 * cmt_cross_attn_fwd(bf16) launch on that device stores its total clock64 count into the last 148 entries
 * (launch duration in SM cycles -> with an event time, the SM clock the kernel really ran at); a library built
 * with -DCMT_ATTN_TRACE also fills the per-step stamps of CTA 0 (tools/attn_trace.py).  Not for production
 * streams: the buffer pointer is process state, one slot per device. */
int cmt_debug_attn_timing(void* dev_buf_i64);

#ifdef __cplusplus
}
#endif
#endif /* CMTCOOP_B200_H_ */
