// Internal launch interface between capi.cu and the kernel translation units.
#pragma once
#include "common.cuh"

namespace cmt {

struct GemmArgs {
    const void* A;
    const void* B;
    const float* bias;
    void* C;
    int M, N, K;
    long long lda, ldb, ldc, cb, cb_stride;
    long long strideA, strideB, strideC;
    float alpha;
    int relu, bias_per_row;
    int out_16;        // 16-bit output: bf16, or fp16 with f16 (else fp32)
    int f16;           // tensor-core path: fp16 operands and 16-bit outputs instead of bf16
    // 16-bit tensor-core path only: element (m, n) of batch z is stored at z*strideC + (n / cb)*cb_stride + (n % cb)*ldc + m
    // (C^T inside each column block, see cmt_gemm_bias_act)
    int transpose_c;
    // 16-bit tensor-core path only: [batch][N/32] atomicMax of the squared norm of every row's 32-column block (attention
    // score bound), or nullptr
    float* norm2_max;
    // ---- tensor-core path only: segmented K (n_seg == 0: ordinary GEMM) ----
    // K = n_seg * seg_k columns of B; segment s multiplies B[:, s*seg_k : (s+1)*seg_k] with the A columns
    // [seg_acol[s], seg_acol[s] + seg_k) read at row (m + a_row_off + seg_shift[s]) of the batch's A matrix, which has
    // a_rows rows and a_cols columns (rows outside [0, a_rows) are zero-filled by the TMA unit).
    int n_seg, seg_k, a_row_off, a_cols;
    long long a_rows;
    int seg_acol[18], seg_shift[18];
    int b_batch_div;   // batch z uses B of batch z / b_batch_div (0 or 1: z)
    // ---- token epilogue of the 3x3 shared_conv (conv_xv != nullptr) ----
    // Output row m is position (y, x) = (m / conv_Wp, m % conv_Wp) of the zero-padded map of frame z; interior positions
    // become token t = (y - 1) * conv_W + (x - 1) and are stored as xv[z][t - tok_begin] = lp(v),
    // xk[z][t - tok_begin] = lp(v + pos[t]) (v = ReLU(acc + bias), lp = rounding to the operand dtype); border rows are dropped.
    void* conv_xk;
    void* conv_xv;
    const float* conv_pos;
    int conv_W, conv_H, conv_Wp, conv_tok_begin, conv_tok_end;
    long long conv_frame_stride;   // elements between frames in xk / xv
};

struct AttnArgs {
    const void* q;
    const void* k;
    const void* vt;
    void* o;
    float* lse;
    int B, H, Nq, N_kv, kv_begin, kv_end;
    long long q_ld, k_bstride, k_hstride, v_bstride, v_hstride, v_ld;
    int f16;                         // tensor-core path: fp16 q / k / vt instead of bf16
    int o_dtype;                     // CMT_F32 | CMT_BF16 | CMT_F16
    const unsigned char* key_keep;   // [B, N_kv] 1 = attend, 0 = padded key (attention.py:76-90), or nullptr
    const float* q_norm2;            // [B*H] max |q|^2 per (frame, head), or nullptr (online softmax)
    const float* k_norm2;            // max |k|^2 per (frame, head) at [b * kn_bstride + h]
    long long kn_bstride;
};

// pe_kernels.cu
int launch_ray_pe(const float* img2lidar, void* out, int n_cam, int H, int W, int D, float pad_h,
                  float pad_w, const float* pc, int out_dtype, cudaStream_t stream);
int launch_ray_query_pe(const float* ref, const float* l2i, const float* i2l, void* out,
                        float* mask, int B, int V, int Nq, int D, float pad_h, float pad_w,
                        const float* pc, int out_dtype, cudaStream_t stream);
int launch_masked_view_sum(const void* emb, const float* mask, const float* base, long long base_bstride, float* out, int B,
                           int V, int Nq, int C, int emb_dtype, const uint8_t* view_valid, cudaStream_t stream);
int launch_pos2embed(const float* pos, void* out, int N, int pos_stride, int F, int out_dtype,
                     cudaStream_t stream);
// gather_kernels.cu
int launch_gather_tokens(const void* x_bev, const void* x_img, const float* bev_pos,
                         const float* rv_pos, void* xk, void* xv, int B, int C, int n_bev, int V,
                         int n_img, int tok_begin, int tok_end, int rv_tok0, int rv_rows, int feat_dtype, int out_dtype,
                         const uint8_t* sensor_valid, cudaStream_t stream);
int launch_nchw_to_padded_nhwc(const void* x, void* out, int B, int C, int H, int W, int guard, int in_dtype,
                               int out_dtype, const uint8_t* frame_valid, cudaStream_t stream);
int launch_sensor_key_keep(const uint8_t* sensor_valid, uint8_t* keep, int B, int n_bev, int V, int n_img,
                           cudaStream_t stream);
int launch_coop_max(const float* a, const float* b, float* out, long long n, cudaStream_t stream);
int launch_lse_merge(const float* o_parts, const float* lse_parts, void* o, float* lse, int G,
                     int B, int H, int Nq, long long o_gstride, long long lse_gstride, int o_dtype, cudaStream_t stream);
int launch_lse_merge_peer(const void* const* records, void* const* ctx, void* const* arrive, void* state, int rank, int G,
                          int B, int H, int Nq, int o_dtype, int scatter, cudaStream_t stream);
// norm_kernels.cu
int launch_add_layernorm(const float* x, const float* r, const float* gamma, const float* beta, float eps, int M, int C,
                         float* y, const float* gamma2, const float* beta2, float* y2, const float* add, void* ylp,
                         void* yadd, int lp_dtype, int flags, cudaStream_t stream);
int launch_task_head_tail(const float* h, const float* gamma, const float* beta, const float* w2, const float* b2, float* out,
                          int L, int M, int NH, int HC, int CMAX, float eps, int ksize, int Nq, const float* ref_logit,
                          const int* dec_comp, const float* dec_scale, const float* dec_offset, const long long* head_off_host,
                          const int* head_cout_host, cudaStream_t stream);
int launch_split3(const float* a, const float* b, void* out, float* merged, long long Z, int Nq, int C, int frames,
                  long long layer_stride_rows, const uint8_t* node_valid, cudaStream_t stream);
// decode_kernels.cu
int launch_bbox_topk_decode(const float* const* task_ptrs, const int* task_classes, int T, int B, int Nq, int num_classes,
                            int max_num, const float* post_center_range, float score_threshold, int use_score_threshold,
                            int bottom_center, float* boxes, float* scores, long long* labels, int* count,
                            long long* topk_index, const uint8_t* node_valid, int n_nodes, cudaStream_t stream);
// simt_kernels.cu
int launch_simt_gemm(const GemmArgs& g, int batch, int in_dtype, cudaStream_t stream);
int launch_simt_attn(const AttnArgs& a, int dtype, cudaStream_t stream);
// gemm_tcgen05.cu
int launch_tc_gemm(const GemmArgs& g, int batch, cudaStream_t stream);
// attn_tcgen05.cu
int tc_attn_set_timing_buffer(long long* dev_buf);
size_t tc_attn_workspace_bytes(int B, int H, int Nq, int n_kv_tokens);
int launch_tc_attn(const AttnArgs& a, void* workspace, size_t workspace_bytes, cudaStream_t stream);

}  // namespace cmt
