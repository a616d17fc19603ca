// extern "C" surface of libcmtcoop_b200 (see include/cmtcoop_b200.h for the contract of every
// entry point and the reference file:line each one replaces).
#include <cstdarg>
#include <cstdio>
#include <mutex>

#include "kernels.cuh"

namespace cmt {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("%s: CUDA error %d (%s)", what, static_cast<int>(e), cudaGetErrorString(e));
    return CMT_ERR_CUDA;
}

struct DevInfo {
    int sms = 0;
    int major = 0, minor = 0;
    bool ok = false;
};
static DevInfo g_dev[64];
static std::once_flag g_dev_once[64];

int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    return dev;
}

static const DevInfo& dev_info() {
    const int dev = current_device();
    std::call_once(g_dev_once[dev], [dev]() {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) {
            g_dev[dev].sms = prop.multiProcessorCount;
            g_dev[dev].major = prop.major;
            g_dev[dev].minor = prop.minor;
            g_dev[dev].ok = true;
        }
    });
    return g_dev[dev];
}

int device_sm_count() {
    const DevInfo& d = dev_info();
    return d.sms > 0 ? d.sms : 148;
}

int require_sm100() {
    const DevInfo& d = dev_info();
    if (!d.ok) {
        set_error("no CUDA device available (libcmtcoop_b200 has no CPU fallback)");
        return CMT_ERR_ARCH;
    }
    if (d.major != 10) {
        set_error("libcmtcoop_b200 requires an sm_100 (B200) device, found sm_%d%d; there is no fallback path",
                  d.major, d.minor);
        return CMT_ERR_ARCH;
    }
    return CMT_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::once_flag g_encode_once;

int encode_tma(CUtensorMap* map, const void* base, int dtype, int rank, const uint64_t* dims,
               const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes) {
    std::call_once(g_encode_once, []() {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    });
    if (!g_encode) {
        set_error("cuTensorMapEncodeTiled not available from the driver");
        return CMT_ERR_CUDA;
    }
    cuuint64_t gdims[5];
    cuuint64_t gstrides[4];
    cuuint32_t gbox[5];
    cuuint32_t estr[5];
    for (int i = 0; i < rank; ++i) {
        gdims[i] = dims[i];
        gbox[i] = box[i];
        estr[i] = 1;
        if (i < rank - 1) gstrides[i] = strides_bytes[i];
    }
    const CUtensorMapSwizzle sw = swizzle_bytes == 128  ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                  : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                        : CU_TENSOR_MAP_SWIZZLE_NONE;
    const CUtensorMapDataType dt = dtype == CMT_F32   ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                   : dtype == CMT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                      : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    CUresult r = g_encode(map, dt, static_cast<cuuint32_t>(rank),
                          const_cast<void*>(base), gdims, gstrides, gbox, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu %llu %llu, stride0 %llu)",
                  static_cast<int>(r), rank, (unsigned long long)dims[0], (unsigned long long)dims[1],
                  (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)strides_bytes[0]);
        return CMT_ERR_CUDA;
    }
    return CMT_OK;
}

}  // namespace cmt

using namespace cmt;

#define CMT_REQUIRE_DEVICE()            \
    do {                                \
        int rc__ = require_sm100();     \
        if (rc__ != CMT_OK) return rc__; \
    } while (0)

extern "C" {

int cmt_version(void) { return 103; }

const char* cmt_last_error_string(void) { return g_err; }

int cmt_check_device(int dev) {
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, dev);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cmt_check_device: no CUDA device %d (%s)", dev, cudaGetErrorString(e));
        return CMT_ERR_ARCH;
    }
    if (prop.major != 10) {
        set_error("cmt_check_device: device %d is sm_%d%d, sm_100 required", dev, prop.major, prop.minor);
        return CMT_ERR_ARCH;
    }
    return CMT_OK;
}

int cmt_ray_pe(const float* img2lidar, void* out, int n_cam, int H, int W, int D, float pad_h, float pad_w,
               const float* pc_range_host, int out_dtype, void* stream) {
    CMT_REQUIRE_DEVICE();
    return launch_ray_pe(img2lidar, out, n_cam, H, W, D, pad_h, pad_w, pc_range_host, out_dtype,
                         static_cast<cudaStream_t>(stream));
}

int cmt_ray_query_pe(const float* ref, const float* lidar2img, const float* img2lidar, void* out, float* mask,
                     int B, int V, int Nq, int D, float pad_h, float pad_w, const float* pc_range_host,
                     int out_dtype, void* stream) {
    CMT_REQUIRE_DEVICE();
    return launch_ray_query_pe(ref, lidar2img, img2lidar, out, mask, B, V, Nq, D, pad_h, pad_w, pc_range_host,
                               out_dtype, static_cast<cudaStream_t>(stream));
}

int cmt_masked_view_sum(const void* emb, const float* mask, const float* base, int64_t base_bstride, float* out, int B, int V,
                        int Nq, int C, int emb_dtype, void* stream, const uint8_t* view_valid) {
    CMT_REQUIRE_DEVICE();
    return launch_masked_view_sum(emb, mask, base, base_bstride, out, B, V, Nq, C, emb_dtype, view_valid,
                                  static_cast<cudaStream_t>(stream));
}

int cmt_pos2embed(const float* pos, void* out, int N, int pos_stride, int F, int out_dtype, void* stream) {
    CMT_REQUIRE_DEVICE();
    return launch_pos2embed(pos, out, N, pos_stride, F, out_dtype, static_cast<cudaStream_t>(stream));
}

int cmt_gather_tokens(const void* x_bev, const void* x_img, const float* bev_pos, const float* rv_pos,
                      void* xk, void* xv, int B, int C, int n_bev, int V, int n_img, int tok_begin, int tok_end,
                      int rv_tok0, int rv_rows, int feat_dtype, int out_dtype, void* stream, const uint8_t* sensor_valid) {
    CMT_REQUIRE_DEVICE();
    return launch_gather_tokens(x_bev, x_img, bev_pos, rv_pos, xk, xv, B, C, n_bev, V, n_img, tok_begin, tok_end,
                                rv_tok0, rv_rows, feat_dtype, out_dtype, sensor_valid, static_cast<cudaStream_t>(stream));
}

int cmt_sensor_key_keep(const uint8_t* sensor_valid, uint8_t* key_keep, int B, int n_bev, int V, int n_img, void* stream) {
    CMT_REQUIRE_DEVICE();
    return launch_sensor_key_keep(sensor_valid, key_keep, B, n_bev, V, n_img, static_cast<cudaStream_t>(stream));
}

int cmt_gemm_bias_act(const void* A, const void* B, const float* bias, void* C, int M, int N, int K,
                      int64_t lda, int64_t ldb, int64_t ldc, int64_t cb, int64_t cb_stride, int batch,
                      int64_t strideA, int64_t strideB, int64_t strideC, float alpha, int flags, int in_dtype,
                      int out_dtype, float* norm2_max, void* stream) {
    CMT_REQUIRE_DEVICE();
    CMT_CHECK_ARG(A && B && C, "cmt_gemm_bias_act: null pointer");
    CMT_CHECK_ARG(M > 0 && N > 0 && K > 0 && batch > 0, "cmt_gemm_bias_act: bad shape M=%d N=%d K=%d batch=%d", M,
                  N, K, batch);
    CMT_CHECK_ARG(lda >= K && ldb >= K && cb > 0, "cmt_gemm_bias_act: bad leading dimensions");
    CMT_CHECK_ARG(in_dtype == CMT_F32 || in_dtype == CMT_BF16 || in_dtype == CMT_F16, "cmt_gemm_bias_act: bad in_dtype");
    CMT_CHECK_ARG(out_dtype == CMT_F32 || out_dtype == CMT_BF16 || out_dtype == CMT_F16, "cmt_gemm_bias_act: bad out_dtype");
    CMT_CHECK_ARG(in_dtype == CMT_F16 ? out_dtype != CMT_BF16 : out_dtype != CMT_F16,
                  "cmt_gemm_bias_act: fp16 operands take an fp16 or fp32 output, and an fp16 output needs fp16 operands");
    CMT_CHECK_ARG(in_dtype != CMT_F16 || !(flags & CMT_GEMM_FORCE_SIMT), "cmt_gemm_bias_act: fp16 operands run on the tensor cores only");
    GemmArgs g{};
    g.A = A;
    g.B = B;
    g.bias = bias;
    g.C = C;
    g.M = M;
    g.N = N;
    g.K = K;
    g.lda = lda;
    g.ldb = ldb;
    g.ldc = ldc;
    g.cb = cb;
    g.cb_stride = cb_stride;
    g.strideA = strideA;
    g.strideB = strideB;
    g.strideC = strideC;
    g.alpha = alpha;
    g.relu = (flags & CMT_GEMM_RELU) ? 1 : 0;
    g.bias_per_row = (flags & CMT_GEMM_BIAS_PER_ROW) ? 1 : 0;
    g.out_16 = out_dtype != CMT_F32;
    g.f16 = in_dtype == CMT_F16;
    g.transpose_c = (flags & CMT_GEMM_TRANSPOSE_OUT) ? 1 : 0;
    g.norm2_max = norm2_max;
    const bool tc = in_dtype != CMT_F32 && !(flags & CMT_GEMM_FORCE_SIMT);
    CMT_CHECK_ARG(norm2_max == nullptr || tc, "cmt_gemm_bias_act: norm2_max is a 16-bit tensor-core path option");
    CMT_CHECK_ARG(!g.transpose_c || tc, "cmt_gemm_bias_act: CMT_GEMM_TRANSPOSE_OUT is a 16-bit tensor-core path option");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (tc) return launch_tc_gemm(g, batch, s);
    return launch_simt_gemm(g, batch, in_dtype, s);
}

int cmt_gemm_segmented(const void* A, const void* B, const float* bias, void* C, int M, int N, int n_seg, int seg_k,
                       const int* seg_acol_host, const int* seg_row_shift_host, int a_row_off, int64_t a_rows, int a_cols,
                       int64_t lda, int64_t ldb, int64_t ldc, int batch, int64_t strideA, int64_t strideB, int b_batch_div,
                       int64_t strideC, float alpha, int flags, int out_dtype, void* stream) {
    CMT_REQUIRE_DEVICE();
    CMT_CHECK_ARG(A && B && C && seg_acol_host && seg_row_shift_host, "cmt_gemm_segmented: null pointer");
    CMT_CHECK_ARG(M > 0 && N > 0 && batch > 0 && n_seg > 0 && n_seg <= 18 && seg_k > 0, "cmt_gemm_segmented: bad shape");
    CMT_CHECK_ARG(out_dtype == CMT_F32 || out_dtype == CMT_BF16, "cmt_gemm_segmented: bad out_dtype");
    CMT_CHECK_ARG(!(flags & (CMT_GEMM_FORCE_SIMT | CMT_GEMM_TRANSPOSE_OUT)), "cmt_gemm_segmented: tensor-core path, plain output only");
    GemmArgs g{};
    g.A = A;
    g.B = B;
    g.bias = bias;
    g.C = C;
    g.M = M;
    g.N = N;
    g.K = n_seg * seg_k;
    g.lda = lda;
    g.ldb = ldb;
    g.ldc = ldc;
    g.cb = N;
    g.cb_stride = 0;
    g.strideA = strideA;
    g.strideB = strideB;
    g.strideC = strideC;
    g.alpha = alpha;
    g.relu = (flags & CMT_GEMM_RELU) ? 1 : 0;
    g.bias_per_row = (flags & CMT_GEMM_BIAS_PER_ROW) ? 1 : 0;
    g.out_16 = out_dtype == CMT_BF16;
    g.n_seg = n_seg;
    g.seg_k = seg_k;
    g.a_row_off = a_row_off;
    g.a_rows = a_rows;
    g.a_cols = a_cols;
    g.b_batch_div = b_batch_div;
    for (int i = 0; i < n_seg; ++i) {
        CMT_CHECK_ARG(seg_acol_host[i] >= 0 && seg_acol_host[i] % 8 == 0 && seg_acol_host[i] + seg_k <= a_cols,
                      "cmt_gemm_segmented: segment %d reads columns [%d, %d) of %d", i, seg_acol_host[i], seg_acol_host[i] + seg_k, a_cols);
        g.seg_acol[i] = seg_acol_host[i];
        g.seg_shift[i] = seg_row_shift_host[i];
    }
    return launch_tc_gemm(g, batch, static_cast<cudaStream_t>(stream));
}

int cmt_nchw_to_padded_nhwc(const void* x, void* out, int B, int C, int H, int W, int guard_rows, int in_dtype, void* stream,
                            int out_dtype, const uint8_t* frame_valid) {
    CMT_REQUIRE_DEVICE();
    return launch_nchw_to_padded_nhwc(x, out, B, C, H, W, guard_rows, in_dtype, out_dtype, frame_valid,
                                      static_cast<cudaStream_t>(stream));
}

int cmt_shared_conv_tokens(const void* xp, const void* w, const float* bias, const float* bev_pos, void* xk, void* xv, int B,
                           int Cin, int Cout, int H, int W, int guard_rows, int64_t out_frame_stride, int tok_begin, int tok_end,
                           void* stream, int dtype) {
    CMT_REQUIRE_DEVICE();
    CMT_CHECK_ARG(xp && w && bias && bev_pos && xk && xv, "cmt_shared_conv_tokens: null pointer");
    CMT_CHECK_ARG(dtype == CMT_BF16 || dtype == CMT_F16, "cmt_shared_conv_tokens: bad dtype");
    CMT_CHECK_ARG(B > 0 && Cin > 0 && Cin % 64 == 0 && Cout > 0 && Cout % 32 == 0 && H > 0 && W > 0 && guard_rows >= W + 3,
                  "cmt_shared_conv_tokens: bad shape (Cin %% 64, Cout %% 32, guard_rows >= W + 3)");
    CMT_CHECK_ARG(0 <= tok_begin && tok_begin < tok_end && tok_end <= H * W, "cmt_shared_conv_tokens: bad token range");
    const int Wp = W + 2, Hp = H + 2;
    const long long rows = 2ll * guard_rows + static_cast<long long>(Hp) * Wp;
    GemmArgs g{};
    g.A = xp;
    g.B = w;
    g.bias = bias;
    g.C = xv;
    g.M = Hp * Wp;
    g.N = Cout;
    g.K = 9 * Cin;
    g.lda = Cin;
    g.ldb = 9ll * Cin;
    g.ldc = Cout;
    g.cb = Cout;
    g.strideA = rows * Cin;
    g.strideB = 0;
    g.strideC = 0;
    g.alpha = 1.0f;
    g.relu = 1;
    g.out_16 = 1;
    g.f16 = dtype == CMT_F16;
    g.n_seg = 9;
    g.seg_k = Cin;
    g.a_row_off = guard_rows;
    g.a_rows = rows;
    g.a_cols = Cin;
    for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) {
            g.seg_acol[ky * 3 + kx] = 0;
            g.seg_shift[ky * 3 + kx] = (ky - 1) * Wp + (kx - 1);
        }
    g.conv_xk = xk;
    g.conv_xv = xv;
    g.conv_pos = bev_pos;
    g.conv_W = W;
    g.conv_H = H;
    g.conv_Wp = Wp;
    g.conv_tok_begin = tok_begin;
    g.conv_tok_end = tok_end;
    g.conv_frame_stride = out_frame_stride;
    return launch_tc_gemm(g, B, static_cast<cudaStream_t>(stream));
}

size_t cmt_cross_attn_workspace_bytes(int B, int H, int Nq, int n_kv_tokens) {
    return tc_attn_workspace_bytes(B, H, Nq, n_kv_tokens);
}

int cmt_cross_attn_fwd(const void* q, const void* k, const void* vt, void* o, float* lse, int B, int H, int Nq,
                       int N_kv, int kv_begin, int kv_end, int64_t q_ld, int64_t k_bstride, int64_t k_hstride,
                       int64_t v_bstride, int64_t v_hstride, int64_t v_ld, const unsigned char* key_keep,
                       const float* q_norm2_max, const float* k_norm2_max, int64_t kn_bstride, int dtype,
                       int o_dtype, void* workspace, size_t workspace_bytes, void* stream) {
    CMT_REQUIRE_DEVICE();
    CMT_CHECK_ARG(q && k && vt && o, "cmt_cross_attn_fwd: null pointer");
    CMT_CHECK_ARG(B > 0 && H > 0 && Nq > 0 && N_kv > 0, "cmt_cross_attn_fwd: bad shape");
    CMT_CHECK_ARG(0 <= kv_begin && kv_begin < kv_end && kv_end <= N_kv,
                  "cmt_cross_attn_fwd: bad token range [%d,%d) of %d", kv_begin, kv_end, N_kv);
    CMT_CHECK_ARG(dtype == CMT_F32 || dtype == CMT_BF16 || dtype == CMT_F16 || dtype == CMT_BF16_SIMT,
                  "cmt_cross_attn_fwd: bad dtype");
    CMT_CHECK_ARG(o_dtype == CMT_F32 || o_dtype == CMT_BF16 || o_dtype == CMT_F16, "cmt_cross_attn_fwd: bad o_dtype");
    CMT_CHECK_ARG(o_dtype != CMT_F16 || dtype == CMT_F16, "cmt_cross_attn_fwd: an fp16 output needs fp16 operands");
    CMT_CHECK_ARG(q_ld >= H * 32 && v_ld >= kv_end, "cmt_cross_attn_fwd: bad leading dimensions");
    AttnArgs a{};
    a.q = q;
    a.k = k;
    a.vt = vt;
    a.o = o;
    a.lse = lse;
    a.B = B;
    a.H = H;
    a.Nq = Nq;
    a.N_kv = N_kv;
    a.kv_begin = kv_begin;
    a.kv_end = kv_end;
    a.q_ld = q_ld;
    a.k_bstride = k_bstride;
    a.k_hstride = k_hstride;
    a.v_bstride = v_bstride;
    a.v_hstride = v_hstride;
    a.v_ld = v_ld;
    a.f16 = dtype == CMT_F16;
    a.o_dtype = o_dtype;
    a.key_keep = key_keep;
    a.q_norm2 = q_norm2_max;
    a.k_norm2 = k_norm2_max;
    a.kn_bstride = kn_bstride;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (dtype == CMT_BF16 || dtype == CMT_F16) return launch_tc_attn(a, workspace, workspace_bytes, s);
    return launch_simt_attn(a, dtype == CMT_BF16_SIMT ? CMT_BF16 : dtype, s);
}

int cmt_task_head_tail(const float* h, const float* gamma, const float* beta, const float* w2, const float* b2, float* out,
                       int L, int M, int NH, int HC, int CMAX, float eps, int ksize, int Nq, const float* ref_logit,
                       const int* dec_comp, const float* dec_scale, const float* dec_offset, const int64_t* head_off_host,
                       const int* head_cout_host, void* stream) {
    CMT_REQUIRE_DEVICE();
    CMT_CHECK_ARG(h && gamma && beta && w2 && b2 && out, "cmt_task_head_tail: null pointer");
    return launch_task_head_tail(h, gamma, beta, w2, b2, out, L, M, NH, HC, CMAX, eps, ksize, Nq, ref_logit, dec_comp, dec_scale,
                                 dec_offset, reinterpret_cast<const long long*>(head_off_host), head_cout_host,
                                 static_cast<cudaStream_t>(stream));
}

int cmt_split3_bf16(const float* a, const float* b, void* out, float* merged, int64_t Z, int Nq, int C, int frames,
                    int64_t layer_stride_rows, void* stream, const uint8_t* node_valid) {
    CMT_REQUIRE_DEVICE();
    return launch_split3(a, b, out, merged, Z, Nq, C, frames, layer_stride_rows, node_valid,
                         static_cast<cudaStream_t>(stream));
}

int cmt_debug_attn_timing(void* dev_buf_i64) { return cmt::tc_attn_set_timing_buffer(static_cast<long long*>(dev_buf_i64)); }

int cmt_lse_merge(const float* o_parts, const float* lse_parts, void* o, float* lse, int G, int B, int H,
                  int Nq, int64_t o_gstride, int64_t lse_gstride, int o_dtype, void* stream) {
    CMT_REQUIRE_DEVICE();
    return launch_lse_merge(o_parts, lse_parts, o, lse, G, B, H, Nq, o_gstride, lse_gstride, o_dtype,
                            static_cast<cudaStream_t>(stream));
}

int cmt_lse_merge_peer(const void* const* records, void* const* ctx, void* const* arrive, void* state, int rank, int G,
                       int B, int H, int Nq, int o_dtype, int scatter, void* stream) {
    CMT_REQUIRE_DEVICE();
    return launch_lse_merge_peer(records, ctx, arrive, state, rank, G, B, H, Nq, o_dtype, scatter, static_cast<cudaStream_t>(stream));
}

int cmt_add_layernorm(const float* x, const float* r, const float* gamma, const float* beta, float eps, int M, int C,
                      float* y, const float* gamma2, const float* beta2, float* y2, const float* add, void* ylp,
                      void* yadd, int lp_dtype, int flags, void* stream) {
    CMT_REQUIRE_DEVICE();
    return launch_add_layernorm(x, r, gamma, beta, eps, M, C, y, gamma2, beta2, y2, add, ylp, yadd, lp_dtype, flags,
                                static_cast<cudaStream_t>(stream));
}

int cmt_bbox_topk_decode(const float* const* task_ptrs_host, const int* task_classes_host, int T, int B, int Nq,
                         int num_classes, int max_num, const float* post_center_range_host, float score_threshold,
                         int use_score_threshold, int bottom_center, float* boxes, float* scores, int64_t* labels,
                         int32_t* count, int64_t* topk_index, void* stream, const uint8_t* node_valid, int n_nodes) {
    CMT_REQUIRE_DEVICE();
    return launch_bbox_topk_decode(task_ptrs_host, task_classes_host, T, B, Nq, num_classes, max_num, post_center_range_host,
                                   score_threshold, use_score_threshold, bottom_center, boxes, scores,
                                   reinterpret_cast<long long*>(labels), count, reinterpret_cast<long long*>(topk_index),
                                   node_valid, n_nodes, static_cast<cudaStream_t>(stream));
}

int cmt_coop_max(const float* a, const float* b, float* out, int64_t n, void* stream) {
    CMT_REQUIRE_DEVICE();
    return launch_coop_max(a, b, out, n, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
