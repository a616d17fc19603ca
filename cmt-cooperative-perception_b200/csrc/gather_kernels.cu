// K4 token gather (NCHW fp32 -> token-major, BEV ++ image concat, +pos, cast), the V2I
// element-wise max merge, and the log-sum-exp merge of attention partials.  HBM bound.
//
// Reference arithmetic followed (never copied):
//   gather : models/utils/cmt_transformer.py:105-110 + models/utils/petr_transformer.py:296-299
//   coop   : models/dense_heads/cmt_head_coop.py:358,383-389
#include <cuda_fp16.h>

#include "kernels.cuh"

namespace cmt {

constexpr int kTileTok = 32;

// Block = one tile of 32 consecutive tokens of one source map (the BEV map of frame b, or one
// camera of frame b) x all C channels.  Phase 1 reads channel rows (128 contiguous bytes per
// warp load) into a transposed smem tile [token][channel] (row pitch C+1 words -> conflict-free
// writes); phase 2 lets each warp emit whole token rows (C contiguous elements) for xk and xv.
//
// kIn: dtype of the feature maps -- CMT_F32, CMT_BF16 or CMT_F16.  The kernel rounds every feature to the
// output dtype anyway, so a backbone / neck (or a host pipeline) that hands over 16-bit features halves the read
// (and, end to end, the PCIe) traffic without changing the result of the bf16 path.  16-bit sources with an even
// token count use 32-bit loads: each half-warp reads the 32 tokens of one channel (64 contiguous bytes), the two
// halves take adjacent channels, which keeps the transposed shared-memory writes conflict-free.
//
// [tok_begin, tok_end): only these tokens of the concatenated BEV ++ image axis are produced (KV-token split across
// GPUs: a rank gathers, projects and attends its own range only); row 0 of xk / xv is token tok_begin.
//
// sensor_valid (nullable): [S, B] bytes, row 0 the BEV map when n_bev > 0, then one row per camera.  The tokens of an
// absent (sensor, frame) are written as zero rows of xk AND xv: neither its features nor its position encoding is
// read (they may hold NaN), so every K / V row stays finite and the attention's key mask only has to drop them.
__device__ __forceinline__ bool sensor_present(const uint8_t* sensor_valid, int row, int b, int B) {
    return sensor_valid == nullptr || sensor_valid[static_cast<long long>(row) * B + b] != 0;
}

template <int kIn>
__device__ __forceinline__ float load_feat(const void* p, long long i) {
    if (kIn == CMT_F32) return __ldg(reinterpret_cast<const float*>(p) + i);
    const unsigned short raw = __ldg(reinterpret_cast<const unsigned short*>(p) + i);
    if (kIn == CMT_BF16) return __uint_as_float(static_cast<uint32_t>(raw) << 16);
    return __half2float(__ushort_as_half(raw));
}
template <int kIn>
__device__ __forceinline__ void unpack_feat2(uint32_t w, float& lo, float& hi) {
    if (kIn == CMT_BF16) {
        lo = __uint_as_float(w << 16);
        hi = __uint_as_float(w & 0xffff0000u);
    } else {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w));
        lo = f.x;
        hi = f.y;
    }
}

// kOut: dtype of xk / xv, CMT_F32 | CMT_BF16 | CMT_F16.
template <int kOut, int kIn>
__global__ void __launch_bounds__(256) gather_tokens_kernel(
    const void* __restrict__ x_bev, const void* __restrict__ x_img,
    const float* __restrict__ bev_pos, const float* __restrict__ rv_pos, void* __restrict__ xk,
    void* __restrict__ xv, int C, int n_bev, int V, int n_img, int tiles_bev, int tiles_img, int tok_begin,
    int tok_end, int rv_tok0, int rv_rows, const uint8_t* __restrict__ sensor_valid) {
    extern __shared__ float tile[];  // [kTileTok][C + 1]
    constexpr int ESZ = kIn == CMT_F32 ? 4 : 2;
    const int b = blockIdx.y;
    const int pitch = C + 1;
    int tix = blockIdx.x;
    const unsigned char* src;   // [C, n_src] channel-major
    const float* pos;           // [n_src, C] token-major (already offset to this source's first token)
    int n_src, t0;
    long long dst_tok0;         // first destination token of this source inside the frame
    bool present;               // block-uniform
    if (tix < tiles_bev) {
        src = reinterpret_cast<const unsigned char*>(x_bev) + static_cast<long long>(b) * C * n_bev * ESZ;
        pos = bev_pos;
        n_src = n_bev;
        t0 = tix * kTileTok;
        dst_tok0 = 0;
        present = sensor_present(sensor_valid, 0, b, gridDim.y);
    } else {
        tix -= tiles_bev;
        const int v = tix / tiles_img;
        const int cam = b * V + v;
        src = reinterpret_cast<const unsigned char*>(x_img) + static_cast<long long>(cam) * C * n_img * ESZ;
        // rv_pos holds rows [rv_tok0, rv_tok0 + rv_rows) of every frame's V * n_img image tokens (all of them by default; a
        // rank of a KV-token split computes the position-encoding MLP for its own image tokens only)
        pos = rv_pos + (static_cast<long long>(b) * rv_rows + static_cast<long long>(v) * n_img - rv_tok0) * C;
        n_src = n_img;
        t0 = (tix % tiles_img) * kTileTok;
        dst_tok0 = n_bev + static_cast<long long>(v) * n_img;
        present = sensor_present(sensor_valid, (n_bev > 0 ? 1 : 0) + v, b, gridDim.y);
    }
    // tiles entirely outside this rank's token range have nothing to do (block-uniform)
    if (dst_tok0 + t0 >= tok_end || dst_tok0 + t0 + kTileTok <= tok_begin) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (kIn != CMT_F32 && (n_src & 1) == 0) {
        // 16-bit features, even token count: lanes 0-15 read channel c, lanes 16-31 channel c + 1, two tokens per lane
        const int half = lane >> 4, l16 = lane & 15;
        const int tok = t0 + 2 * l16;
        for (int c = 2 * warp + half; c < C; c += 16) {
            float lo = 0.0f, hi = 0.0f;
            if (tok < n_src && present)   // n_src even and tok even: both tokens are in range
                unpack_feat2<kIn>(__ldg(reinterpret_cast<const uint32_t*>(src + (static_cast<long long>(c) * n_src + tok) * 2)), lo, hi);
            tile[(2 * l16) * pitch + c] = lo;
            tile[(2 * l16 + 1) * pitch + c] = hi;
        }
    } else {
        const int tok = t0 + lane;
        const bool tok_ok = tok < n_src && present;
        for (int c = warp; c < C; c += 8)
            tile[lane * pitch + c] = tok_ok ? load_feat<kIn>(src, static_cast<long long>(c) * n_src + tok) : 0.0f;
    }
    __syncthreads();
    const long long n_out = tok_end - tok_begin;
    for (int r = warp; r < kTileTok; r += 8) {
        const int st = t0 + r;
        if (st >= n_src) break;
        const long long gtok = dst_tok0 + st;
        if (gtok < tok_begin || gtok >= tok_end) continue;
        const long long drow = (static_cast<long long>(b) * n_out + (gtok - tok_begin)) * C;
        const float* prow = pos + static_cast<long long>(st) * C;
        const float* trow = tile + r * pitch;
        for (int c = lane * 2; c < C; c += 64) {
            const float m0 = trow[c], m1 = trow[c + 1];
            const float2 pp = present ? *reinterpret_cast<const float2*>(prow + c) : make_float2(0.0f, 0.0f);
            if (kOut != CMT_F32) {
                reinterpret_cast<uint32_t*>(xk)[(drow + c) >> 1] = pack_lp2<kOut>(m0 + pp.x, m1 + pp.y);
                reinterpret_cast<uint32_t*>(xv)[(drow + c) >> 1] = pack_lp2<kOut>(m0, m1);
            } else {
                *reinterpret_cast<float2*>(reinterpret_cast<float*>(xk) + drow + c) =
                    make_float2(m0 + pp.x, m1 + pp.y);
                *reinterpret_cast<float2*>(reinterpret_cast<float*>(xv) + drow + c) =
                    make_float2(m0, m1);
            }
        }
    }
}

int launch_gather_tokens(const void* x_bev, const void* x_img, const float* bev_pos,
                         const float* rv_pos, void* xk, void* xv, int B, int C, int n_bev, int V,
                         int n_img, int tok_begin, int tok_end, int rv_tok0, int rv_rows, int feat_dtype, int out_dtype,
                         const uint8_t* sensor_valid, cudaStream_t stream) {
    CMT_CHECK_ARG(xk && xv, "cmt_gather_tokens: null output");
    CMT_CHECK_ARG(B > 0 && C > 0 && (C % 2) == 0, "cmt_gather_tokens: bad B/C");
    CMT_CHECK_ARG(n_bev >= 0 && V >= 0 && n_img >= 0, "cmt_gather_tokens: bad token counts");
    CMT_CHECK_ARG(n_bev == 0 || x_bev == nullptr || bev_pos, "cmt_gather_tokens: BEV position encoding missing");
    CMT_CHECK_ARG(V == 0 || n_img == 0 || (x_img && rv_pos), "cmt_gather_tokens: image pointers missing");
    CMT_CHECK_ARG(out_dtype == CMT_F32 || out_dtype == CMT_BF16 || out_dtype == CMT_F16, "cmt_gather_tokens: bad output dtype");
    CMT_CHECK_ARG(feat_dtype == CMT_F32 || feat_dtype == CMT_BF16 || feat_dtype == CMT_F16, "cmt_gather_tokens: bad feature dtype");
    CMT_CHECK_ARG(B <= 65535, "cmt_gather_tokens: batch too large for one launch");
    const long long n_kv = n_bev + static_cast<long long>(V) * n_img;
    CMT_CHECK_ARG(0 <= tok_begin && tok_begin <= tok_end && tok_end <= n_kv, "cmt_gather_tokens: bad token range [%d,%d) of %lld",
                  tok_begin, tok_end, n_kv);
    if (rv_rows <= 0) {   // default: rv_pos covers every image token
        rv_tok0 = 0;
        rv_rows = V * n_img;
    }
    {
        // image tokens actually gathered must lie inside the rows rv_pos holds
        const long long img_lo = tok_begin > n_bev ? tok_begin - n_bev : 0, img_hi = tok_end > n_bev ? tok_end - n_bev : 0;
        CMT_CHECK_ARG(img_hi <= img_lo || (rv_tok0 <= img_lo && img_hi <= static_cast<long long>(rv_tok0) + rv_rows),
                      "cmt_gather_tokens: rv_pos rows [%d, %d) do not cover the gathered image tokens [%lld, %lld)", rv_tok0,
                      rv_tok0 + rv_rows, img_lo, img_hi);
    }
    CMT_CHECK_ARG(feat_dtype == CMT_F32 || ((reinterpret_cast<uintptr_t>(x_bev) | reinterpret_cast<uintptr_t>(x_img)) & 3) == 0,
                  "cmt_gather_tokens: 16-bit feature maps must be 4-byte aligned");
    // x_bev == NULL with n_bev > 0: the BEV rows [0, n_bev) of xk / xv are produced elsewhere (the shared_conv epilogue,
    // cmt_shared_conv_tokens); only the image tokens are gathered, at their usual row offset
    const int tiles_bev = x_bev != nullptr ? (n_bev + kTileTok - 1) / kTileTok : 0;
    const int tiles_img = (n_img + kTileTok - 1) / kTileTok;
    const int tiles = tiles_bev + V * tiles_img;
    if (tiles == 0 || tok_begin == tok_end) return CMT_OK;
    const size_t smem = static_cast<size_t>(kTileTok) * (C + 1) * sizeof(float);
    CMT_CHECK_ARG(smem <= 48 * 1024, "cmt_gather_tokens: C too large (%d)", C);
    dim3 grid(tiles, B);
#define CMT_GATHER_LAUNCH(OUT, IN)                                                                            \
    gather_tokens_kernel<OUT, IN><<<grid, 256, smem, stream>>>(x_bev, x_img, bev_pos, rv_pos, xk, xv, C, n_bev, V, \
                                                               n_img, tiles_bev, tiles_img, tok_begin, tok_end, rv_tok0, rv_rows, \
                                                               sensor_valid)
#define CMT_GATHER_LAUNCH_OUT(IN)                                                                             \
    do {                                                                                                      \
        if (out_dtype == CMT_BF16) CMT_GATHER_LAUNCH(CMT_BF16, IN);                                          \
        else if (out_dtype == CMT_F16) CMT_GATHER_LAUNCH(CMT_F16, IN);                                       \
        else CMT_GATHER_LAUNCH(CMT_F32, IN);                                                                 \
    } while (0)
    if (feat_dtype == CMT_F32) CMT_GATHER_LAUNCH_OUT(CMT_F32);
    else if (feat_dtype == CMT_BF16) CMT_GATHER_LAUNCH_OUT(CMT_BF16);
    else CMT_GATHER_LAUNCH_OUT(CMT_F16);
#undef CMT_GATHER_LAUNCH_OUT
#undef CMT_GATHER_LAUNCH
    CMT_LAUNCH_CHECK("cmt_gather_tokens");
    return CMT_OK;
}

// ---------------------------------------------------------------------------
// NCHW feature map -> zero-padded, channel-last 16-bit rows (kOut = CMT_BF16 | CMT_F16): the A operand of the 3x3 shared_conv implicit GEMM
// (cmt_head.py:280-287,481).  Frame b occupies `rows_per_frame = 2 * guard + (H + 2) * (W + 2)` rows of C channels; pixel
// (y, x) lands in row guard + (y + 1) * (W + 2) + (x + 1).  Only interior rows are written: the border and guard rows
// are zero from the (one-time) allocation, so a filter tap is a pure row shift of -(W+2)-1 .. +(W+2)+1 with no edge
// handling.  Block = 32 consecutive pixels x one block of up to 256 channels, same transpose tile as the token gather.
// frame_valid (nullable): [B] bytes; the interior rows of a frame whose map is absent are written as zeros (its input,
// which may hold NaN, is not read), so the implicit GEMM produces finite BEV rows for it.
template <int kIn, int kOut>
__global__ void __launch_bounds__(256) nchw_to_padded_nhwc_kernel(const void* __restrict__ x, uint16_t* __restrict__ out,
                                                                  int C, int H, int W, int guard, long long rows_per_frame,
                                                                  const uint8_t* __restrict__ frame_valid) {
    extern __shared__ float tile[];  // [32][257]
    constexpr int ESZ = kIn == CMT_F32 ? 4 : 2;
    constexpr int CB = 256, pitch = CB + 1;
    const int b = blockIdx.y, c0 = blockIdx.z * CB;
    const int nc = min(CB, C - c0);
    const int n_src = H * W;
    const int t0 = blockIdx.x * kTileTok;
    const unsigned char* src = reinterpret_cast<const unsigned char*>(x) + (static_cast<long long>(b) * C + c0) * n_src * ESZ;
    const bool present = frame_valid == nullptr || frame_valid[b] != 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (kIn != CMT_F32 && (n_src & 1) == 0) {
        const int half = lane >> 4, l16 = lane & 15;
        const int tok = t0 + 2 * l16;
        for (int c = 2 * warp + half; c < nc; c += 16) {
            float lo = 0.0f, hi = 0.0f;
            if (tok < n_src && present)
                unpack_feat2<kIn>(__ldg(reinterpret_cast<const uint32_t*>(src + (static_cast<long long>(c) * n_src + tok) * 2)), lo, hi);
            tile[(2 * l16) * pitch + c] = lo;
            tile[(2 * l16 + 1) * pitch + c] = hi;
        }
    } else {
        const int tok = t0 + lane;
        const bool tok_ok = tok < n_src && present;
        for (int c = warp; c < nc; c += 8)
            tile[lane * pitch + c] = tok_ok ? load_feat<kIn>(src, static_cast<long long>(c) * n_src + tok) : 0.0f;
    }
    __syncthreads();
    for (int r = warp; r < kTileTok; r += 8) {
        const int st = t0 + r;
        if (st >= n_src) break;
        const int y = st / W, xx = st - y * W;
        const long long row = static_cast<long long>(b) * rows_per_frame + guard + static_cast<long long>(y + 1) * (W + 2) + (xx + 1);
        uint32_t* dst = reinterpret_cast<uint32_t*>(out + row * C + c0);
        const float* trow = tile + r * pitch;
        for (int c = lane * 2; c < nc; c += 64) dst[c >> 1] = pack_lp2<kOut>(trow[c], trow[c + 1]);
    }
}

int launch_nchw_to_padded_nhwc(const void* x, void* out, int B, int C, int H, int W, int guard, int in_dtype,
                               int out_dtype, const uint8_t* frame_valid, cudaStream_t stream) {
    CMT_CHECK_ARG(x && out && B > 0 && C > 0 && C % 2 == 0 && H > 0 && W > 0 && guard >= W + 3,
                  "cmt_nchw_to_padded_nhwc: bad arguments (guard must be >= W + 3)");
    CMT_CHECK_ARG(in_dtype == CMT_F32 || in_dtype == CMT_BF16 || in_dtype == CMT_F16, "cmt_nchw_to_padded_nhwc: bad dtype");
    CMT_CHECK_ARG(out_dtype == CMT_BF16 || out_dtype == CMT_F16, "cmt_nchw_to_padded_nhwc: bad output dtype");
    CMT_CHECK_ARG(B <= 65535, "cmt_nchw_to_padded_nhwc: batch too large");
    CMT_CHECK_ARG(in_dtype == CMT_F32 || (reinterpret_cast<uintptr_t>(x) & 3) == 0, "cmt_nchw_to_padded_nhwc: unaligned input");
    const long long rows = 2ll * guard + static_cast<long long>(H + 2) * (W + 2);
    dim3 grid((H * W + kTileTok - 1) / kTileTok, B, (C + 255) / 256);
    const size_t smem = static_cast<size_t>(kTileTok) * 257 * sizeof(float);
    uint16_t* o = reinterpret_cast<uint16_t*>(out);
#define CMT_LAYOUT_LAUNCH(IN, OUT) \
    nchw_to_padded_nhwc_kernel<IN, OUT><<<grid, 256, smem, stream>>>(x, o, C, H, W, guard, rows, frame_valid)
    if (out_dtype == CMT_BF16) {
        if (in_dtype == CMT_F32) CMT_LAYOUT_LAUNCH(CMT_F32, CMT_BF16);
        else if (in_dtype == CMT_BF16) CMT_LAYOUT_LAUNCH(CMT_BF16, CMT_BF16);
        else CMT_LAYOUT_LAUNCH(CMT_F16, CMT_BF16);
    } else {
        if (in_dtype == CMT_F32) CMT_LAYOUT_LAUNCH(CMT_F32, CMT_F16);
        else if (in_dtype == CMT_BF16) CMT_LAYOUT_LAUNCH(CMT_BF16, CMT_F16);
        else CMT_LAYOUT_LAUNCH(CMT_F16, CMT_F16);
    }
#undef CMT_LAYOUT_LAUNCH
    CMT_LAUNCH_CHECK("cmt_nchw_to_padded_nhwc");
    return CMT_OK;
}

// ---------------------------------------------------------------------------
// Key-keep bytes of the cross-attention from the per-frame sensor mask: keep[b][t] = sensor_valid[s(t)][b] for the
// concatenated BEV ++ image token axis, s = 0 for the n_bev BEV tokens (when n_bev > 0), then one row per camera of
// n_img tokens.  One thread per byte (a few hundred KB per batch).
__global__ void __launch_bounds__(256) sensor_key_keep_kernel(const uint8_t* __restrict__ sensor_valid,
                                                              uint8_t* __restrict__ keep, int B, int n_bev, int n_img,
                                                              long long n_kv) {
    const long long total = n_kv * B;
    const int cam0 = n_bev > 0 ? 1 : 0;
    for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int b = static_cast<int>(t / n_kv);
        const long long tok = t - static_cast<long long>(b) * n_kv;
        const int row = tok < n_bev ? 0 : cam0 + static_cast<int>((tok - n_bev) / n_img);
        keep[t] = sensor_valid[static_cast<long long>(row) * B + b] != 0 ? 1 : 0;
    }
}

int launch_sensor_key_keep(const uint8_t* sensor_valid, uint8_t* keep, int B, int n_bev, int V, int n_img,
                           cudaStream_t stream) {
    CMT_CHECK_ARG(sensor_valid && keep, "cmt_sensor_key_keep: null pointer");
    CMT_CHECK_ARG(B > 0 && n_bev >= 0 && V >= 0 && n_img >= 0, "cmt_sensor_key_keep: bad shape");
    const long long n_kv = n_bev + static_cast<long long>(V) * n_img;
    CMT_CHECK_ARG(n_kv > 0, "cmt_sensor_key_keep: no tokens");
    const long long total = n_kv * B;
    long long blocks = (total + 255) / 256;
    const long long cap = static_cast<long long>(device_sm_count()) * 16;
    if (blocks > cap) blocks = cap;
    sensor_key_keep_kernel<<<static_cast<int>(blocks), 256, 0, stream>>>(sensor_valid, keep, B, n_bev, n_img, n_kv);
    CMT_LAUNCH_CHECK("cmt_sensor_key_keep");
    return CMT_OK;
}

// ---------------------------------------------------------------------------
__device__ __forceinline__ float nan_to_num(float x) {
    if (x != x) return 0.0f;
    if (x == __int_as_float(0x7f800000)) return 3.4028234663852886e38f;
    if (x == __int_as_float(0xff800000)) return -3.4028234663852886e38f;
    return x;
}

__global__ void __launch_bounds__(256) coop_max_kernel(const float* __restrict__ a,
                                                       const float* __restrict__ b,
                                                       float* __restrict__ out, long long n) {
    const long long n4 = n >> 2;
    for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < n4;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const float4 x = reinterpret_cast<const float4*>(a)[t];
        const float4 y = reinterpret_cast<const float4*>(b)[t];
        float4 r;
        r.x = fmaxf(nan_to_num(x.x), nan_to_num(y.x));
        r.y = fmaxf(nan_to_num(x.y), nan_to_num(y.y));
        r.z = fmaxf(nan_to_num(x.z), nan_to_num(y.z));
        r.w = fmaxf(nan_to_num(x.w), nan_to_num(y.w));
        reinterpret_cast<float4*>(out)[t] = r;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const long long t = (n4 << 2) + threadIdx.x;
        out[t] = fmaxf(nan_to_num(a[t]), nan_to_num(b[t]));
    }
}

int launch_coop_max(const float* a, const float* b, float* out, long long n, cudaStream_t stream) {
    CMT_CHECK_ARG(a && b && out && n >= 0, "cmt_coop_max: bad arguments");
    CMT_CHECK_ARG(((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) |
                    reinterpret_cast<uintptr_t>(out)) & 15) == 0,
                  "cmt_coop_max: pointers must be 16-byte aligned");
    if (n == 0) return CMT_OK;
    long long blocks = ((n >> 2) + 255) / 256;
    const long long cap = static_cast<long long>(device_sm_count()) * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    coop_max_kernel<<<static_cast<int>(blocks), 256, 0, stream>>>(a, b, out, n);
    CMT_LAUNCH_CHECK("cmt_coop_max");
    return CMT_OK;
}

// ---------------------------------------------------------------------------
// o = sum_g exp(lse_g - lse) * o_g ,  lse = log(sum_g exp(lse_g)).  One thread per (b, n, h, 4 dims).  kOut: dtype of o.
template <int kOut>
__global__ void __launch_bounds__(256) lse_merge_kernel(const float* __restrict__ o_parts,
                                                        const float* __restrict__ lse_parts,
                                                        void* __restrict__ o,
                                                        float* __restrict__ lse, int G, int B, int H,
                                                        int Nq, long long part_o, long long part_l) {
    const long long total = static_cast<long long>(B) * Nq * H * 8;
    for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int q4 = static_cast<int>(t & 7);
        const int h = static_cast<int>((t >> 3) % H);
        const int n = static_cast<int>(((t >> 3) / H) % Nq);
        const int b = static_cast<int>((t >> 3) / (static_cast<long long>(H) * Nq));
        const long long li = (static_cast<long long>(b) * H + h) * Nq + n;
        float mx = -INFINITY;
        for (int g = 0; g < G; ++g) mx = fmaxf(mx, lse_parts[g * part_l + li]);
        float den = 0.0f;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int g = 0; g < G; ++g) {
            const float l = lse_parts[g * part_l + li];
            const float w = (l == -INFINITY) ? 0.0f : __expf(l - mx);
            den += w;
            const float4 x = reinterpret_cast<const float4*>(o_parts + g * part_o)[t];
            acc.x = fmaf(w, x.x, acc.x);
            acc.y = fmaf(w, x.y, acc.y);
            acc.z = fmaf(w, x.z, acc.z);
            acc.w = fmaf(w, x.w, acc.w);
        }
        const float inv = den > 0.0f ? 1.0f / den : 0.0f;
        acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
        if (kOut != CMT_F32) {
            uint2 w;
            w.x = pack_lp2<kOut>(acc.x, acc.y);
            w.y = pack_lp2<kOut>(acc.z, acc.w);
            reinterpret_cast<uint2*>(o)[t] = w;
        } else {
            reinterpret_cast<float4*>(o)[t] = acc;
        }
        if (lse != nullptr && q4 == 0) lse[li] = mx + logf(den);
    }
}

int launch_lse_merge(const float* o_parts, const float* lse_parts, void* o, float* lse, int G,
                     int B, int H, int Nq, long long o_gstride, long long lse_gstride, int o_dtype, cudaStream_t stream) {
    if (o_gstride <= 0) o_gstride = static_cast<long long>(B) * Nq * H * 32;
    if (lse_gstride <= 0) lse_gstride = static_cast<long long>(B) * H * Nq;
    CMT_CHECK_ARG(o_gstride % 4 == 0 && (reinterpret_cast<uintptr_t>(o_parts) & 15) == 0, "cmt_lse_merge: o parts must be 16-byte aligned");
    CMT_CHECK_ARG(o_parts && lse_parts && o, "cmt_lse_merge: null pointer");
    CMT_CHECK_ARG(G > 0 && B > 0 && H > 0 && Nq > 0, "cmt_lse_merge: bad shape");
    const long long total = static_cast<long long>(B) * Nq * H * 8;
    long long blocks = (total + 255) / 256;
    const long long cap = static_cast<long long>(device_sm_count()) * 16;
    if (blocks > cap) blocks = cap;
    if (o_dtype == CMT_BF16)
        lse_merge_kernel<CMT_BF16><<<static_cast<int>(blocks), 256, 0, stream>>>(o_parts, lse_parts, o,
                                                                                lse, G, B, H, Nq, o_gstride, lse_gstride);
    else if (o_dtype == CMT_F16)
        lse_merge_kernel<CMT_F16><<<static_cast<int>(blocks), 256, 0, stream>>>(o_parts, lse_parts, o,
                                                                               lse, G, B, H, Nq, o_gstride, lse_gstride);
    else if (o_dtype == CMT_F32)
        lse_merge_kernel<CMT_F32><<<static_cast<int>(blocks), 256, 0, stream>>>(o_parts, lse_parts, o,
                                                                               lse, G, B, H, Nq, o_gstride, lse_gstride);
    else
        CMT_CHECK_ARG(false, "cmt_lse_merge: bad dtype");
    CMT_LAUNCH_CHECK("cmt_lse_merge");
    return CMT_OK;
}

// ---------------------------------------------------------------------------
// KV-token split: exchange + merge + redistribution in ONE kernel over peer memory (NVLink / NVSwitch loads and stores,
// no NCCL call on the path).  Every rank keeps its packed (O | LSE) record of the layer, and a context buffer, in memory
// mapped into all ranks of the group (torch symmetric memory on the host side).  The kernel is a reduce-scatter and an
// all-gather folded around the merge:
//   1. announce "my record of exchange `seq` is complete" to every rank: fence.sys + one 32-bit store per peer into
//      that peer's arrival counters (the record was written by the preceding kernels of this stream),
//   2. wait until every rank has announced `seq` (acquire loads of the rank's OWN counters: local memory, no NVLink polling),
//   3. merge 1/G of the rows: the thread reads the G records' values for its 4 elements -- G - 1 of them through NVLink --
//      and stores the merged result into EVERY rank's context buffer (G - 1 remote stores of 8 or 16 bytes, coalesced),
//   4. the last block to finish announces "my rows are in your context buffer" to every rank, waits for the same from all
//      of them and publishes the exchange number; when the kernel ends the local context buffer is complete.
// Per rank and exchange NVLink carries (G-1)/G of a record in and (G-1)/G of a context out (7.6 MB + 3.7 MB at the bench
// shape whatever G is), where an all-gather of records delivers (G-1) records (53 MB at G = 8).
// `seq` lives in device memory (state[0]; state[1] counts finished blocks), so the kernel replays unchanged from a CUDA
// graph.  Reuse: a rank announces exchange e + 1 only after its kernel of exchange e has completed, hence (a) a record
// slot may be rewritten as soon as its owner has passed the NEXT exchange -- consecutive exchanges must use different
// record slots, which the host guarantees (one slot per decoder layer, at least two) -- and (b) peers write exchange
// e + 1's context only after the local consumer of context e (earlier in this stream than kernel e + 1) has finished.
constexpr int MAX_PEERS = 8;
struct PeerMergeParams {
    const float* rec[MAX_PEERS];        // rank g's record of this exchange (peer-mapped)
    void* ctx[MAX_PEERS];               // rank g's context buffer of this exchange (peer-mapped)
    unsigned int* arrive[MAX_PEERS];    // rank g's counters (peer-mapped): [0..7] record announced by rank r, [8..15] context rows written by rank r
    unsigned int* state;                // local {seq, done_blocks}
    long long lse_off;                  // element offset of the LSE block inside a record
    long long t_begin, t_end;           // this rank's share of the B*Nq*H*8 four-element groups
    int rank, G, B, H, Nq;
};

__device__ __forceinline__ float4 ld_sys_f4(const float* p) {
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ld_sys_f(const float* p) {
    float v;
    asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}
// all ranks' counters `which` (0: records, 8: context rows) must reach seq; called by threads < G; ~30 s, then trap
// (a rank that never arrives must not hang the box)
__device__ __forceinline__ void peer_wait(const unsigned int* flag, unsigned int seq) {
    unsigned long long t0 = 0;
    for (unsigned int spins = 0;; ++spins) {
        unsigned int v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (static_cast<int>(v - seq) >= 0) break;
        __nanosleep(100);
        if ((spins & 1023u) == 1023u) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 30000000000ull) __trap();
        }
    }
}

// kScatter = false (small groups): every rank merges ALL rows from the G records (G - 1 records over NVLink) into its own
// context buffer; steps 3b / 4 disappear and the exchange costs one handshake instead of two.  kOut: context dtype.
template <int kOut, bool kScatter>
__global__ void __launch_bounds__(256) lse_merge_peer_kernel(const PeerMergeParams p) {
    __shared__ unsigned int seq_s;
    __shared__ int last_s;
    if (threadIdx.x == 0) {
        unsigned int seq;
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(seq) : "l"(p.state) : "memory");
        seq_s = seq + 1;
    }
    __syncthreads();
    const unsigned int seq = seq_s;
    if (blockIdx.x == 0 && threadIdx.x < p.G) {
        __threadfence_system();   // the record (written by earlier kernels of this stream) before the announcement
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.arrive[threadIdx.x] + p.rank), "r"(seq) : "memory");
    }
    if (threadIdx.x < p.G) peer_wait(p.arrive[p.rank] + threadIdx.x, seq);
    __syncthreads();
    for (long long t = p.t_begin + blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < p.t_end;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int h = static_cast<int>((t >> 3) % p.H);
        const int n = static_cast<int>(((t >> 3) / p.H) % p.Nq);
        const int b = static_cast<int>((t >> 3) / (static_cast<long long>(p.H) * p.Nq));
        const long long li = p.lse_off + (static_cast<long long>(b) * p.H + h) * p.Nq + n;
        float l[MAX_PEERS];
        float4 x[MAX_PEERS];
        // all loads first: G independent round trips in flight per thread
#pragma unroll
        for (int g = 0; g < MAX_PEERS; ++g) {
            if (g < p.G) {
                l[g] = ld_sys_f(p.rec[g] + li);
                x[g] = ld_sys_f4(p.rec[g] + 4 * t);
            }
        }
        float mx = -INFINITY;
#pragma unroll
        for (int g = 0; g < MAX_PEERS; ++g)
            if (g < p.G) mx = fmaxf(mx, l[g]);
        float den = 0.0f;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int g = 0; g < MAX_PEERS; ++g) {
            if (g < p.G) {
                const float w = (l[g] == -INFINITY) ? 0.0f : __expf(l[g] - mx);
                den += w;
                acc.x = fmaf(w, x[g].x, acc.x);
                acc.y = fmaf(w, x[g].y, acc.y);
                acc.z = fmaf(w, x[g].z, acc.z);
                acc.w = fmaf(w, x[g].w, acc.w);
            }
        }
        const float inv = den > 0.0f ? 1.0f / den : 0.0f;
        acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
        if (kOut != CMT_F32) {
            uint2 w;
            w.x = pack_lp2<kOut>(acc.x, acc.y);
            w.y = pack_lp2<kOut>(acc.z, acc.w);
            if (!kScatter) {
                reinterpret_cast<uint2*>(p.ctx[0])[t] = w;
            } else {
#pragma unroll
                for (int g = 0; g < MAX_PEERS; ++g)
                    if (g < p.G) reinterpret_cast<uint2*>(p.ctx[g])[t] = w;
            }
        } else {
            if (!kScatter) {
                reinterpret_cast<float4*>(p.ctx[0])[t] = acc;
            } else {
#pragma unroll
                for (int g = 0; g < MAX_PEERS; ++g)
                    if (g < p.G) reinterpret_cast<float4*>(p.ctx[g])[t] = acc;
            }
        }
    }
    // the last block to finish tells every rank that this rank's rows have landed, waits for the same from everybody,
    // and publishes the exchange number for the next launch
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) last_s = atomicAdd(p.state + 1, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last_s) return;
    if (kScatter && threadIdx.x < p.G) {
        __threadfence_system();
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.arrive[threadIdx.x] + 8 + p.rank), "r"(seq) : "memory");
        peer_wait(p.arrive[p.rank] + 8 + threadIdx.x, seq);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        p.state[1] = 0;
        __threadfence();
        asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p.state), "r"(seq) : "memory");
    }
}

int launch_lse_merge_peer(const void* const* records, void* const* ctx, void* const* arrive, void* state, int rank, int G,
                          int B, int H, int Nq, int o_dtype, int scatter, cudaStream_t stream) {
    CMT_CHECK_ARG(records && ctx && arrive && state, "cmt_lse_merge_peer: null pointer");
    CMT_CHECK_ARG(G > 0 && G <= MAX_PEERS && rank >= 0 && rank < G, "cmt_lse_merge_peer: 1 <= G <= 8, 0 <= rank < G");
    CMT_CHECK_ARG(B > 0 && H > 0 && Nq > 0, "cmt_lse_merge_peer: bad shape");
    CMT_CHECK_ARG(o_dtype == CMT_BF16 || o_dtype == CMT_F16 || o_dtype == CMT_F32, "cmt_lse_merge_peer: bad dtype");
    PeerMergeParams p{};
    for (int g = 0; g < G; ++g) {
        CMT_CHECK_ARG(records[g] && arrive[g] && ctx[g] && (reinterpret_cast<uintptr_t>(records[g]) & 15) == 0 &&
                          (reinterpret_cast<uintptr_t>(ctx[g]) & 15) == 0,
                      "cmt_lse_merge_peer: records / contexts must be non-null and 16-byte aligned");
        p.rec[g] = static_cast<const float*>(records[g]);
        p.ctx[g] = ctx[g];
        p.arrive[g] = static_cast<unsigned int*>(arrive[g]);
    }
    p.state = static_cast<unsigned int*>(state);
    p.lse_off = static_cast<long long>(B) * Nq * H * 32;
    p.rank = rank; p.G = G; p.B = B; p.H = H; p.Nq = Nq;
    const long long total = static_cast<long long>(B) * Nq * H * 8;
    if (scatter < 0) scatter = G > 2;   // measured: two handshakes cost more than reading one whole remote record
    if (scatter) {
        const long long chunk = ((total + G - 1) / G + 31) / 32 * 32;   // whole warps: full 256 / 512-byte stores
        p.t_begin = chunk * rank < total ? chunk * rank : total;
        p.t_end = chunk * (rank + 1) < total ? chunk * (rank + 1) : total;
    } else {
        p.t_begin = 0;
        p.t_end = total;
        p.ctx[0] = ctx[rank];   // the only context this mode writes
    }
    long long blocks = (p.t_end - p.t_begin + 255) / 256;
    const long long cap = static_cast<long long>(device_sm_count()) * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;   // a rank without rows still takes part in the handshakes
    const int nb = static_cast<int>(blocks);
    if (o_dtype == CMT_BF16) {
        if (scatter) lse_merge_peer_kernel<CMT_BF16, true><<<nb, 256, 0, stream>>>(p);
        else lse_merge_peer_kernel<CMT_BF16, false><<<nb, 256, 0, stream>>>(p);
    } else if (o_dtype == CMT_F16) {
        if (scatter) lse_merge_peer_kernel<CMT_F16, true><<<nb, 256, 0, stream>>>(p);
        else lse_merge_peer_kernel<CMT_F16, false><<<nb, 256, 0, stream>>>(p);
    } else {
        if (scatter) lse_merge_peer_kernel<CMT_F32, true><<<nb, 256, 0, stream>>>(p);
        else lse_merge_peer_kernel<CMT_F32, false><<<nb, 256, 0, stream>>>(p);
    }
    CMT_LAUNCH_CHECK("cmt_lse_merge_peer");
    return CMT_OK;
}

}  // namespace cmt
