// Fused residual-add + LayerNorm for the decoder's small ops (mmcv BaseTransformerLayer order
// self_attn, norm, cross_attn, norm, ffn, norm + PETRTransformerDecoder's shared post_norm,
// projects/mmdet3d_plugin/models/utils/petr_transformer.py:347-371).  One warp per 256-wide row:
//   y   = LN(x + r; gamma, beta)                               fp32
//   y2  = LN(y; gamma2, beta2)            (optional: the stacked post-normed intermediate)
//   ylp = cast(y), yadd = cast(y + add)   (optional: bf16|fp16|fp32 A operands of the next projections,
//                                          `add` = query_pos)
// HBM/launch bound; replaces ~6 eager torch launches per norm.
#include "kernels.cuh"

namespace cmt {

template <int kPerLane, int kLp>
__global__ void __launch_bounds__(256) add_layernorm_kernel(const float* __restrict__ x, const float* __restrict__ r,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float eps, int M,
                                                            float* __restrict__ y, const float* __restrict__ gamma2,
                                                            const float* __restrict__ beta2, float* __restrict__ y2,
                                                            const float* __restrict__ add, void* __restrict__ ylp,
                                                            void* __restrict__ yadd, int x_row_broadcast) {
    constexpr int C = kPerLane * 32;
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    for (int row = blockIdx.x * warps_per_block + (threadIdx.x >> 5); row < M; row += gridDim.x * warps_per_block) {
        const long long base = static_cast<long long>(row) * C;
        const long long xbase = x_row_broadcast ? 0 : base;   // x is ONE row shared by every output row
        float v[kPerLane];
        float s = 0.f;
        // lane owns 4-element groups: element index = (g * 32 + lane) * 4 + e  (coalesced 16 B accesses)
#pragma unroll
        for (int g = 0; g < kPerLane / 4; ++g) {
            const int idx = (g * 32 + lane) * 4;
            float4 a = *reinterpret_cast<const float4*>(x + xbase + idx);
            if (r != nullptr) {
                const float4 b = *reinterpret_cast<const float4*>(r + base + idx);
                a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
            }
            v[4 * g] = a.x; v[4 * g + 1] = a.y; v[4 * g + 2] = a.z; v[4 * g + 3] = a.w;
            s += (a.x + a.y) + (a.z + a.w);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        const float mean = s * (1.0f / C);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < kPerLane; ++i) { const float d = v[i] - mean; q = fmaf(d, d, q); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        const float rstd = rsqrtf(q * (1.0f / C) + eps);
        float s2 = 0.f;
#pragma unroll
        for (int g = 0; g < kPerLane / 4; ++g) {
            const int idx = (g * 32 + lane) * 4;
            const float4 ga = __ldg(reinterpret_cast<const float4*>(gamma + idx));
            const float4 be = __ldg(reinterpret_cast<const float4*>(beta + idx));
            v[4 * g] = (v[4 * g] - mean) * rstd * ga.x + be.x;
            v[4 * g + 1] = (v[4 * g + 1] - mean) * rstd * ga.y + be.y;
            v[4 * g + 2] = (v[4 * g + 2] - mean) * rstd * ga.z + be.z;
            v[4 * g + 3] = (v[4 * g + 3] - mean) * rstd * ga.w + be.w;
            *reinterpret_cast<float4*>(y + base + idx) = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
            s2 += (v[4 * g] + v[4 * g + 1]) + (v[4 * g + 2] + v[4 * g + 3]);
            if (ylp != nullptr) {
                if (kLp != CMT_F32) {
                    uint2 w;
                    w.x = pack_lp2<kLp>(v[4 * g], v[4 * g + 1]);
                    w.y = pack_lp2<kLp>(v[4 * g + 2], v[4 * g + 3]);
                    *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(ylp) + base + idx) = w;
                } else {
                    *reinterpret_cast<float4*>(reinterpret_cast<float*>(ylp) + base + idx) =
                        make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
                }
            }
            if (yadd != nullptr) {
                const float4 ad = *reinterpret_cast<const float4*>(add + base + idx);
                const float a0 = v[4 * g] + ad.x, a1 = v[4 * g + 1] + ad.y, a2 = v[4 * g + 2] + ad.z,
                            a3 = v[4 * g + 3] + ad.w;
                if (kLp != CMT_F32) {
                    uint2 w;
                    w.x = pack_lp2<kLp>(a0, a1);
                    w.y = pack_lp2<kLp>(a2, a3);
                    *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(yadd) + base + idx) = w;
                } else {
                    *reinterpret_cast<float4*>(reinterpret_cast<float*>(yadd) + base + idx) = make_float4(a0, a1, a2, a3);
                }
            }
        }
        if (y2 != nullptr) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
            const float mean2 = s2 * (1.0f / C);
            float q2 = 0.f;
#pragma unroll
            for (int i = 0; i < kPerLane; ++i) { const float d = v[i] - mean2; q2 = fmaf(d, d, q2); }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) q2 += __shfl_xor_sync(0xffffffffu, q2, o);
            const float rstd2 = rsqrtf(q2 * (1.0f / C) + eps);
#pragma unroll
            for (int g = 0; g < kPerLane / 4; ++g) {
                const int idx = (g * 32 + lane) * 4;
                const float4 ga = __ldg(reinterpret_cast<const float4*>(gamma2 + idx));
                const float4 be = __ldg(reinterpret_cast<const float4*>(beta2 + idx));
                *reinterpret_cast<float4*>(y2 + base + idx) =
                    make_float4((v[4 * g] - mean2) * rstd2 * ga.x + be.x, (v[4 * g + 1] - mean2) * rstd2 * ga.y + be.y,
                                (v[4 * g + 2] - mean2) * rstd2 * ga.z + be.z, (v[4 * g + 3] - mean2) * rstd2 * ga.w + be.w);
            }
        }
    }
}

int launch_add_layernorm(const float* x, const float* r, const float* gamma, const float* beta, float eps, int M, int C,
                         float* y, const float* gamma2, const float* beta2, float* y2, const float* add, void* ylp,
                         void* yadd, int lp_dtype, int flags, cudaStream_t stream) {
    CMT_CHECK_ARG(x && gamma && beta && y && M > 0, "cmt_add_layernorm: bad arguments");
    const int x_row_broadcast = (flags & CMT_LN_X_ROW_BROADCAST) ? 1 : 0;
    CMT_CHECK_ARG(C == 256, "cmt_add_layernorm: embed dim 256 only (got %d)", C);
    CMT_CHECK_ARG(y2 == nullptr || (gamma2 && beta2), "cmt_add_layernorm: second norm needs gamma2/beta2");
    CMT_CHECK_ARG(yadd == nullptr || add != nullptr, "cmt_add_layernorm: yadd needs add");
    CMT_CHECK_ARG(lp_dtype == CMT_F32 || lp_dtype == CMT_BF16 || lp_dtype == CMT_F16, "cmt_add_layernorm: bad lp dtype");
    const int rows_per_block = 8;
    long long blocks = (M + rows_per_block - 1) / rows_per_block;
    const long long cap = static_cast<long long>(device_sm_count()) * 8;
    if (blocks > cap) blocks = cap;
    if (lp_dtype == CMT_BF16)
        launch_pdl(add_layernorm_kernel<8, CMT_BF16>, dim3(static_cast<int>(blocks)), dim3(256), 0, stream, x, r, gamma, beta, eps, M, y,
                   gamma2, beta2, y2, add, ylp, yadd, x_row_broadcast);
    else if (lp_dtype == CMT_F16)
        launch_pdl(add_layernorm_kernel<8, CMT_F16>, dim3(static_cast<int>(blocks)), dim3(256), 0, stream, x, r, gamma, beta, eps, M, y,
                   gamma2, beta2, y2, add, ylp, yadd, x_row_broadcast);
    else
        launch_pdl(add_layernorm_kernel<8, CMT_F32>, dim3(static_cast<int>(blocks)), dim3(256), 0, stream, x, r, gamma, beta, eps, M, y,
                   gamma2, beta2, y2, add, ylp, yadd, x_row_broadcast);
    CMT_LAUNCH_CHECK("cmt_add_layernorm");
    return CMT_OK;
}

// ---------------------------------------------------------------------------------------------
// Three-term bf16 split of the stacked decoder outputs, the A operand of the task heads' first convolution
// (SeparateTaskHead, cmt_head.py:116-150) on the tensor cores: x = x1 + x2 + x3 with x1 = bf16(x), x2 = bf16(x - x1),
// x3 = bf16(x - x1 - x2) carries all 24 mantissa bits, and the six products x1w1, x1w2, x2w1, x1w3, x2w2, x3w1 of
// cmt_gemm_segmented reproduce the fp32 convolution to ~2^-22 -- these logits feed the top-k, so bf16 alone will not do.
// Fused on the way: torch.nan_to_num of the decoder outputs (cmt_head.py:499) and, for the cooperative heads, the
// element-wise max over the two nodes' stacks (cmt_head_coop.py:383-389).
// in: a (and optionally b) [Z, Nq, 256] fp32; out: [Z, Nq + 2, 768] bf16 = [x1 | x2 | x3] per row, rows 0 and Nq + 1 of
// every z are zero (the k = 3 convolutions over the query axis read them as padding).  One warp per output row.
// node_valid (nullable, with b): [2, frames] per-frame presence of the two nodes; a frame takes max(a, b) with both,
// the present node's rows with one, and zero rows with none.  An absent node's rows are not read.
__device__ __forceinline__ float nan_to_num_f(float x) {
    if (x != x) return 0.0f;
    if (x == __int_as_float(0x7f800000)) return 3.4028234663852886e38f;
    if (x == __int_as_float(0xff800000)) return -3.4028234663852886e38f;
    return x;
}

__global__ void __launch_bounds__(256) split3_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                     __nv_bfloat16* __restrict__ out, float* __restrict__ merged, long long Z, int Nq,
                                                     int frames, long long layer_stride,
                                                     const uint8_t* __restrict__ node_valid) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const long long rows = Z * (Nq + 2);
    for (long long row = blockIdx.x * 8ll + (threadIdx.x >> 5); row < rows; row += gridDim.x * 8ll) {
        const long long z = row / (Nq + 2);
        const int q = static_cast<int>(row - z * (Nq + 2)) - 1;
        uint4* dst = reinterpret_cast<uint4*>(out + row * 768);
        if (q < 0 || q >= Nq) {
            const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
            dst[lane] = zero;
            dst[32 + lane] = zero;
            dst[64 + lane] = zero;
            continue;
        }
        // input row of (layer, frame) = (z / frames, z % frames): layers may be further apart than frames * Nq rows (two
        // nodes' frames stacked in one decoder pass: a = first half of every layer, b = second half)
        const long long frame = z % frames;
        const long long src = ((z / frames) * layer_stride + frame * Nq + q) * 256 + lane * 8;
        const long long dense = (z * Nq + q) * 256 + lane * 8;
        const bool has_a = node_valid == nullptr || node_valid[frame] != 0;
        const bool has_b = b != nullptr && (node_valid == nullptr || node_valid[frames + frame] != 0);
        float v[8] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
        if (has_a) {
            const float4 p0 = *reinterpret_cast<const float4*>(a + src), p1 = *reinterpret_cast<const float4*>(a + src + 4);
            v[0] = p0.x; v[1] = p0.y; v[2] = p0.z; v[3] = p0.w; v[4] = p1.x; v[5] = p1.y; v[6] = p1.z; v[7] = p1.w;
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = nan_to_num_f(v[i]);
        }
        if (has_b) {
            const float4 p0 = *reinterpret_cast<const float4*>(b + src), p1 = *reinterpret_cast<const float4*>(b + src + 4);
            const float w[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = has_a ? fmaxf(v[i], nan_to_num_f(w[i])) : nan_to_num_f(w[i]);
        }
        if (merged != nullptr) {
            *reinterpret_cast<float4*>(merged + dense) = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4*>(merged + dense + 4) = make_float4(v[4], v[5], v[6], v[7]);
        }
        uint32_t t1[4], t2[4], t3[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float x0 = v[2 * i], x1 = v[2 * i + 1];
            t1[i] = pack_bf16x2(x0, x1);
            // a finite fp32 above the largest bf16 (nan_to_num turns inf into 3.4e38) must not round to infinity
            if ((t1[i] & 0x00007f80u) == 0x00007f80u) t1[i] = (t1[i] & 0xffff8000u) | 0x00007f7fu;
            if ((t1[i] & 0x7f800000u) == 0x7f800000u) t1[i] = (t1[i] & 0x8000ffffu) | 0x7f7f0000u;
            const float r0 = x0 - __uint_as_float(t1[i] << 16), r1 = x1 - __uint_as_float(t1[i] & 0xffff0000u);
            t2[i] = pack_bf16x2(r0, r1);
            const float s0 = r0 - __uint_as_float(t2[i] << 16), s1 = r1 - __uint_as_float(t2[i] & 0xffff0000u);
            t3[i] = pack_bf16x2(s0, s1);
        }
        dst[lane] = make_uint4(t1[0], t1[1], t1[2], t1[3]);
        dst[32 + lane] = make_uint4(t2[0], t2[1], t2[2], t2[3]);
        dst[64 + lane] = make_uint4(t3[0], t3[1], t3[2], t3[3]);
    }
}

int launch_split3(const float* a, const float* b, void* out, float* merged, long long Z, int Nq, int C, int frames,
                  long long layer_stride_rows, const uint8_t* node_valid, cudaStream_t stream) {
    CMT_CHECK_ARG(a && out && Z > 0 && Nq > 0, "cmt_split3_bf16: bad arguments");
    CMT_CHECK_ARG(node_valid == nullptr || (b != nullptr && frames > 0),
                  "cmt_split3_bf16: node_valid needs the second stack b and frames > 0");
    if (frames <= 0) {   // dense input [Z, Nq, C]
        frames = 1;
        layer_stride_rows = Nq;
    }
    CMT_CHECK_ARG(Z % frames == 0 && layer_stride_rows >= static_cast<long long>(frames) * Nq, "cmt_split3_bf16: bad layer stride");
    CMT_CHECK_ARG(C == 256, "cmt_split3_bf16: embed dim 256 only (got %d)", C);
    CMT_CHECK_ARG(((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(out) |
                    reinterpret_cast<uintptr_t>(merged)) & 15) == 0, "cmt_split3_bf16: pointers must be 16-byte aligned");
    const long long rows = Z * (Nq + 2);
    long long blocks = (rows + 7) / 8;
    const long long cap = static_cast<long long>(device_sm_count()) * 16;
    if (blocks > cap) blocks = cap;
    launch_pdl(split3_kernel, dim3(static_cast<int>(blocks)), dim3(256), 0, stream, a, b, reinterpret_cast<__nv_bfloat16*>(out), merged, Z, Nq, frames, layer_stride_rows,
               node_valid);
    CMT_LAUNCH_CHECK("cmt_split3_bf16");
    return CMT_OK;
}

// ---------------------------------------------------------------------------------------------
// Task-head tail (SeparateTaskHead, cmt_head.py:116-150 + GroupLayerNorm1d :53-94): after the first grouped conv
// (a per-decoder-layer GEMM, h = conv1(x)), every (layer, query row, output head) needs
//   y = ReLU(LN_64(h) * gamma + beta),   out[o] = sum_t y[q + t - KS/2] . w2[o][t] + b2[o]      (o < c_out <= CMAX)
// with KS = final_kernel (1 in the fusion / camera configs, 3 in the LiDAR ones, where the second convolution mixes
// neighbouring QUERIES and pads the hidden activations with zeros at both ends of a frame's query axis), followed by the
// reference-point decode of the center / height outputs (cmt_head.py:501-513):
//   out = sigmoid(out + ref_logit[row][comp]) * scale + offset.
// Eager torch runs this as ~10 elementwise / reduction passes over the 66 MB h tensor plus an einsum (0.45 ms per
// forward at B = 8) and ~15 more element-wise launches for the decode.  Here one THREAD owns a (layer, row): per output
// head and tap it pulls the 64 hidden values of the (neighbouring) row into registers (sixteen 16-byte loads of 256
// contiguous bytes), takes the statistics and the affine + ReLU in registers, and accumulates the CMAX 64-long dot products
// against w2 held in shared memory (all lanes of a warp read the same weight: broadcast).  No shuffles, fp32 throughout
// (these outputs feed the top-k).  KS = 3 recomputes the LayerNorm of the two neighbours (cheap next to the dots).
constexpr int TH_HC = 64;   // hidden channels per head (head_conv = 64 in every reference config)

struct TaskTailDecode {
    const float* ref_logit;   // [M][3] inverse_sigmoid(reference points) per row, or nullptr: no decode
    const int* comp;          // [NH*CMAX] reference component added before the sigmoid, -1 = plain output
    const float* scale;       // [NH*CMAX]
    const float* offset;      // [NH*CMAX]
};

// Output placement: padded [L, M, NH, CMAX] (packed == 0), or one contiguous [L, M, c_out(head)] tensor per head inside
// `out` (packed == 1): element (l, m, head, o) at off[head] + (l * M + m) * co[head] + o.
struct TaskTailOut {
    long long off[8];
    int co[8];
    int packed;
};

template <int KS, int CT>
__global__ void __launch_bounds__(128) task_head_tail_kernel(const float* __restrict__ h, const float* __restrict__ gamma,
                                                             const float* __restrict__ beta, const float* __restrict__ w2,
                                                             const float* __restrict__ b2, float* __restrict__ out, int M,
                                                             int NH, int CMAX, float eps, int Nq, TaskTailDecode dec,
                                                             TaskTailOut oo) {
    extern __shared__ float th_smem[];
    const int l = blockIdx.y;
    float* w2s = th_smem;                            // [NH][CMAX][KS][64]
    float* gs = w2s + NH * CMAX * KS * TH_HC;        // [NH][64]
    float* bs = gs + NH * TH_HC;                     // [NH][64]
    float* b2s = bs + NH * TH_HC;                    // [NH][CMAX]
    float* dsc = b2s + NH * CMAX;                    // [NH][CMAX] decode scale
    float* dof = dsc + NH * CMAX;                    // [NH][CMAX] decode offset
    int* dcp = reinterpret_cast<int*>(dof + NH * CMAX);   // [NH][CMAX] decode component
    pdl_trigger();
    pdl_wait();
    for (int i = threadIdx.x; i < NH * CMAX * KS * TH_HC; i += blockDim.x)
        w2s[i] = w2[static_cast<long long>(l) * NH * CMAX * KS * TH_HC + i];
    for (int i = threadIdx.x; i < NH * TH_HC; i += blockDim.x) {
        gs[i] = gamma[l * NH * TH_HC + i];
        bs[i] = beta[l * NH * TH_HC + i];
    }
    for (int i = threadIdx.x; i < NH * CMAX; i += blockDim.x) {
        b2s[i] = b2[l * NH * CMAX + i];
        dcp[i] = dec.ref_logit != nullptr ? dec.comp[i] : -1;
        dsc[i] = dec.ref_logit != nullptr ? dec.scale[i] : 1.0f;
        dof[i] = dec.ref_logit != nullptr ? dec.offset[i] : 0.0f;
    }
    __syncthreads();
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < M; m += gridDim.x * blockDim.x) {
        const int q = m % Nq;
        float* orow = out + (static_cast<long long>(l) * M + m) * NH * CMAX;
        float ref[3] = {0.0f, 0.0f, 0.0f};
        if (dec.ref_logit != nullptr) {
            ref[0] = dec.ref_logit[static_cast<long long>(m) * 3];
            ref[1] = dec.ref_logit[static_cast<long long>(m) * 3 + 1];
            ref[2] = dec.ref_logit[static_cast<long long>(m) * 3 + 2];
        }
        for (int hd = 0; hd < NH; ++hd) {
            float acc[CT];
#pragma unroll
            for (int o = 0; o < CT; ++o) acc[o] = 0.0f;
#pragma unroll
            for (int t = 0; t < KS; ++t) {
                const int dq = t - KS / 2;
                if (q + dq < 0 || q + dq >= Nq) continue;   // zero padding of the hidden activations at the frame's ends
                const float4* hrow = reinterpret_cast<const float4*>(h + (static_cast<long long>(l) * M + m + dq) * NH * TH_HC);
                float y[TH_HC];
                float sum = 0.0f;
#pragma unroll
                for (int i = 0; i < TH_HC / 4; ++i) {
                    const float4 v = __ldg(hrow + hd * (TH_HC / 4) + i);
                    y[4 * i] = v.x; y[4 * i + 1] = v.y; y[4 * i + 2] = v.z; y[4 * i + 3] = v.w;
                    sum += (v.x + v.y) + (v.z + v.w);
                }
                const float mu = sum * (1.0f / TH_HC);
                float sq = 0.0f;
#pragma unroll
                for (int c = 0; c < TH_HC; ++c) {
                    y[c] -= mu;
                    sq = fmaf(y[c], y[c], sq);
                }
                const float sd = sqrtf(sq * (1.0f / TH_HC) + eps);
                const float4* g4 = reinterpret_cast<const float4*>(gs + hd * TH_HC);
                const float4* b4 = reinterpret_cast<const float4*>(bs + hd * TH_HC);
#pragma unroll
                for (int i = 0; i < TH_HC / 4; ++i) {
                    const float4 g = g4[i], b = b4[i];
                    y[4 * i] = fmaxf(y[4 * i] / sd * g.x + b.x, 0.0f);
                    y[4 * i + 1] = fmaxf(y[4 * i + 1] / sd * g.y + b.y, 0.0f);
                    y[4 * i + 2] = fmaxf(y[4 * i + 2] / sd * g.z + b.z, 0.0f);
                    y[4 * i + 3] = fmaxf(y[4 * i + 3] / sd * g.w + b.w, 0.0f);
                }
#pragma unroll
                for (int o = 0; o < CT; ++o) {
                    if (o < CMAX) {
                        const float4* w4 = reinterpret_cast<const float4*>(w2s + ((hd * CMAX + o) * KS + t) * TH_HC);
                        float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
#pragma unroll
                        for (int i = 0; i < TH_HC / 4; ++i) {
                            const float4 w = w4[i];
                            a0 = fmaf(y[4 * i], w.x, a0);
                            a1 = fmaf(y[4 * i + 1], w.y, a1);
                            a2 = fmaf(y[4 * i + 2], w.z, a2);
                            a3 = fmaf(y[4 * i + 3], w.w, a3);
                        }
                        acc[o] += (a0 + a1) + (a2 + a3);
                    }
                }
            }
            float* dst = oo.packed ? out + oo.off[hd] + (static_cast<long long>(l) * M + m) * oo.co[hd] : orow + hd * CMAX;
            const int n_out = oo.packed ? oo.co[hd] : CMAX;
#pragma unroll
            for (int o = 0; o < CT; ++o) {
                if (o < n_out) {
                    float v = acc[o] + b2s[hd * CMAX + o];
                    const int comp = dcp[hd * CMAX + o];
                    if (comp >= 0) v = 1.0f / (1.0f + expf(-(v + ref[comp]))) * dsc[hd * CMAX + o] + dof[hd * CMAX + o];
                    dst[o] = v;
                }
            }
        }
    }
}

int launch_task_head_tail(const float* h, const float* gamma, const float* beta, const float* w2, const float* b2, float* out,
                          int L, int M, int NH, int HC, int CMAX, float eps, int ksize, int Nq, const float* ref_logit,
                          const int* dec_comp, const float* dec_scale, const float* dec_offset, const long long* head_off_host,
                          const int* head_cout_host, cudaStream_t stream) {
    CMT_CHECK_ARG(HC == TH_HC, "cmt_task_head_tail: head_conv must be %d (got %d)", TH_HC, HC);
    CMT_CHECK_ARG(L > 0 && M > 0 && NH > 0 && CMAX > 0 && CMAX <= 32, "cmt_task_head_tail: bad shape L=%d M=%d NH=%d CMAX=%d", L, M,
                  NH, CMAX);
    CMT_CHECK_ARG(ksize == 1 || ksize == 3, "cmt_task_head_tail: final_kernel must be 1 or 3 (got %d)", ksize);
    CMT_CHECK_ARG(Nq > 0 && M % Nq == 0, "cmt_task_head_tail: M must be a multiple of Nq");
    CMT_CHECK_ARG(ref_logit == nullptr || (dec_comp && dec_scale && dec_offset), "cmt_task_head_tail: decode tables missing");
    const size_t smem = static_cast<size_t>(NH) * (CMAX * ksize * TH_HC + 2 * TH_HC + 4 * CMAX) * sizeof(float);
    CMT_CHECK_ARG(smem <= 200 * 1024, "cmt_task_head_tail: weights do not fit in shared memory");
    TaskTailDecode dec{ref_logit, dec_comp, dec_scale, dec_offset};
    TaskTailOut oo{};
    if (head_off_host != nullptr) {
        CMT_CHECK_ARG(head_cout_host != nullptr && NH <= 8, "cmt_task_head_tail: per-head output needs head_cout and NH <= 8");
        for (int i = 0; i < NH; ++i) {
            CMT_CHECK_ARG(head_cout_host[i] > 0 && head_cout_host[i] <= CMAX && head_off_host[i] >= 0, "cmt_task_head_tail: bad per-head output table");
            oo.off[i] = head_off_host[i];
            oo.co[i] = head_cout_host[i];
        }
        oo.packed = 1;
    }
    const int bx = (M + 127) / 128;
    auto launch = [&](auto kernel) -> int {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
            if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(task_head_tail)");
        }
        cudaError_t e = launch_pdl(kernel, dim3(bx, L), dim3(128), smem, stream, h, gamma, beta, w2, b2, out, M, NH, CMAX, eps, Nq, dec, oo);
        if (e != cudaSuccess) return cuda_fail(e, "cmt_task_head_tail launch");
        return CMT_OK;
    };
    int rc;
    if (ksize == 1) rc = CMAX <= 16 ? launch(task_head_tail_kernel<1, 16>) : launch(task_head_tail_kernel<1, 32>);
    else rc = CMAX <= 16 ? launch(task_head_tail_kernel<3, 16>) : launch(task_head_tail_kernel<3, 32>);
    if (rc != CMT_OK) return rc;
    CMT_LAUNCH_CHECK("cmt_task_head_tail");
    return CMT_OK;
}

}  // namespace cmt
