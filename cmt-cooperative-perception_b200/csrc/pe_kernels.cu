// Position-encoding kernels: camera-ray lift (K1), reference-point re-projection (K1b),
// masked view sum, sine/cosine BEV embedding.  All HBM/launch bound, fp32 math on CUDA cores.
//
// Reference arithmetic followed here (never copied):
//   K1   : projects/mmdet3d_plugin/models/dense_heads/cmt_head.py:417-432
//   K1b  : cmt_head.py:439-464
//   sum  : cmt_head.py:466
//   sincos: cmt_head.py:40-50
#include "kernels.cuh"

namespace cmt {

struct RayPeParams {
    float pc_min[3];
    float pc_rng[3];
    float pc_inv[3];       // float(1 / pc_rng) for the 3-instruction correctly rounded division
    float depth_step_num;  // (pc_range[3] - 1)
    float pad_h, pad_w;
    int n_cam, H, W, D;
};

// Correctly rounded a / b for normal operands given inv = float(1 / b): one residual correction of the
// reciprocal product (3 instructions instead of the ~15 of the generic IEEE division sequence).
__device__ __forceinline__ float div_by_const(float a, float b, float inv) {
    const float q = a * inv;
    const float r = fmaf(-q, b, a);
    return fmaf(r, inv, q);
}

// One block = one feature-map row of one camera (W pixels x D*3 features, contiguous in the output);
// one thread-item = 8 consecutive depth bins x 3 coordinates = 24 consecutive features of one pixel
// (48 bytes bf16 / 96 bytes fp32, written as 16-byte vectors; a warp covers 1536 / 3072 contiguous bytes).
// With that unit every index is a compile-time constant: the camera matrix and pc_range constants sit in
// registers, depth bins and pixel abscissae come from two small shared-memory tables (filled with true
// divisions once per block), and the normalising division is a 3-instruction correctly rounded sequence.
// ~9 instructions per output value, so the kernel is bound by the HBM write instead of by issue.
// kBins = depth bins per thread-item: 16 (D % 16 == 0: 96 bytes of bf16 = three 256-bit stores, every store instruction
// writes whole 32-byte sectors) or 8 (48 bytes = three 128-bit stores at a 48-byte lane stride: half-filled sectors).
// kOut: output dtype, CMT_F32 | CMT_BF16 | CMT_F16 (the 16-bit forms differ only in the rounding).
template <int kOut, int kBins>
__global__ void __launch_bounds__(256) ray_pe_kernel(const float* __restrict__ img2lidar,
                                                     void* __restrict__ out, RayPeParams p) {
    extern __shared__ float sm[];
    float* dtab = sm;            // [D]   coords_d = 1 + arange(D) * (pc_range[3] - 1) / D      (cmt_head.py:422)
    float* utab = sm + p.D;      // [W]   coords_w = arange(W) * pad_w / W                      (cmt_head.py:421)
    const int cam = blockIdx.x / p.H;
    const int i = blockIdx.x - cam * p.H;
    for (int k = threadIdx.x; k < p.D; k += blockDim.x)
        dtab[k] = 1.0f + (static_cast<float>(k) * p.depth_step_num) / static_cast<float>(p.D);
    for (int j = threadIdx.x; j < p.W; j += blockDim.x)
        utab[j] = (static_cast<float>(j) * p.pad_w) / static_cast<float>(p.W);
    float M[3][4];               // rows 0..2 of float32(inv(lidar2img))                          (cmt_head.py:428-429)
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int o = 0; o < 4; ++o) M[c][o] = __ldg(img2lidar + cam * 16 + c * 4 + o);
    __syncthreads();
    const float v = (static_cast<float>(i) * p.pad_h) / static_cast<float>(p.H);  // coords_h (cmt_head.py:420)
    const int units = p.D / kBins;  // kBins-bin units per pixel
    const int items = p.W * units;
    const long long row_base = static_cast<long long>(blockIdx.x) * items;
    constexpr int NV = kBins * 3;   // values per item
    for (int tl = threadIdx.x; tl < items; tl += blockDim.x) {
        const int j = tl / units;
        const int k0 = (tl - j * units) * kBins;
        const float u = utab[j];
        float vals[NV];
#pragma unroll
        for (int kk = 0; kk < kBins; ++kk) {
            const float d = dtab[k0 + kk];
            const float x0 = u * d, x1 = v * d;  // coords[..., :2] *= coords[..., 2:3]   (cmt_head.py:426)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float acc = x0 * M[c][0];
                acc = fmaf(x1, M[c][1], acc);
                acc = fmaf(d, M[c][2], acc);
                acc = acc + M[c][3];
                vals[kk * 3 + c] = div_by_const(acc - p.pc_min[c], p.pc_rng[c], p.pc_inv[c]);  // (:431-432)
            }
        }
        const long long t = row_base + tl;  // in NV-feature units
        if (kOut != CMT_F32) {
            if (kBins == 16) {
                uint8_t* o = reinterpret_cast<uint8_t*>(out) + t * (NV * 2);
#pragma unroll
                for (int q = 0; q < 3; ++q)
                    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(o + 32 * q),
                                 "r"(pack_lp2<kOut>(vals[16 * q + 0], vals[16 * q + 1])), "r"(pack_lp2<kOut>(vals[16 * q + 2], vals[16 * q + 3])),
                                 "r"(pack_lp2<kOut>(vals[16 * q + 4], vals[16 * q + 5])), "r"(pack_lp2<kOut>(vals[16 * q + 6], vals[16 * q + 7])),
                                 "r"(pack_lp2<kOut>(vals[16 * q + 8], vals[16 * q + 9])), "r"(pack_lp2<kOut>(vals[16 * q + 10], vals[16 * q + 11])),
                                 "r"(pack_lp2<kOut>(vals[16 * q + 12], vals[16 * q + 13])), "r"(pack_lp2<kOut>(vals[16 * q + 14], vals[16 * q + 15]))
                                 : "memory");
            } else {
                uint4* o = reinterpret_cast<uint4*>(out) + 3 * t;
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    uint4 w;
                    w.x = pack_lp2<kOut>(vals[8 * q + 0], vals[8 * q + 1]);
                    w.y = pack_lp2<kOut>(vals[8 * q + 2], vals[8 * q + 3]);
                    w.z = pack_lp2<kOut>(vals[8 * q + 4], vals[8 * q + 5]);
                    w.w = pack_lp2<kOut>(vals[8 * q + 6], vals[8 * q + 7]);
                    o[q] = w;
                }
            }
        } else {
            float4* o = reinterpret_cast<float4*>(out) + (NV / 4) * t;
#pragma unroll
            for (int q = 0; q < NV / 4; ++q) o[q] = make_float4(vals[4 * q], vals[4 * q + 1], vals[4 * q + 2], vals[4 * q + 3]);
        }
    }
}

struct RayQueryParams {
    float pc_min[3];
    float pc_rng[3];
    float depth_step_num;
    float pad_h, pad_w;
    int B, V, Nq, D;
};

template <int kOut>
__global__ void __launch_bounds__(256) ray_query_pe_kernel(const float* __restrict__ ref,
                                                           const float* __restrict__ l2i,
                                                           const float* __restrict__ i2l,
                                                           void* __restrict__ out,
                                                           float* __restrict__ mask,
                                                           RayQueryParams p) {
    const int feats = p.D * 3;
    const int groups = feats >> 3;
    const long long total = static_cast<long long>(p.B) * p.V * p.Nq * groups;
    for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int g = static_cast<int>(t % groups);
        const long long pt = t / groups;  // (b, v, n)
        const int n = static_cast<int>(pt % p.Nq);
        const int v = static_cast<int>((pt / p.Nq) % p.V);
        const int b = static_cast<int>(pt / (static_cast<long long>(p.Nq) * p.V));
        const float* r3 = ref + (static_cast<long long>(b) * p.Nq + n) * 3;
        // ref * (max - min) + min                                                (cmt_head.py:446)
        const float P0 = r3[0] * p.pc_rng[0] + p.pc_min[0];
        const float P1 = r3[1] * p.pc_rng[1] + p.pc_min[1];
        const float P2 = r3[2] * p.pc_rng[2] + p.pc_min[2];
        const float* L = l2i + (static_cast<long long>(b) * p.V + v) * 16;
        float s[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float acc = P0 * L[c * 4 + 0];
            acc = fmaf(P1, L[c * 4 + 1], acc);
            acc = fmaf(P2, L[c * 4 + 2], acc);
            s[c] = acc + L[c * 4 + 3];
        }
        const bool zpos = s[2] > 0.0f;
        const float den = zpos ? (s[2] + 1e-6f) : (s[2] - 1e-6f);  // (:450-451)
        const float px = s[0] / den, py = s[1] / den, pz = s[2] / den;
        const bool inside = (px < p.pad_w) && (px >= 0.0f) && (py < p.pad_h) && (py >= 0.0f) && zpos;
        if (g == 0) mask[pt] = inside ? 1.0f : 0.0f;
        const float* M = i2l + (static_cast<long long>(b) * p.V + v) * 16;
        // A point outside the view enters the view sum as emb * 0 (cmt_head.py:466) whatever its features, so they are
        // written as zeros.  Their true values are unbounded: near the camera plane (s[2] -> 0) px and py reach ~1e8
        // and the lifted coordinates overflow fp16 to inf, which the rv-PE MLP turns into NaN and the view sum into
        // NaN * 0.
        float vals[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int f = g * 8 + e;
            const int k = f / 3;
            const int c = f - 3 * k;
            const float d = 1.0f + (static_cast<float>(k) * p.depth_step_num) / static_cast<float>(p.D);
            const float* r = M + c * 4;
            float acc = (px * d) * r[0];
            acc = fmaf(py * d, r[1], acc);
            acc = fmaf(pz * d, r[2], acc);
            acc = acc + r[3];
            vals[e] = inside ? (acc - p.pc_min[c]) / p.pc_rng[c] : 0.0f;
        }
        if (kOut != CMT_F32) {
            uint4 w;
            w.x = pack_lp2<kOut>(vals[0], vals[1]);
            w.y = pack_lp2<kOut>(vals[2], vals[3]);
            w.z = pack_lp2<kOut>(vals[4], vals[5]);
            w.w = pack_lp2<kOut>(vals[6], vals[7]);
            reinterpret_cast<uint4*>(out)[t] = w;
        } else {
            float4* o = reinterpret_cast<float4*>(out) + 2 * t;
            o[0] = make_float4(vals[0], vals[1], vals[2], vals[3]);
            o[1] = make_float4(vals[4], vals[5], vals[6], vals[7]);
        }
    }
}

template <int kIn>
__global__ void __launch_bounds__(256) masked_view_sum_kernel(const void* __restrict__ emb,
                                                              const float* __restrict__ mask,
                                                              const float* __restrict__ base, long long base_bstride,
                                                              float* __restrict__ out, int B, int V,
                                                              int Nq, int C, const uint8_t* __restrict__ view_valid) {
    const long long total = static_cast<long long>(B) * Nq * C;
    for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int c = static_cast<int>(t % C);
        const int n = static_cast<int>((t / C) % Nq);
        const int b = static_cast<int>(t / (static_cast<long long>(C) * Nq));
        float acc = 0.0f;
        for (int v = 0; v < V; ++v) {
            // an absent camera is skipped, not weighted by zero: its embedding may be NaN (garbage calibration)
            if (view_valid != nullptr && view_valid[static_cast<long long>(v) * B + b] == 0) continue;
            const long long row = (static_cast<long long>(b) * V + v) * Nq + n;
            const float m = mask[row];
            float e;
            if (kIn != CMT_F32)
                e = load_lp<kIn>(emb, row * C + c);
            else
                e = reinterpret_cast<const float*>(emb)[row * C + c];
            acc += e * m;
        }
        // query_embeds = bev_query_embeds + rv_query_embeds (cmt_head.py:492): the view sum first, then the BEV part
        if (base != nullptr) acc = base[static_cast<long long>(b) * base_bstride + static_cast<long long>(n) * C + c] + acc;
        out[t] = acc;
    }
}

template <int kOut>
__global__ void __launch_bounds__(256) pos2embed_kernel(const float* __restrict__ pos,
                                                        void* __restrict__ out, int N,
                                                        int pos_stride, int F) {
    const long long total = static_cast<long long>(N) * 2 * F;
    const float scale = 6.283185307179586f;  // 2*pi rounded to fp32, as `pos * scale` does
    for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
         t += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int f2 = static_cast<int>(t % (2 * F));
        const long long n = t / (2 * F);
        const bool is_x = f2 >= F;  // cat((pos_y, pos_x))                        (cmt_head.py:49)
        const int m = is_x ? f2 - F : f2;
        const float pv = pos[n * pos_stride + (is_x ? 0 : 1)] * scale;
        // dim_t = 2 * (m // 2) / F + 1  (the `temperature` argument is unused, cmt_head.py:43-44)
        const float dim_t = (2.0f * static_cast<float>(m / 2)) / static_cast<float>(F) + 1.0f;
        const float a = pv / dim_t;
        const float r = (m & 1) ? cosf(a) : sinf(a);
        if (kOut != CMT_F32)
            store_lp<kOut>(out, t, r);
        else
            reinterpret_cast<float*>(out)[t] = r;
    }
}

static int grid_for(long long total_threads, int block) {
    const int sms = device_sm_count();
    long long blocks = (total_threads + block - 1) / block;
    const long long cap = static_cast<long long>(sms) * 16;  // multiple of the SM count
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return static_cast<int>(blocks);
}

int launch_ray_pe(const float* img2lidar, void* out, int n_cam, int H, int W, int D, float pad_h,
                  float pad_w, const float* pc, int out_dtype, cudaStream_t stream) {
    CMT_CHECK_ARG(img2lidar && out && pc, "cmt_ray_pe: null pointer");
    CMT_CHECK_ARG(n_cam > 0 && H > 0 && W > 0 && D > 0, "cmt_ray_pe: bad shape");
    CMT_CHECK_ARG(D % 8 == 0, "cmt_ray_pe: depth_num must be a multiple of 8 (got D=%d)", D);
    CMT_CHECK_ARG(out_dtype == CMT_F32 || out_dtype == CMT_BF16 || out_dtype == CMT_F16, "cmt_ray_pe: bad dtype");
    RayPeParams p{};
    for (int c = 0; c < 3; ++c) {
        p.pc_min[c] = pc[c];
        p.pc_rng[c] = pc[c + 3] - pc[c];
        p.pc_inv[c] = static_cast<float>(1.0 / static_cast<double>(p.pc_rng[c]));
    }
    p.depth_step_num = pc[3] - 1.0f;
    p.pad_h = pad_h;
    p.pad_w = pad_w;
    p.n_cam = n_cam;
    p.H = H;
    p.W = W;
    p.D = D;
    const long long blocks = static_cast<long long>(n_cam) * H;
    CMT_CHECK_ARG(blocks < (1ll << 31), "cmt_ray_pe: too many feature rows");
    const int grid = static_cast<int>(blocks);
    const size_t smem = static_cast<size_t>(D + W) * sizeof(float);
    CMT_CHECK_ARG(smem <= 48 * 1024, "cmt_ray_pe: W + D too large");
    const bool wide = D % 16 == 0 && (reinterpret_cast<uintptr_t>(out) & 31) == 0;
    if (out_dtype == CMT_BF16 && wide)
        ray_pe_kernel<CMT_BF16, 16><<<grid, 256, smem, stream>>>(img2lidar, out, p);
    else if (out_dtype == CMT_BF16)
        ray_pe_kernel<CMT_BF16, 8><<<grid, 256, smem, stream>>>(img2lidar, out, p);
    else if (out_dtype == CMT_F16 && wide)
        ray_pe_kernel<CMT_F16, 16><<<grid, 256, smem, stream>>>(img2lidar, out, p);
    else if (out_dtype == CMT_F16)
        ray_pe_kernel<CMT_F16, 8><<<grid, 256, smem, stream>>>(img2lidar, out, p);
    else
        ray_pe_kernel<CMT_F32, 8><<<grid, 256, smem, stream>>>(img2lidar, out, p);
    CMT_LAUNCH_CHECK("cmt_ray_pe");
    return CMT_OK;
}

int launch_ray_query_pe(const float* ref, const float* l2i, const float* i2l, void* out,
                        float* mask, int B, int V, int Nq, int D, float pad_h, float pad_w,
                        const float* pc, int out_dtype, cudaStream_t stream) {
    CMT_CHECK_ARG(ref && l2i && i2l && out && mask && pc, "cmt_ray_query_pe: null pointer");
    CMT_CHECK_ARG(B > 0 && V > 0 && Nq > 0 && D > 0, "cmt_ray_query_pe: bad shape");
    CMT_CHECK_ARG((D * 3) % 8 == 0, "cmt_ray_query_pe: depth_num*3 must be a multiple of 8");
    CMT_CHECK_ARG(out_dtype == CMT_F32 || out_dtype == CMT_BF16 || out_dtype == CMT_F16, "cmt_ray_query_pe: bad dtype");
    RayQueryParams p{};
    for (int c = 0; c < 3; ++c) {
        p.pc_min[c] = pc[c];
        p.pc_rng[c] = pc[c + 3] - pc[c];
    }
    p.depth_step_num = pc[3] - 1.0f;
    p.pad_h = pad_h;
    p.pad_w = pad_w;
    p.B = B;
    p.V = V;
    p.Nq = Nq;
    p.D = D;
    const long long total = static_cast<long long>(B) * V * Nq * (D * 3 / 8);
    const int grid = grid_for(total, 256);
    if (out_dtype == CMT_BF16)
        ray_query_pe_kernel<CMT_BF16><<<grid, 256, 0, stream>>>(ref, l2i, i2l, out, mask, p);
    else if (out_dtype == CMT_F16)
        ray_query_pe_kernel<CMT_F16><<<grid, 256, 0, stream>>>(ref, l2i, i2l, out, mask, p);
    else
        ray_query_pe_kernel<CMT_F32><<<grid, 256, 0, stream>>>(ref, l2i, i2l, out, mask, p);
    CMT_LAUNCH_CHECK("cmt_ray_query_pe");
    return CMT_OK;
}

int launch_masked_view_sum(const void* emb, const float* mask, const float* base, long long base_bstride, float* out, int B,
                           int V, int Nq, int C, int emb_dtype, const uint8_t* view_valid, cudaStream_t stream) {
    CMT_CHECK_ARG(emb && mask && out, "cmt_masked_view_sum: null pointer");
    CMT_CHECK_ARG(B > 0 && V > 0 && Nq > 0 && C > 0, "cmt_masked_view_sum: bad shape");
    const long long total = static_cast<long long>(B) * Nq * C;
    const int grid = grid_for(total, 256);
    if (emb_dtype == CMT_BF16)
        masked_view_sum_kernel<CMT_BF16><<<grid, 256, 0, stream>>>(emb, mask, base, base_bstride, out, B, V, Nq, C, view_valid);
    else if (emb_dtype == CMT_F16)
        masked_view_sum_kernel<CMT_F16><<<grid, 256, 0, stream>>>(emb, mask, base, base_bstride, out, B, V, Nq, C, view_valid);
    else if (emb_dtype == CMT_F32)
        masked_view_sum_kernel<CMT_F32><<<grid, 256, 0, stream>>>(emb, mask, base, base_bstride, out, B, V, Nq, C, view_valid);
    else
        CMT_CHECK_ARG(false, "cmt_masked_view_sum: bad dtype");
    CMT_LAUNCH_CHECK("cmt_masked_view_sum");
    return CMT_OK;
}

int launch_pos2embed(const float* pos, void* out, int N, int pos_stride, int F, int out_dtype,
                     cudaStream_t stream) {
    CMT_CHECK_ARG(pos && out, "cmt_pos2embed: null pointer");
    CMT_CHECK_ARG(N > 0 && F > 0 && pos_stride >= 2, "cmt_pos2embed: bad shape");
    const long long total = static_cast<long long>(N) * 2 * F;
    const int grid = grid_for(total, 256);
    if (out_dtype == CMT_BF16)
        pos2embed_kernel<CMT_BF16><<<grid, 256, 0, stream>>>(pos, out, N, pos_stride, F);
    else if (out_dtype == CMT_F16)
        pos2embed_kernel<CMT_F16><<<grid, 256, 0, stream>>>(pos, out, N, pos_stride, F);
    else if (out_dtype == CMT_F32)
        pos2embed_kernel<CMT_F32><<<grid, 256, 0, stream>>>(pos, out, N, pos_stride, F);
    else
        CMT_CHECK_ARG(false, "cmt_pos2embed: bad dtype");
    CMT_LAUNCH_CHECK("cmt_pos2embed");
    return CMT_OK;
}

}  // namespace cmt
