// fp32 CUDA-core kernels: the "fp32 verification mode" of the projection GEMM and of the
// cross-attention (north star: decoder outputs within rel-L2 <= 1e-4 of the reference's fp32
// path).  Same operand layouts and output addressing as the tcgen05 kernels, so the two
// implementations can be compared against each other on the GPU.  Correctness mode, not a
// performance mode.
#include "kernels.cuh"

namespace cmt {

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename TIn>
__global__ void __launch_bounds__(256) simt_gemm_kernel(GemmArgs g) {
    __shared__ float As[16][65];
    __shared__ float Bs[16][65];
    const int z = blockIdx.z;
    const TIn* A = reinterpret_cast<const TIn*>(g.A) + z * g.strideA;
    const TIn* B = reinterpret_cast<const TIn*>(g.B) + z * g.strideB;
    const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < g.K; k0 += 16) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = threadIdx.x + i * 256;
            const int row = idx >> 4, kk = idx & 15;
            const int k = k0 + kk;
            const int m = m0 + row, n = n0 + row;
            As[kk][row] = (m < g.M && k < g.K) ? to_f32<TIn>(A[static_cast<long long>(m) * g.lda + k]) : 0.0f;
            Bs[kk][row] = (n < g.N && k < g.K) ? to_f32<TIn>(B[static_cast<long long>(n) * g.ldb + k]) : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= g.M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= g.N) continue;
            float v = acc[i][j];
            if (g.bias) v += g.bias_per_row ? g.bias[m] : g.bias[n];
            v *= g.alpha;
            if (g.relu) v = fmaxf(v, 0.0f);
            const long long off = z * g.strideC + (n / g.cb) * g.cb_stride +
                                  static_cast<long long>(m) * g.ldc + (n % g.cb);
            if (g.out_16)
                reinterpret_cast<__nv_bfloat16*>(g.C)[off] = __float2bfloat16_rn(v);
            else
                reinterpret_cast<float*>(g.C)[off] = v;
        }
    }
}

int launch_simt_gemm(const GemmArgs& g, int batch, int in_dtype, cudaStream_t stream) {
    dim3 grid((g.N + 63) / 64, (g.M + 63) / 64, batch);
    CMT_CHECK_ARG(grid.y <= 65535 && grid.z <= 65535, "cmt_gemm_bias_act(simt): grid too large");
    if (in_dtype == CMT_BF16)
        simt_gemm_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(g);
    else
        simt_gemm_kernel<float><<<grid, 256, 0, stream>>>(g);
    CMT_LAUNCH_CHECK("cmt_gemm_bias_act(simt)");
    return CMT_OK;
}

// ---------------------------------------------------------------------------
// One thread = one query row of one head; block = 128 rows; K/V^T tiles of 64 tokens in smem.
template <typename TIn>
__global__ void __launch_bounds__(128) simt_attn_kernel(AttnArgs a) {
    __shared__ float Ks[64][32];
    __shared__ float Vs[32][65];
    const int b = blockIdx.z, h = blockIdx.y;
    const int row = blockIdx.x * 128 + threadIdx.x;
    const bool row_ok = row < a.Nq;
    const TIn* Q = reinterpret_cast<const TIn*>(a.q);
    const TIn* K = reinterpret_cast<const TIn*>(a.k) + b * a.k_bstride + h * a.k_hstride;
    const TIn* Vt = reinterpret_cast<const TIn*>(a.vt) + b * a.v_bstride + h * a.v_hstride;
    float q[32], o[32];
#pragma unroll
    for (int d = 0; d < 32; ++d) {
        q[d] = row_ok ? to_f32<TIn>(Q[(static_cast<long long>(b) * a.Nq + row) * a.q_ld + h * 32 + d]) : 0.0f;
        o[d] = 0.0f;
    }
    float m = -INFINITY, l = 0.0f;
    for (int t0 = a.kv_begin; t0 < a.kv_end; t0 += 64) {
        __syncthreads();
        for (int idx = threadIdx.x; idx < 64 * 32; idx += 128) {
            const int t = idx >> 5, d = idx & 31;
            Ks[t][d] = (t0 + t < a.kv_end) ? to_f32<TIn>(K[static_cast<long long>(t0 + t) * 32 + d]) : 0.0f;
        }
        for (int idx = threadIdx.x; idx < 32 * 64; idx += 128) {
            const int d = idx >> 6, t = idx & 63;
            Vs[d][t] = (t0 + t < a.kv_end) ? to_f32<TIn>(Vt[static_cast<long long>(d) * a.v_ld + t0 + t]) : 0.0f;
        }
        __syncthreads();
        const int nt = min(64, a.kv_end - t0);
        for (int c0 = 0; c0 < nt; c0 += 16) {
            float s[16];
            float cmax = -INFINITY;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                float acc = 0.0f;
#pragma unroll
                for (int d = 0; d < 32; ++d) acc = fmaf(q[d], Ks[c0 + i][d], acc);
                const bool keep = c0 + i < nt && (a.key_keep == nullptr ||
                                                  a.key_keep[static_cast<long long>(b) * a.N_kv + t0 + c0 + i] != 0);
                s[i] = keep ? acc : -INFINITY;
                cmax = fmaxf(cmax, s[i]);
            }
            if (cmax == -INFINITY) continue;   // every key of the chunk is padding
            const float m_new = fmaxf(m, cmax);
            const float alpha = (m == -INFINITY) ? 0.0f : exp2f(m - m_new);
            l *= alpha;
#pragma unroll
            for (int d = 0; d < 32; ++d) o[d] *= alpha;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float p = (s[i] == -INFINITY) ? 0.0f : exp2f(s[i] - m_new);
                l += p;
#pragma unroll
                for (int d = 0; d < 32; ++d) o[d] = fmaf(p, Vs[d][c0 + i], o[d]);
            }
            m = m_new;
        }
    }
    if (!row_ok) return;
    const float inv = l > 0.0f ? 1.0f / l : 0.0f;
    const long long obase = (static_cast<long long>(b) * a.Nq + row) * (a.H * 32) + h * 32;
#pragma unroll
    for (int d = 0; d < 32; ++d) {
        const float v = o[d] * inv;
        if (a.o_dtype == CMT_BF16)
            reinterpret_cast<__nv_bfloat16*>(a.o)[obase + d] = __float2bfloat16_rn(v);
        else
            reinterpret_cast<float*>(a.o)[obase + d] = v;
    }
    if (a.lse)
        a.lse[(static_cast<long long>(b) * a.H + h) * a.Nq + row] =
            (l > 0.0f) ? (m + log2f(l)) * 0.6931471805599453f : -INFINITY;
}

int launch_simt_attn(const AttnArgs& a, int dtype, cudaStream_t stream) {
    dim3 grid((a.Nq + 127) / 128, a.H, a.B);
    CMT_CHECK_ARG(grid.z <= 65535, "cmt_cross_attn_fwd(simt): batch too large");
    if (dtype == CMT_BF16)
        simt_attn_kernel<__nv_bfloat16><<<grid, 128, 0, stream>>>(a);
    else
        simt_attn_kernel<float><<<grid, 128, 0, stream>>>(a);
    CMT_LAUNCH_CHECK("cmt_cross_attn_fwd(simt)");
    return CMT_OK;
}

}  // namespace cmt
