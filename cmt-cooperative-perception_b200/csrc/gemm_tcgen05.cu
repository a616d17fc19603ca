// K2: projection / MLP GEMM on the 5th-gen tensor cores.
//
//   C = act((A * B^T + bias) * alpha),  A:[M,K] bf16, B:[N,K] bf16 (both K-major), fp32 accumulate.
//
// Persistent, warp-specialised kernel, one CTA per SM:
//   warp 0      TMA producer  : 3-D tensor maps (K, rows, batch), 128B swizzle.  Streaming mode: 4-stage ring of
//                               A+B k-blocks.  B-resident mode (K <= 256, B not batched): the CTA's n-tile of B is
//                               loaded once, the ring carries A only (5 stages).
//   warp 1      MMA issuer    : one elected thread, tcgen05.mma cta_group::1 kind::f16,
//                               M=128 x N=256 x K=16 per instruction, accumulator in TMEM
//   warp 2      TMEM allocator (512 columns = two 128x256 fp32 accumulators, ping-pong)
//   warps 4..11 epilogue      : tcgen05.ld 32x32b -> bias (cached in shared memory) / alpha / ReLU -> bf16|fp32 ->
//                               256-bit global stores straight from registers (a thread owns 32 consecutive
//                               columns of one row: 64 / 128 contiguous bytes), overlapped with the next tile's
//                               main loop.  No shared-memory staging: the MMAs already read 96 of the 128 B/clk.
//
// Replaces F.linear in models/utils/attention.py:21-27,138 and the PE MLPs of
// models/dense_heads/cmt_head.py:292-301 (reference runs them as fp32 cuBLAS SGEMMs).
#include <cstdlib>
#include "kernels.cuh"

namespace cmt {

namespace gemm {
constexpr int BM = 128, BN = 256, BK = 64;
constexpr int A_BYTES = BM * BK * 2;  // 16 KB
constexpr int B_BYTES = BN * BK * 2;  // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
// B-resident mode (K <= 256, B shared by the batch): a CTA keeps ONE n-tile of B (all of K) in shared memory for its
// whole life and streams only A tiles through the ring.  A 128x256 tile with K = 256 otherwise pulls 192 KB through
// the TMA for 16.8 MFLOP (87 flop/B); with B resident a tile loads 64 KB (262 flop/B) and the n-tiles of one
// m-tile run on neighbouring CTAs at the same time, so A comes from DRAM once and from L2 the other n_tiles - 1 times.
constexpr int RES_KB = 4;                       // K blocks the resident B can hold (K <= 256)
constexpr int B_RES_BYTES = RES_KB * B_BYTES;   // 128 KB
constexpr int STREAM_STAGES = 4;   // streaming mode: 4 x (A 16 KB + B 32 KB)
constexpr int RES_STAGES = 5;      // B-resident mode: A-only stages of 16 KB after the 128 KB of B
constexpr int MAX_STAGES = STREAM_STAGES > RES_STAGES ? STREAM_STAGES : RES_STAGES;
constexpr int RING_BYTES = (STREAM_STAGES * STAGE_BYTES > B_RES_BYTES + RES_STAGES * A_BYTES)
                               ? STREAM_STAGES * STAGE_BYTES : B_RES_BYTES + RES_STAGES * A_BYTES;
// column bias cached in shared memory (the K/V projections have N = 1536): the epilogue's bias fetch becomes a
// broadcast LDS instead of a ~500-cycle global load sitting between the TMEM load and the stores of a round
constexpr int BIAS_CAP = 2048;
constexpr int SMEM_BYTES = RING_BYTES + BIAS_CAP * 4 + 1024 /*align slack*/ + 256 /*barriers*/;
static_assert(SMEM_BYTES <= 232448, "shared memory budget");
constexpr int THREADS = 384;  // 4 control warps + 8 epilogue warps
// The producer and accumulator hand-over waits use mbar_wait_sleep: they sleep in hardware and leave the issue slots
// to the epilogue.
}  // namespace gemm

constexpr int MAX_SEG = 18;

struct TcGemmParams {
    const float* bias;
    void* C;
    int M, N, K;
    long long ldc, cb, cb_stride, strideC;
    float alpha;
    int relu, bias_per_row, out_bf16;
    int a_batched, b_batched;
    int m_tiles, n_tiles, total_tiles, num_kb;
    int direct;     // 1: lean epilogue, 256-bit stores straight from registers (alignment / bias conditions hold)
    float* norm2_max; // [batch][N/32]: atomicMax of the squared norm of every row's 32-column block (attention score bound), or nullptr
    int transpose_c; // 1: element (m, n) of batch z is stored at z*strideC + (n / cb)*cb_stride + (n % cb)*ldc + m (bf16)
    int b_resident; // 1: gridDim.x = Gm * n_tiles, CTA c owns n-tile c % n_tiles and the (batch, m-tile) pairs c / n_tiles + i * Gm
    // Segmented K (implicit convolutions and split-precision products): K block kb belongs to segment s = kb / kb_per_seg;
    // its A tile is read at column seg_acol[s] + (kb % kb_per_seg) * BK and at row m0 + a_row_off + seg_shift[s] of the
    // batch's A matrix (rows outside it are zero-filled by the TMA unit), while B is read at column kb * BK as usual.
    // n_seg == 0: ordinary GEMM.
    int n_seg, kb_per_seg, a_row_off;
    int seg_acol[MAX_SEG], seg_shift[MAX_SEG];
    int b_batch_div;   // batch z reads B of batch z / b_batch_div (task heads: one weight set per decoder layer, B frames each)
    // Token epilogue of the 3x3 shared_conv (conv_xv != nullptr): output row m is position (y, x) = (m / conv_Wp, m % conv_Wp)
    // of the zero-padded map of frame z; interior positions become token t = (y - 1) * conv_W + (x - 1) and are stored as
    // xv[z][t - tok_begin] = bf16(v), xk[z][t - tok_begin] = bf16(v + pos[t]) (v = ReLU(acc + bias)); border rows are dropped.
    void* conv_xk;
    void* conv_xv;
    const float* conv_pos;
    int conv_W, conv_H, conv_Wp, conv_tok_begin, conv_tok_end;
    long long conv_frame_stride;   // elements between frames in xk / xv
    int mt_off;                    // first m-tile (conv with a token sub-range computes only the rows that hold its tokens)
};

// The three roles walk the same tile sequence.
struct TileWalk {
    int cur, step, end, nt_fixed;
    __device__ __forceinline__ TileWalk(const TcGemmParams& p) {
        if (p.b_resident) {
            step = gridDim.x / p.n_tiles;
            cur = blockIdx.x / p.n_tiles;
            nt_fixed = blockIdx.x - cur * p.n_tiles;
            end = p.total_tiles / p.n_tiles;   // batch * m_tiles
        } else {
            step = gridDim.x;
            cur = blockIdx.x;
            nt_fixed = -1;
            end = p.total_tiles;
        }
    }
    __device__ __forceinline__ bool valid() const { return cur < end; }
    __device__ __forceinline__ void next() { cur += step; }
    __device__ __forceinline__ void decode(const TcGemmParams& p, int& z, int& mt, int& nt) const {
        if (nt_fixed >= 0) {
            z = cur / p.m_tiles;
            mt = cur - z * p.m_tiles;
            nt = nt_fixed;
        } else {
            const int tiles_per_batch = p.m_tiles * p.n_tiles;
            z = cur / tiles_per_batch;
            const int r = cur - z * tiles_per_batch;
            mt = r / p.n_tiles;
            nt = r - mt * p.n_tiles;
        }
        mt += p.mt_off;
    }
};

__global__ void __launch_bounds__(gemm::THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
               const TcGemmParams p) {
    using namespace gemm;
    pdl_trigger();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    float* bias_s = reinterpret_cast<float*>(smem + RING_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + RING_BYTES + BIAS_CAP * 4);
    uint64_t* full_bar = bars;                   // [MAX_STAGES]
    uint64_t* empty_bar = bars + MAX_STAGES;     // [MAX_STAGES]
    uint64_t* tmem_full = bars + 2 * MAX_STAGES;     // [2]
    uint64_t* tmem_empty = bars + 2 * MAX_STAGES + 2;  // [2]
    uint64_t* bres_full = bars + 2 * MAX_STAGES + 4;   // resident B landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 5);
    const int n_stages = p.b_resident ? RES_STAGES : STREAM_STAGES;
    // ring geometry: streaming = 4 x (A 16 KB + B 32 KB); B-resident = B (128 KB) then RES_STAGES x A 16 KB
    uint8_t* ring = p.b_resident ? smem + B_RES_BYTES : smem;
    const int ring_stride = p.b_resident ? A_BYTES : STAGE_BYTES;

    // warp index / TMEM base through shuffles: provably warp-uniform, so the producer and issuer warps keep
    // their descriptors in uniform registers and TMA / tcgen05.mma instructions issue back to back (a divergent
    // `lane == 0` role costs a ~12-instruction ELECT/R2UR waterfall per instruction).
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tma_a);
        tma_prefetch_desc(&tma_b);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < MAX_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&tmem_full[s], 1);
            mbar_init(&tmem_empty[s], 8);  // one arrival per epilogue warp
        }
        mbar_init(bres_full, 1);
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    const bool bias_cached = p.bias != nullptr && !p.bias_per_row && p.N <= BIAS_CAP - 64;
    pdl_wait();   // everything above (barriers, TMEM, descriptor prefetch) overlapped the predecessor
    // the bias may have been produced on the stream by a predecessor (C-ABI callers, rebuilt weight caches): read it
    // only after the dependency wait (plain loads: __ldg's non-coherent path could serve a stale line)
    if (bias_cached)
        for (int i = threadIdx.x; i < BIAS_CAP; i += THREADS) bias_s[i] = i < p.N ? p.bias[i] : 0.0f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    if (warp == 0) {
        // ----------------------------- TMA producer -----------------------------
        {
            const bool leader = elect_one();
            int stage = 0;
            uint32_t phase = 0;
            TileWalk w(p);
            if (p.b_resident && w.valid() && leader) {
                mbar_arrive_expect_tx(bres_full, p.num_kb * B_BYTES);
                for (int kb = 0; kb < p.num_kb; ++kb)
                    tma_load_3d(smem + kb * B_BYTES, &tma_b, bres_full, kb * BK, w.nt_fixed * BN, 0);
            }
            for (; w.valid(); w.next()) {
                int z, mt, nt;
                w.decode(p, z, mt, nt);
                const int zb = p.b_batched ? z / p.b_batch_div : 0;
                for (int kb = 0; kb < p.num_kb; ++kb) {
                    int acol = kb * BK, arow = mt * BM;
                    if (p.n_seg > 0) {
                        const int seg = kb / p.kb_per_seg;
                        acol = p.seg_acol[seg] + (kb - seg * p.kb_per_seg) * BK;
                        arow += p.a_row_off + p.seg_shift[seg];
                    }
                    mbar_wait_sleep(&empty_bar[stage], phase ^ 1);
                    if (leader) {
                        uint8_t* sa = ring + stage * ring_stride;
                        if (p.b_resident) {
                            mbar_arrive_expect_tx(&full_bar[stage], A_BYTES);
                            tma_load_3d(sa, &tma_a, &full_bar[stage], acol, arow, p.a_batched ? z : 0);
                        } else {
                            mbar_arrive_expect_tx(&full_bar[stage], STAGE_BYTES);
                            tma_load_3d(sa, &tma_a, &full_bar[stage], acol, arow, p.a_batched ? z : 0);
                            tma_load_3d(sa + A_BYTES, &tma_b, &full_bar[stage], kb * BK, nt * BN, zb);
                        }
                    }
                    __syncwarp();
                    if (++stage == n_stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------ MMA issuer ------------------------------
        {
            const bool leader = elect_one();
            constexpr uint32_t idesc = make_idesc_bf16(BM, BN);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            if (p.b_resident) {
                mbar_wait_sleep(bres_full, 0);
                tc_fence_after();
            }
            for (TileWalk w(p); w.valid(); w.next()) {
                mbar_wait_sleep(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < p.num_kb; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    if (leader) {
                        const uint32_t sa = smem_u32(ring + stage * ring_stride);
                        const uint64_t adesc = make_kmajor_desc(sa, 128);
                        const uint64_t bdesc = make_kmajor_desc(p.b_resident ? smem_u32(smem + kb * B_BYTES) : sa + A_BYTES, 128);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) {
                            // +32 bytes per K=16 step inside the 128B swizzle atom (>>4 -> +2)
                            tc_mma_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
                        }
                        tc_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs retire
                    }
                    __syncwarp();
                    if (++stage == n_stages) { stage = 0; phase ^= 1; }
                }
                if (leader) tc_commit(&tmem_full[acc]);
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else if (warp >= 4 && p.conv_xv != nullptr) {
        // ------------------- epilogue of the 3x3 shared_conv: ReLU(acc + bias) -> token-major bf16 xv, xk = xv + pos -------------------
        // (cmt_head.py:280-287,481 + cmt_transformer.py:105-110 + petr_transformer.py:296-299 for the BEV tokens: the NCHW
        // fp32 map the reference writes and re-reads never exists.)  A thread owns one padded position and 32 consecutive
        // channels per chunk: 64 contiguous bytes of each output row, 128 contiguous bytes of the position encoding.
        const int quad = warp & 3;
        const int half = (warp - 4) >> 2;
        const uint32_t bias_addr = smem_u32(bias_s);
        int acc = 0;
        uint32_t acc_phase = 0;
        for (TileWalk w(p); w.valid(); w.next()) {
            int z, mt, nt;
            w.decode(p, z, mt, nt);
            const int m = mt * BM + quad * 32 + lane;
            const int y = m / p.conv_Wp, x = m - y * p.conv_Wp;
            const int tok = (y - 1) * p.conv_W + (x - 1);
            const bool ok = m < p.M && y >= 1 && y <= p.conv_H && x >= 1 && x <= p.conv_W && tok >= p.conv_tok_begin && tok < p.conv_tok_end;
            const long long orow = static_cast<long long>(z) * p.conv_frame_stride + static_cast<long long>(tok - p.conv_tok_begin) * p.N;
            mbar_wait_sleep(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const int n_first = nt * BN + half * (BN / 2);
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * BN + half * (BN / 2);
            const int n_chunks = min(4, (p.N - n_first + 31) >> 5);
            uint32_t v[2][32];
            if (n_chunks > 0) {
                tmem_ld32(t_row, v[0]);
                tc_wait_ld();
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (c >= n_chunks) break;
                if (c + 1 < n_chunks) tmem_ld32(t_row + (c + 1) * 32, v[(c + 1) & 1]);
                const int n0 = n_first + c * 32;
                if (ok) {
                    const uint32_t (&vc)[32] = v[c & 1];
                    float f[32];
                    const uint32_t baddr = bias_addr + n0 * 4;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float4 b;
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(baddr + i * 16));
                        f[4 * i] = fmaxf(b.x + __uint_as_float(vc[4 * i]), 0.0f);
                        f[4 * i + 1] = fmaxf(b.y + __uint_as_float(vc[4 * i + 1]), 0.0f);
                        f[4 * i + 2] = fmaxf(b.z + __uint_as_float(vc[4 * i + 2]), 0.0f);
                        f[4 * i + 3] = fmaxf(b.w + __uint_as_float(vc[4 * i + 3]), 0.0f);
                    }
                    uint8_t* dv = reinterpret_cast<uint8_t*>(p.conv_xv) + (orow + n0) * 2;
                    uint8_t* dk = reinterpret_cast<uint8_t*>(p.conv_xk) + (orow + n0) * 2;
                    const float4* pp = reinterpret_cast<const float4*>(p.conv_pos + static_cast<long long>(tok) * p.N + n0);
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dv + 32 * i),
                                     "r"(pack_bf16x2(f[16 * i + 0], f[16 * i + 1])), "r"(pack_bf16x2(f[16 * i + 2], f[16 * i + 3])),
                                     "r"(pack_bf16x2(f[16 * i + 4], f[16 * i + 5])), "r"(pack_bf16x2(f[16 * i + 6], f[16 * i + 7])),
                                     "r"(pack_bf16x2(f[16 * i + 8], f[16 * i + 9])), "r"(pack_bf16x2(f[16 * i + 10], f[16 * i + 11])),
                                     "r"(pack_bf16x2(f[16 * i + 12], f[16 * i + 13])), "r"(pack_bf16x2(f[16 * i + 14], f[16 * i + 15]))
                                     : "memory");
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 q = __ldg(pp + i);
                        f[4 * i] += q.x; f[4 * i + 1] += q.y; f[4 * i + 2] += q.z; f[4 * i + 3] += q.w;
                    }
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dk + 32 * i),
                                     "r"(pack_bf16x2(f[16 * i + 0], f[16 * i + 1])), "r"(pack_bf16x2(f[16 * i + 2], f[16 * i + 3])),
                                     "r"(pack_bf16x2(f[16 * i + 4], f[16 * i + 5])), "r"(pack_bf16x2(f[16 * i + 6], f[16 * i + 7])),
                                     "r"(pack_bf16x2(f[16 * i + 8], f[16 * i + 9])), "r"(pack_bf16x2(f[16 * i + 10], f[16 * i + 11])),
                                     "r"(pack_bf16x2(f[16 * i + 12], f[16 * i + 13])), "r"(pack_bf16x2(f[16 * i + 14], f[16 * i + 15]))
                                     : "memory");
                    }
                }
                if (c + 1 < n_chunks) tc_wait_ld();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    } else if (warp >= 4 && p.direct) {
        // ------------------- epilogue, lean path: registers -> 256-bit global stores -------------------
        // ncu on the K projection: l1tex (shared-memory) throughput 78 %, tensor pipe 42 %.  With cta_group::1 the MMAs
        // alone read 96 B/clk of operands out of the 128 B/clk shared memory (A 4 KB + B 8 KB per 128-cycle
        // instruction), so an epilogue that stages the tile in shared memory for a TMA store (64 KB written +
        // 64 KB read per tile) competes for the kernel's scarcest resource.  A thread owns one output row and 32
        // consecutive columns of it, i.e. 64 contiguous bytes of bf16 (128 of fp32) in EVERY layout this kernel
        // writes: two (four) st.global.v8.b32 per chunk are full-sector writes with no staging at all.
        // Transposed output (V^T: element (m, n) at (n % cb) * ldc + m): a warp instruction writes the 32 rows of
        // one column, 64 contiguous bytes.
        const int quad = warp & 3;
        const int half = (warp - 4) >> 2;
        const bool scale = p.alpha != 1.0f;
        const bool relu = p.relu != 0;
        const int esz = p.out_bf16 ? 2 : 4;
        const uint32_t bias_addr = smem_u32(bias_s);
        int acc = 0;
        uint32_t acc_phase = 0;
        for (TileWalk w(p); w.valid(); w.next()) {
            int z, mt, nt;
            w.decode(p, z, mt, nt);
            const int m = mt * BM + quad * 32 + lane;
            const bool m_ok = m < p.M;
            const float row_bias = (p.bias != nullptr && p.bias_per_row && m_ok) ? __ldg(p.bias + m) : 0.0f;
            // column block of the warp's first chunk: one division per tile, then +32 columns per chunk
            const int n_first = nt * BN + half * (BN / 2);
            long long nb = n_first / p.cb;
            long long rem = n_first - nb * p.cb;
            const long long row_off = z * p.strideC + (p.transpose_c ? static_cast<long long>(m) : static_cast<long long>(m) * p.ldc);
            mbar_wait_sleep(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * BN + half * (BN / 2);
            // software pipeline over the warp's four 32-column chunks: the TMEM load of chunk c + 1 is in flight while
            // chunk c is biased / packed / stored (tcgen05.wait::ld waits for every outstanding load, so the wait
            // comes after the work on the current chunk)
            const int n_chunks = min(4, (p.N - n_first + 31) >> 5);   // warp-uniform; <= 0: nothing to do
            uint32_t v[2][32];
            if (n_chunks > 0) {
                tmem_ld32(t_row, v[0]);
                tc_wait_ld();
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (c >= n_chunks) break;
                if (c + 1 < n_chunks) tmem_ld32(t_row + (c + 1) * 32, v[(c + 1) & 1]);
                const int n0 = n_first + c * 32;
                {
                    float f[32];
                    const uint32_t (&vc)[32] = v[c & 1];
                    if (bias_cached) {
                        const uint32_t baddr = bias_addr + n0 * 4;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            float4 b;
                            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(baddr + i * 16));
                            f[4 * i] = b.x + __uint_as_float(vc[4 * i]);
                            f[4 * i + 1] = b.y + __uint_as_float(vc[4 * i + 1]);
                            f[4 * i + 2] = b.z + __uint_as_float(vc[4 * i + 2]);
                            f[4 * i + 3] = b.w + __uint_as_float(vc[4 * i + 3]);
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; ++i) f[i] = row_bias + __uint_as_float(vc[i]);
                    }
                    if (scale) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) f[i] *= p.alpha;
                    }
                    if (relu) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.0f);
                    }
                    if (p.norm2_max != nullptr) {
                        // max over the tile's rows of |row block|^2 (non-negative floats order like their bit patterns)
                        float n2 = 0.0f;
#pragma unroll
                        for (int i = 0; i < 32; ++i) n2 = fmaf(f[i], f[i], n2);
                        const unsigned int wmax = __reduce_max_sync(0xffffffffu, m_ok ? __float_as_uint(n2) : 0u);
                        if (lane == 0)
                            atomicMax(reinterpret_cast<unsigned int*>(p.norm2_max) + static_cast<long long>(z) * (p.N >> 5) + (n0 >> 5), wmax);
                    }
                    const long long blk_off = nb * p.cb_stride;
                    if (p.transpose_c) {
                        // element (m, n) -> blk_off + (n % cb) * ldc + m  (bf16 only)
                        uint16_t* dst = reinterpret_cast<uint16_t*>(p.C) + row_off + blk_off + rem * p.ldc;
                        if (m_ok) {
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const uint32_t w2 = pack_bf16x2(f[2 * i], f[2 * i + 1]);
                                dst[static_cast<long long>(2 * i) * p.ldc] = static_cast<uint16_t>(w2 & 0xffffu);
                                dst[static_cast<long long>(2 * i + 1) * p.ldc] = static_cast<uint16_t>(w2 >> 16);
                            }
                        }
                    } else if (p.out_bf16) {
                        uint8_t* dst = reinterpret_cast<uint8_t*>(p.C) + (row_off + blk_off + rem) * esz;
                        if (m_ok) {
#pragma unroll
                            for (int i = 0; i < 2; ++i)
                                asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + 32 * i),
                                             "r"(pack_bf16x2(f[16 * i + 0], f[16 * i + 1])), "r"(pack_bf16x2(f[16 * i + 2], f[16 * i + 3])),
                                             "r"(pack_bf16x2(f[16 * i + 4], f[16 * i + 5])), "r"(pack_bf16x2(f[16 * i + 6], f[16 * i + 7])),
                                             "r"(pack_bf16x2(f[16 * i + 8], f[16 * i + 9])), "r"(pack_bf16x2(f[16 * i + 10], f[16 * i + 11])),
                                             "r"(pack_bf16x2(f[16 * i + 12], f[16 * i + 13])), "r"(pack_bf16x2(f[16 * i + 14], f[16 * i + 15]))
                                             : "memory");
                        }
                    } else {
                        uint8_t* dst = reinterpret_cast<uint8_t*>(p.C) + (row_off + blk_off + rem) * esz;
                        if (m_ok) {
#pragma unroll
                            for (int i = 0; i < 4; ++i)
                                asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + 32 * i),
                                             "r"(__float_as_uint(f[8 * i + 0])), "r"(__float_as_uint(f[8 * i + 1])),
                                             "r"(__float_as_uint(f[8 * i + 2])), "r"(__float_as_uint(f[8 * i + 3])),
                                             "r"(__float_as_uint(f[8 * i + 4])), "r"(__float_as_uint(f[8 * i + 5])),
                                             "r"(__float_as_uint(f[8 * i + 6])), "r"(__float_as_uint(f[8 * i + 7]))
                                             : "memory");
                        }
                    }
                    rem += 32;
                    if (rem >= p.cb) { rem -= p.cb; ++nb; }
                }
                if (c + 1 < n_chunks) tc_wait_ld();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    } else if (warp >= 4) {
        // ------------------------------- epilogue -------------------------------
        // 8 warps: warp w reads TMEM lane quadrant (w & 3) and column half ((w - 4) >> 2), so every
        // scheduler has two epilogue warps to overlap TMEM / global latencies.  All option tests
        // (bias kind, alpha, relu, dtype) are hoisted out of the per-element loops.
        const int quad = warp & 3;
        const int half = (warp - 4) >> 2;
        const bool has_bias = p.bias != nullptr;
        const bool col_bias = has_bias && !p.bias_per_row;
        const bool scale = p.alpha != 1.0f;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (TileWalk w(p); w.valid(); w.next()) {
            int z, mt, nt;
            w.decode(p, z, mt, nt);
            const int m = mt * BM + quad * 32 + lane;
            const bool m_ok = m < p.M;
            const float row_bias = (has_bias && p.bias_per_row && m_ok) ? __ldg(p.bias + m) : 0.0f;
            mbar_wait_sleep(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * BN;
            // column-block addressing without a 64-bit division per chunk: one division per tile, then the
            // (block, offset-in-block) pair advances by 32 columns per chunk
            const int c_first = half * (BN / 64);
            const long long n_first = static_cast<long long>(nt) * BN + c_first * 32;
            long long blk = n_first / p.cb;
            long long rem = n_first - blk * p.cb;
            const long long row_off = z * p.strideC + static_cast<long long>(m) * p.ldc;
            // bias for one 32-column chunk (independent of the accumulator: issued before the TMEM wait)
            auto load_bias = [&](int n0, float (&f)[32]) {
                if (bias_cached) {
                    // n0 + 32 may pass N in the last tile: the extra values only reach columns the store clips
                    const float4* b4 = reinterpret_cast<const float4*>(bias_s + n0);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 b = (n0 + 4 * i + 4 <= BIAS_CAP) ? b4[i] : make_float4(0.f, 0.f, 0.f, 0.f);
                        f[4 * i] = b.x; f[4 * i + 1] = b.y; f[4 * i + 2] = b.z; f[4 * i + 3] = b.w;
                    }
                } else if (col_bias) {
                    if (n0 + 32 <= p.N) {
                        const float4* b4 = reinterpret_cast<const float4*>(p.bias + n0);  // n0 % 32 == 0
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float4 b = __ldg(b4 + i);
                            f[4 * i] = b.x; f[4 * i + 1] = b.y; f[4 * i + 2] = b.z; f[4 * i + 3] = b.w;
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; ++i) f[i] = (n0 + i < p.N) ? __ldg(p.bias + n0 + i) : 0.0f;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) f[i] = row_bias;
                }
            };
            auto finish = [&](int n0, long long off, const uint32_t (&v)[32], float (&f)[32]) {
                const bool full = (n0 + 32 <= p.N);
#pragma unroll
                for (int i = 0; i < 32; ++i) f[i] += __uint_as_float(v[i]);
                if (scale) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) f[i] *= p.alpha;
                }
                if (p.relu) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.0f);
                }
                if (!m_ok) return;
                if (p.out_bf16) {
                    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.C) + off;
                    if (full && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            uint4 w;
                            w.x = pack_bf16x2(f[8 * i + 0], f[8 * i + 1]);
                            w.y = pack_bf16x2(f[8 * i + 2], f[8 * i + 3]);
                            w.z = pack_bf16x2(f[8 * i + 4], f[8 * i + 5]);
                            w.w = pack_bf16x2(f[8 * i + 6], f[8 * i + 7]);
                            reinterpret_cast<uint4*>(dst)[i] = w;
                        }
                    } else {
                        for (int i = 0; i < 32; ++i)
                            if (n0 + i < p.N) dst[i] = __float2bfloat16_rn(f[i]);
                    }
                } else {
                    float* dst = reinterpret_cast<float*>(p.C) + off;
                    if (full && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            reinterpret_cast<float4*>(dst)[i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
                    } else {
                        for (int i = 0; i < 32; ++i)
                            if (n0 + i < p.N) dst[i] = f[i];
                    }
                }
            };
            // two 32-column chunks per round: both TMEM loads and both bias fetches are in flight together
#pragma unroll 1
            for (int c = c_first; c < c_first + BN / 64; c += 2) {
                const int n0a = nt * BN + c * 32, n0b = n0a + 32;
                if (n0a >= p.N) break;  // warp-uniform
                const bool has_b = n0b < p.N;
                const long long offa = row_off + blk * p.cb_stride + rem;
                rem += 32;
                if (rem >= p.cb) { rem -= p.cb; ++blk; }
                const long long offb = row_off + blk * p.cb_stride + rem;
                rem += 32;
                if (rem >= p.cb) { rem -= p.cb; ++blk; }
                uint32_t va[32], vb[32];
                float fa[32], fb[32];
                tmem_ld32(t_row + c * 32, va);
                if (has_b) tmem_ld32(t_row + (c + 1) * 32, vb);
                load_bias(n0a, fa);
                if (has_b) load_bias(n0b, fb);
                tc_wait_ld();
                finish(n0a, offa, va, fa);
                if (has_b) finish(n0b, offb, vb, fb);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

int launch_tc_gemm(const GemmArgs& g, int batch, cudaStream_t stream) {
    using namespace gemm;
    CMT_CHECK_ARG(g.n_seg >= 0 && g.n_seg <= MAX_SEG, "cmt_gemm(bf16): at most %d K segments", MAX_SEG);
    CMT_CHECK_ARG(g.n_seg == 0 || (g.seg_k > 0 && g.seg_k % BK == 0 && g.K == g.n_seg * g.seg_k && g.a_cols > 0 && g.a_rows > 0),
                  "cmt_gemm(bf16): segmented K needs seg_k %% %d == 0 and K == n_seg * seg_k", BK);
    CMT_CHECK_ARG(g.K % 8 == 0 && g.lda % 8 == 0 && g.ldb % 8 == 0,
                  "cmt_gemm_bias_act(bf16): K, lda, ldb must be multiples of 8 (K=%d lda=%lld ldb=%lld)",
                  g.K, g.lda, g.ldb);
    CMT_CHECK_ARG(((reinterpret_cast<uintptr_t>(g.A) | reinterpret_cast<uintptr_t>(g.B)) & 15) == 0,
                  "cmt_gemm_bias_act(bf16): operands must be 16-byte aligned");
    CMT_CHECK_ARG(g.cb >= g.N || g.cb % 32 == 0,
                  "cmt_gemm_bias_act(bf16): column block must be >= N or a multiple of 32");
    CMT_CHECK_ARG(g.strideA % 8 == 0 && g.strideB % 8 == 0, "cmt_gemm_bias_act(bf16): batch strides must be multiples of 8");

    static DeviceOnce attr_once;
    int attr_dev;
    if (attr_once.need(&attr_dev)) {
        cudaError_t e = cudaFuncSetAttribute(tc_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             SMEM_BYTES);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(tc_gemm)");
        attr_once.mark(attr_dev);
    }

    CUtensorMap ta, tb;
    {
        const bool batched = g.strideA != 0 && batch > 1;
        const long long a_rows = g.n_seg > 0 ? g.a_rows : g.M;
        uint64_t dims[3] = {static_cast<uint64_t>(g.n_seg > 0 ? g.a_cols : g.K), static_cast<uint64_t>(a_rows),
                            static_cast<uint64_t>(batched ? batch : 1)};
        uint64_t strides[2] = {static_cast<uint64_t>(g.lda) * 2,
                               static_cast<uint64_t>(batched ? g.strideA : a_rows * g.lda) * 2};
        uint32_t box[3] = {BK, BM, 1};
        int rc = encode_tma_bf16(&ta, g.A, 3, dims, strides, box, 128);
        if (rc) return rc;
    }
    {
        const bool batched = g.strideB != 0 && batch > 1;
        const int b_div = g.b_batch_div > 1 ? g.b_batch_div : 1;
        uint64_t dims[3] = {static_cast<uint64_t>(g.K), static_cast<uint64_t>(g.N),
                            static_cast<uint64_t>(batched ? (batch + b_div - 1) / b_div : 1)};
        uint64_t strides[2] = {static_cast<uint64_t>(g.ldb) * 2,
                               static_cast<uint64_t>(batched ? g.strideB : (long long)g.N * g.ldb) * 2};
        uint32_t box[3] = {BK, BN, 1};
        int rc = encode_tma_bf16(&tb, g.B, 3, dims, strides, box, 128);
        if (rc) return rc;
    }

    const int esz = g.out_bf16 ? 2 : 4;
    const bool plain = g.cb >= g.N;

    TcGemmParams p{};
    p.transpose_c = g.transpose_c;
    p.norm2_max = g.norm2_max;
    p.n_seg = g.n_seg;
    p.kb_per_seg = g.n_seg > 0 ? g.seg_k / BK : 0;
    p.a_row_off = g.a_row_off;
    for (int i = 0; i < g.n_seg; ++i) {
        p.seg_acol[i] = g.seg_acol[i];
        p.seg_shift[i] = g.seg_shift[i];
    }
    p.b_batch_div = g.b_batch_div > 1 ? g.b_batch_div : 1;
    p.conv_xk = g.conv_xk;
    p.conv_xv = g.conv_xv;
    p.conv_pos = g.conv_pos;
    p.conv_W = g.conv_W;
    p.conv_H = g.conv_H;
    p.conv_Wp = g.conv_Wp;
    p.conv_tok_begin = g.conv_tok_begin;
    p.conv_tok_end = g.conv_tok_end;
    p.conv_frame_stride = g.conv_frame_stride;
    if (g.conv_xv != nullptr)
        CMT_CHECK_ARG(g.conv_xk && g.conv_pos && g.bias && !g.bias_per_row && g.N % 32 == 0 && g.N <= BIAS_CAP - 64 &&
                          (reinterpret_cast<uintptr_t>(g.conv_xk) & 31) == 0 && (reinterpret_cast<uintptr_t>(g.conv_xv) & 31) == 0 &&
                          (reinterpret_cast<uintptr_t>(g.conv_pos) & 15) == 0 && g.conv_frame_stride % 16 == 0,
                      "cmt_shared_conv_tokens: bias, pos, 32-byte aligned outputs and N %% 32 == 0 required");
    static const bool no_direct = getenv("CMT_GEMM_NO_DIRECT") != nullptr;
    const bool bias_ok = g.bias == nullptr || g.bias_per_row || g.N <= BIAS_CAP - 64;
    if (g.transpose_c) {
        CMT_CHECK_ARG(g.out_bf16 && g.cb % 32 == 0 && g.N % 32 == 0 && bias_ok && !plain,
                      "cmt_gemm_bias_act(bf16): transposed output needs bf16, cb %% 32 == 0, N %% 32 == 0, N <= %d", BIAS_CAP - 64);
        p.direct = 1;
    } else {
        const bool aligned = (reinterpret_cast<uintptr_t>(g.C) & 31) == 0 && (g.ldc * esz) % 32 == 0 &&
                             (plain || ((g.cb_stride * esz) % 32 == 0 && g.cb % 32 == 0)) &&
                             (batch == 1 || (g.strideC * esz) % 32 == 0);
        p.direct = (aligned && g.N % 32 == 0 && bias_ok && !no_direct) ? 1 : 0;
    }
    CMT_CHECK_ARG(g.norm2_max == nullptr || p.direct, "cmt_gemm_bias_act(bf16): norm2_max needs N %% 32 == 0, 32-byte aligned C rows "
                                                      "and N <= %d with a column bias", BIAS_CAP - 64);
    p.bias = g.bias;
    p.C = g.C;
    p.M = g.M;
    p.N = g.N;
    p.K = g.K;
    p.ldc = g.ldc;
    p.cb = g.cb;
    p.cb_stride = g.cb_stride;
    p.strideC = g.strideC;
    p.alpha = g.alpha;
    p.relu = g.relu;
    p.bias_per_row = g.bias_per_row;
    p.out_bf16 = g.out_bf16;
    p.a_batched = (g.strideA != 0 && batch > 1) ? 1 : 0;
    p.b_batched = (g.strideB != 0 && batch > 1) ? 1 : 0;
    p.m_tiles = (g.M + BM - 1) / BM;
    p.n_tiles = (g.N + BN - 1) / BN;
    if (g.conv_xv != nullptr) {
        // only the m-tiles whose padded rows hold tokens of [tok_begin, tok_end)
        const int y_lo = g.conv_tok_begin / g.conv_W, y_hi = (g.conv_tok_end - 1) / g.conv_W;
        const int p_lo = (y_lo + 1) * g.conv_Wp + 1, p_hi = (y_hi + 1) * g.conv_Wp + g.conv_W + 1;   // [p_lo, p_hi)
        p.mt_off = p_lo / BM;
        p.m_tiles = (p_hi + BM - 1) / BM - p.mt_off;
    }
    const long long total = static_cast<long long>(p.m_tiles) * p.n_tiles * batch;
    CMT_CHECK_ARG(total < (1ll << 31), "cmt_gemm_bias_act(bf16): too many tiles");
    p.total_tiles = static_cast<int>(total);
    p.num_kb = (g.K + BK - 1) / BK;
    int grid = device_sm_count();
    if (grid > p.total_tiles) grid = p.total_tiles;
    const long long mz = static_cast<long long>(p.m_tiles) * batch;
    static const bool no_resident = getenv("CMT_GEMM_NO_B_RESIDENT") != nullptr;
    if (p.num_kb <= RES_KB && !p.b_batched && p.n_tiles <= device_sm_count() && !no_resident) {
        long long gm = device_sm_count() / p.n_tiles;
        if (gm > mz) gm = mz;
        p.b_resident = 1;
        grid = static_cast<int>(gm) * p.n_tiles;
    }
    {
        cudaError_t e = launch_pdl(tc_gemm_kernel, dim3(grid), dim3(THREADS), SMEM_BYTES, stream, ta, tb, p);
        if (e != cudaSuccess) return cuda_fail(e, "cmt_gemm_bias_act(tcgen05) launch");
    }
    CMT_LAUNCH_CHECK("cmt_gemm_bias_act(tcgen05)");
    return CMT_OK;
}

}  // namespace cmt
