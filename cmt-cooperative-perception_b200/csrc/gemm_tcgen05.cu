// K2: projection / MLP GEMM on the 5th-gen tensor cores.
//
//   C = act((A * B^T + bias) * alpha),  A:[M,K], B:[N,K] both bf16 or both fp16 (K-major), fp32 accumulate.
//
// Persistent, warp-specialised kernel, one CTA per SM:
//   warp 0      TMA producer  : 3-D tensor maps (K, rows, batch), 128B swizzle.  Streaming mode: 4-stage ring of
//                               A+B k-blocks.  B-resident mode (K <= 256, B not batched): the CTA's n-tile of B is
//                               loaded once, the ring carries A only (5 stages).
//   warp 1      MMA issuer    : one elected thread, tcgen05.mma cta_group::1 kind::f16,
//                               M=128 x N=256 x K=16 per instruction, accumulator in TMEM
//   warp 2      TMEM allocator (512 columns = two 128x256 fp32 accumulators, ping-pong)
//   warps 4..11 epilogue      : one loop for every output layout: tcgen05.ld 32x32b -> bias (cached in shared memory,
//                               or per row) / alpha / ReLU -> bf16|fp16|fp32 -> global stores straight from registers (a
//                               thread owns 32 consecutive columns of one row: 64 / 128 contiguous bytes), overlapped
//                               with the next tile's main loop.  Store form (one instantiation each): 256-bit where the
//                               layout is 32-byte aligned, masked scalar, transposed for V^T, or the shared_conv token
//                               pair.  No shared-memory staging: the MMAs already read 96 of the 128 B/clk.
//
// Replaces F.linear in models/utils/attention.py:21-27,138 and the PE MLPs of
// models/dense_heads/cmt_head.py:292-301 (reference runs them as fp32 cuBLAS SGEMMs).
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

constexpr int MAX_SEG = sizeof(GemmArgs::seg_acol) / sizeof(int);

// The caller's arguments and what the host derives from them.
struct TcGemmParams {
    GemmArgs g;        // b_batch_div normalised to >= 1
    int a_batched, b_batched;
    int m_tiles, n_tiles, total_tiles, num_kb;
    int kb_per_seg;    // segmented K: K block kb belongs to segment kb / kb_per_seg (B is read at column kb * BK as usual)
    int mt_off;        // first m-tile (conv with a token sub-range computes only the rows that hold its tokens)
    int b_resident;    // 1: gridDim.x = Gm * n_tiles, CTA c owns n-tile c % n_tiles and the (batch, m-tile) pairs c / n_tiles + i * Gm
    int vec_store;     // 1: C, ldc, cb_stride and strideC put every full 32-column chunk of a row on a 32-byte boundary
};

// How the epilogue stores a chunk.  The host picks one instantiation of the kernel per launch, so the hot layouts run
// a loop body with no tests for the forms they do not use.
enum class Store {
    Vec,          // row-major, 32-byte aligned layout, N % 32 == 0, no column bias too wide for the cache: 256-bit stores
    Masked,       // row-major otherwise: 256-bit stores for the full chunks of an aligned layout, masked scalar stores else;
                  // the only form that reads a column bias too wide for the cache
    Transposed,   // C^T inside each column block (V^T), 16-bit
    Conv,         // shared_conv token pair xv / xk
};

// 32 consecutive outputs of one row as 256-bit stores (dst 32-byte aligned): 16-bit (kLp = CMT_BF16 | CMT_F16), 64 bytes /
// fp32, 128 bytes
template <int kLp>
__device__ __forceinline__ void st_lp16x32(uint8_t* dst, const float (&f)[32]) {
#pragma unroll
    for (int i = 0; i < 2; ++i)
        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + 32 * i),
                     "r"(pack_lp2<kLp>(f[16 * i + 0], f[16 * i + 1])), "r"(pack_lp2<kLp>(f[16 * i + 2], f[16 * i + 3])),
                     "r"(pack_lp2<kLp>(f[16 * i + 4], f[16 * i + 5])), "r"(pack_lp2<kLp>(f[16 * i + 6], f[16 * i + 7])),
                     "r"(pack_lp2<kLp>(f[16 * i + 8], f[16 * i + 9])), "r"(pack_lp2<kLp>(f[16 * i + 10], f[16 * i + 11])),
                     "r"(pack_lp2<kLp>(f[16 * i + 12], f[16 * i + 13])), "r"(pack_lp2<kLp>(f[16 * i + 14], f[16 * i + 15]))
                     : "memory");
}

__device__ __forceinline__ void st_f32x32(uint8_t* dst, const float (&f)[32]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + 32 * i),
                     "r"(__float_as_uint(f[8 * i + 0])), "r"(__float_as_uint(f[8 * i + 1])),
                     "r"(__float_as_uint(f[8 * i + 2])), "r"(__float_as_uint(f[8 * i + 3])),
                     "r"(__float_as_uint(f[8 * i + 4])), "r"(__float_as_uint(f[8 * i + 5])),
                     "r"(__float_as_uint(f[8 * i + 6])), "r"(__float_as_uint(f[8 * i + 7]))
                     : "memory");
}

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

// kF16: fp16 operands and 16-bit outputs (g.f16), bf16 otherwise -- its own instantiations, so the bf16 kernels are
// exactly what they were before fp16 existed.
template <Store S, bool kF16>
__global__ void __launch_bounds__(gemm::THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
               const TcGemmParams p) {
    using namespace gemm;
    constexpr int LP = kF16 ? CMT_F16 : CMT_BF16;
    const GemmArgs& g = p.g;
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
    const bool bias_cached = g.bias != nullptr && !g.bias_per_row && g.N <= BIAS_CAP - 64;
    pdl_wait();   // everything above (barriers, TMEM, descriptor prefetch) overlapped the predecessor
    // the bias may have been produced on the stream by a predecessor (C-ABI callers, rebuilt weight caches): read it
    // only after the dependency wait (plain loads: __ldg's non-coherent path could serve a stale line)
    if (bias_cached)
        for (int i = threadIdx.x; i < BIAS_CAP; i += THREADS) bias_s[i] = i < g.N ? g.bias[i] : 0.0f;
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
                const int zb = p.b_batched ? z / g.b_batch_div : 0;
                for (int kb = 0; kb < p.num_kb; ++kb) {
                    int acol = kb * BK, arow = mt * BM;
                    if (g.n_seg > 0) {
                        const int seg = kb / p.kb_per_seg;
                        acol = g.seg_acol[seg] + (kb - seg * p.kb_per_seg) * BK;
                        arow += g.a_row_off + g.seg_shift[seg];
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
            constexpr uint32_t idesc = make_idesc(BM, BN, kF16);
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
    } else if (warp >= 4) {
        // ---------------------- epilogue: TMEM -> bias / alpha / ReLU -> global, straight from registers ----------------------
        // ncu on the K projection: l1tex (shared-memory) throughput 78 %, tensor pipe 42 %.  With cta_group::1 the MMAs
        // alone read 96 B/clk of operands out of the 128 B/clk shared memory (A 4 KB + B 8 KB per 128-cycle
        // instruction), so an epilogue that stages the tile in shared memory for a TMA store (64 KB written +
        // 64 KB read per tile) competes for the kernel's scarcest resource.  Warp w reads TMEM lane quadrant (w & 3) and
        // column half ((w - 4) >> 2), so every scheduler has two epilogue warps.  A thread owns one output row and 32
        // consecutive columns of it per chunk, i.e. 64 contiguous bytes of bf16 (128 of fp32): where the host found the
        // layout 32-byte aligned, two (four) st.global.v8.b32 per chunk are full-sector writes with no staging at all;
        // other layouts and the ragged last chunk take masked scalar stores.
        // Transposed output (V^T: element (m, n) at (n % cb) * ldc + m): a warp instruction writes the 32 rows of
        // one column, 64 contiguous bytes.
        // shared_conv tokens (cmt_head.py:280-287,481 + cmt_transformer.py:105-110 + petr_transformer.py:296-299 for the
        // BEV tokens: the NCHW fp32 map the reference writes and re-reads never exists): the thread's row is a padded
        // position, stored as xv = lp(ReLU(acc + bias)) and xk = lp(that + pos), 64 contiguous bytes each.
        const int quad = warp & 3;
        const int half = (warp - 4) >> 2;
        constexpr bool conv = S == Store::Conv;   // ReLU(acc + bias) with the bias cached (host checks), no alpha
        const bool col_bias = g.bias != nullptr && !g.bias_per_row;   // from bias_s when bias_cached, else from global
        const bool scale = !conv && g.alpha != 1.0f;
        const bool relu = conv || g.relu != 0;
        const int esz = g.out_16 ? 2 : 4;
        const uint32_t bias_addr = smem_u32(bias_s);
        int acc = 0;
        uint32_t acc_phase = 0;
        for (TileWalk w(p); w.valid(); w.next()) {
            int z, mt, nt;
            w.decode(p, z, mt, nt);
            const int m = mt * BM + quad * 32 + lane;
            bool row_ok = m < g.M;
            long long row_off;   // element offset of the thread's row
            int tok = 0;
            if constexpr (conv) {
                const int y = m / g.conv_Wp, x = m - y * g.conv_Wp;
                tok = (y - 1) * g.conv_W + (x - 1);
                row_ok = row_ok && y >= 1 && y <= g.conv_H && x >= 1 && x <= g.conv_W && tok >= g.conv_tok_begin && tok < g.conv_tok_end;
                row_off = static_cast<long long>(z) * g.conv_frame_stride + static_cast<long long>(tok - g.conv_tok_begin) * g.N;
            } else {
                row_off = z * g.strideC + (S == Store::Transposed ? static_cast<long long>(m) : static_cast<long long>(m) * g.ldc);
            }
            const float row_bias = (g.bias != nullptr && g.bias_per_row && row_ok) ? __ldg(g.bias + m) : 0.0f;
            // column block of the warp's first chunk: one division per tile, then +32 columns per chunk
            const int n_first = nt * BN + half * (BN / 2);
            long long nb = n_first / g.cb;
            long long rem = n_first - nb * g.cb;
            mbar_wait_sleep(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * BN + half * (BN / 2);
            // software pipeline over the warp's four 32-column chunks: the TMEM load of chunk c + 1 is in flight while
            // chunk c is biased / packed / stored (tcgen05.wait::ld waits for every outstanding load, so the wait
            // comes after the work on the current chunk)
            const int n_chunks = min(4, (g.N - n_first + 31) >> 5);   // warp-uniform; <= 0: nothing to do
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
                    if (conv || bias_cached) {
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
                    } else if (S == Store::Masked && col_bias) {
                        // wider than the cache (N > BIAS_CAP - 64)
#pragma unroll
                        for (int i = 0; i < 32; ++i) f[i] = (n0 + i < g.N ? __ldg(g.bias + n0 + i) : 0.0f) + __uint_as_float(vc[i]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; ++i) f[i] = row_bias + __uint_as_float(vc[i]);
                    }
                    if (scale) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) f[i] *= g.alpha;
                    }
                    if (relu) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) f[i] = fmaxf(f[i], 0.0f);
                    }
                    if (!conv && g.norm2_max != nullptr) {
                        // max over the tile's rows of |row block|^2 (non-negative floats order like their bit patterns)
                        float n2 = 0.0f;
#pragma unroll
                        for (int i = 0; i < 32; ++i) n2 = fmaf(f[i], f[i], n2);
                        const unsigned int wmax = __reduce_max_sync(0xffffffffu, row_ok ? __float_as_uint(n2) : 0u);
                        if (lane == 0)
                            atomicMax(reinterpret_cast<unsigned int*>(g.norm2_max) + static_cast<long long>(z) * (g.N >> 5) + (n0 >> 5), wmax);
                    }
                    const long long blk_off = row_off + nb * g.cb_stride;
                    if (row_ok) {
                        if constexpr (conv) {
                            st_lp16x32<LP>(reinterpret_cast<uint8_t*>(g.conv_xv) + (row_off + n0) * 2, f);
                            const float4* pp = reinterpret_cast<const float4*>(g.conv_pos + static_cast<long long>(tok) * g.N + n0);
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const float4 q = __ldg(pp + i);
                                f[4 * i] += q.x; f[4 * i + 1] += q.y; f[4 * i + 2] += q.z; f[4 * i + 3] += q.w;
                            }
                            st_lp16x32<LP>(reinterpret_cast<uint8_t*>(g.conv_xk) + (row_off + n0) * 2, f);
                        } else if constexpr (S == Store::Transposed) {
                            // element (m, n) -> blk_off + (n % cb) * ldc + m  (16-bit only)
                            uint16_t* dst = reinterpret_cast<uint16_t*>(g.C) + blk_off + rem * g.ldc;
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const uint32_t w2 = pack_lp2<LP>(f[2 * i], f[2 * i + 1]);
                                dst[static_cast<long long>(2 * i) * g.ldc] = static_cast<uint16_t>(w2 & 0xffffu);
                                dst[static_cast<long long>(2 * i + 1) * g.ldc] = static_cast<uint16_t>(w2 >> 16);
                            }
                        } else if (S == Store::Vec || (p.vec_store && n0 + 32 <= g.N)) {
                            uint8_t* dst = reinterpret_cast<uint8_t*>(g.C) + (blk_off + rem) * esz;
                            if (g.out_16) st_lp16x32<LP>(dst, f);
                            else st_f32x32(dst, f);
                        } else if (g.out_16 && kF16) {
                            __half* dst = reinterpret_cast<__half*>(g.C) + blk_off + rem;
#pragma unroll
                            for (int i = 0; i < 32; ++i)
                                if (n0 + i < g.N) dst[i] = __float2half_rn(f[i]);
                        } else if (g.out_16) {
                            __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(g.C) + blk_off + rem;
#pragma unroll
                            for (int i = 0; i < 32; ++i)
                                if (n0 + i < g.N) dst[i] = __float2bfloat16_rn(f[i]);
                        } else {
                            float* dst = reinterpret_cast<float*>(g.C) + blk_off + rem;
#pragma unroll
                            for (int i = 0; i < 32; ++i)
                                if (n0 + i < g.N) dst[i] = f[i];
                        }
                    }
                    rem += 32;
                    if (rem >= g.cb) { rem -= g.cb; ++nb; }
                }
                if (c + 1 < n_chunks) tc_wait_ld();
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

    // one instantiation per store form, in the order of Store: bf16, then fp16
    static void (*const kernels[])(CUtensorMap, CUtensorMap, TcGemmParams) = {
        tc_gemm_kernel<Store::Vec, false>, tc_gemm_kernel<Store::Masked, false>, tc_gemm_kernel<Store::Transposed, false>,
        tc_gemm_kernel<Store::Conv, false>, tc_gemm_kernel<Store::Vec, true>, tc_gemm_kernel<Store::Masked, true>,
        tc_gemm_kernel<Store::Transposed, true>, tc_gemm_kernel<Store::Conv, true>};
    static DeviceOnce attr_once;
    int attr_dev;
    if (attr_once.need(&attr_dev)) {
        for (auto kernel : kernels) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
            if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(tc_gemm)");
        }
        attr_once.mark(attr_dev);
    }

    const int b_div = g.b_batch_div > 1 ? g.b_batch_div : 1;
    CUtensorMap ta, tb;
    {
        const bool batched = g.strideA != 0 && batch > 1;
        const long long a_rows = g.n_seg > 0 ? g.a_rows : g.M;
        uint64_t dims[3] = {static_cast<uint64_t>(g.n_seg > 0 ? g.a_cols : g.K), static_cast<uint64_t>(a_rows),
                            static_cast<uint64_t>(batched ? batch : 1)};
        uint64_t strides[2] = {static_cast<uint64_t>(g.lda) * 2,
                               static_cast<uint64_t>(batched ? g.strideA : a_rows * g.lda) * 2};
        uint32_t box[3] = {BK, BM, 1};
        int rc = encode_tma(&ta, g.A, g.f16 ? CMT_F16 : CMT_BF16, 3, dims, strides, box, 128);
        if (rc) return rc;
    }
    {
        const bool batched = g.strideB != 0 && batch > 1;
        uint64_t dims[3] = {static_cast<uint64_t>(g.K), static_cast<uint64_t>(g.N),
                            static_cast<uint64_t>(batched ? (batch + b_div - 1) / b_div : 1)};
        uint64_t strides[2] = {static_cast<uint64_t>(g.ldb) * 2,
                               static_cast<uint64_t>(batched ? g.strideB : (long long)g.N * g.ldb) * 2};
        uint32_t box[3] = {BK, BN, 1};
        int rc = encode_tma(&tb, g.B, g.f16 ? CMT_F16 : CMT_BF16, 3, dims, strides, box, 128);
        if (rc) return rc;
    }

    const int esz = g.out_16 ? 2 : 4;
    const bool plain = g.cb >= g.N;
    if (g.conv_xv != nullptr)
        CMT_CHECK_ARG(g.conv_xk && g.conv_pos && g.bias && !g.bias_per_row && g.N % 32 == 0 && g.N <= BIAS_CAP - 64 &&
                          (reinterpret_cast<uintptr_t>(g.conv_xk) & 31) == 0 && (reinterpret_cast<uintptr_t>(g.conv_xv) & 31) == 0 &&
                          (reinterpret_cast<uintptr_t>(g.conv_pos) & 15) == 0 && g.conv_frame_stride % 16 == 0,
                      "cmt_shared_conv_tokens: bias, pos, 32-byte aligned outputs and N %% 32 == 0 required");
    const bool bias_ok = g.bias == nullptr || g.bias_per_row || g.N <= BIAS_CAP - 64;
    if (g.transpose_c)
        CMT_CHECK_ARG(g.out_16 && g.cb % 32 == 0 && g.N % 32 == 0 && bias_ok && !plain,
                      "cmt_gemm_bias_act(bf16): transposed output needs a 16-bit output, cb %% 32 == 0, N %% 32 == 0, N <= %d", BIAS_CAP - 64);
    const bool aligned = (reinterpret_cast<uintptr_t>(g.C) & 31) == 0 && (g.ldc * esz) % 32 == 0 &&
                         (plain || ((g.cb_stride * esz) % 32 == 0 && g.cb % 32 == 0)) &&
                         (batch == 1 || (g.strideC * esz) % 32 == 0);
    CMT_CHECK_ARG(g.norm2_max == nullptr || g.transpose_c || (aligned && g.N % 32 == 0 && bias_ok),
                  "cmt_gemm_bias_act(bf16): norm2_max needs N %% 32 == 0, 32-byte aligned C rows and N <= %d with a column bias",
                  BIAS_CAP - 64);

    const Store form = g.conv_xv != nullptr ? Store::Conv
                       : g.transpose_c        ? Store::Transposed
                       : (aligned && g.N % 32 == 0 && bias_ok) ? Store::Vec : Store::Masked;

    TcGemmParams p{};
    p.g = g;
    p.g.b_batch_div = b_div;
    p.vec_store = aligned;
    p.kb_per_seg = g.n_seg > 0 ? g.seg_k / BK : 0;
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
    if (p.num_kb <= RES_KB && !p.b_batched && p.n_tiles <= device_sm_count()) {
        long long gm = device_sm_count() / p.n_tiles;
        if (gm > mz) gm = mz;
        p.b_resident = 1;
        grid = static_cast<int>(gm) * p.n_tiles;
    }
    {
        cudaError_t e = launch_pdl(kernels[static_cast<int>(form) + (g.f16 ? 4 : 0)], dim3(grid), dim3(THREADS), SMEM_BYTES, stream, ta, tb, p);
        if (e != cudaSuccess) return cuda_fail(e, "cmt_gemm_bias_act(tcgen05) launch");
    }
    CMT_LAUNCH_CHECK("cmt_gemm_bias_act(tcgen05)");
    return CMT_OK;
}

}  // namespace cmt
