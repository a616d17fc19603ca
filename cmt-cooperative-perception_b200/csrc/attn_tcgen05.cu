// K3: flash-style cross-attention of the object queries over the BEV ++ image tokens on the
// 5th-gen tensor cores (head dim 32, bf16 operands, fp32 accumulate / softmax statistics).
//
// Replaces flash_attn_unpadded_kvpacked_func as called from
// projects/mmdet3d_plugin/models/utils/attention.py:46-92 (softmax(QK^T/sqrt(d))V, non-causal).
//
// Work decomposition.  An "item" is (frame b, head h, block of 384 queries = three 128-row tiles, one per softmax
// warpgroup); it needs T = ceil(n_tokens/64) KV tile-steps.  The flat space items x T is cut into equal WEIGHTED
// contiguous ranges (stream-K), one per persistent CTA, so that any batch size fills all 148 SMs;
// every (item, range) overlap ("segment") writes a normalised fp32 partial + log2-sum-exp into the workspace and
// a second kernel merges the segments of each item.  The same partial/LSE algebra serves the multi-GPU KV-token
// split (cmt_lse_merge).  The kernel layout is described at tc_attn_db_kernel below.
//
// Softmax uses exp2 (Q arrives pre-multiplied by log2(e)/sqrt(d)).  Two instantiations of the kernel:
//   online  : running row maximum with a lazy rescale -- the maximum is only raised (and O rescaled in TMEM) when
//             it grows by more than 2^8, so the common tile does no accumulator traffic at all;
//   static  : when the caller passes the operand-norm maxima of the projections, |q.k| <= |q||k| bounds every score
//             of a (frame, head); where the bound is <= 60 the weights 2^s need no shift at all (no row maximum, no
//             subtraction, no rescale).  Items above the bound fall to the online kernel.
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "kernels.cuh"

namespace cmt {


// 2^x for x <= ~8 on the FMA/ALU pipes: split x = n + f, f in [-0.5, 0.5] with the 1.5*2^23 rounding trick,
// 2^f by the minimax cubic (relative error 7.5e-5, far below the 2^-9 rounding P gets anyway), 2^n by adding n to the
// exponent field.  Inputs below -125 (masked scores are -inf) clamp to 2^-125, i.e. nothing after rounding.
__device__ __forceinline__ float ex2_poly(float x) {
    x = fmaxf(x, -125.0f);
    const float t = x + 12582912.0f;
    const float n = t - 12582912.0f;
    const float f = x - n;
    float p = fmaf(f, 0.05517167f, 0.24261113f);   // minimax cubic of 2^f on [-0.5, 0.5]: 7.5e-5 relative
    p = fmaf(p, f, 0.69326097f);
    p = fmaf(p, f, 0.99992806f);
    return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}

// The same cubic on a PAIR of inputs with the packed fp32 instructions (FADD2 / FFMA2): 2 clamps, 3 FADD2,
// 3 FFMA2 and 2 integer ops for two exponentials, i.e. ~5 issue slots per exponential and no MUFU slot.
// kClamp = false: the caller guarantees x >= -126 (static-shift path: scores in [-60, 60], masked tail set to -126).
template <bool kClamp = true>
__device__ __forceinline__ void ex2_poly_pair(uint64_t x2, float& e0, float& e1) {
    if (kClamp) {
        float x0, x1;
        unpack_f32x2(x2, x0, x1);
        x2 = pack_f32x2(fmaxf(x0, -125.0f), fmaxf(x1, -125.0f));
    }
    const uint64_t magic = pack_f32x2(12582912.0f, 12582912.0f);
    const uint64_t nmagic = pack_f32x2(-12582912.0f, -12582912.0f);
    const uint64_t m1 = pack_f32x2(-1.0f, -1.0f);
    const uint64_t t2 = add_f32x2(x2, magic);
    const uint64_t n2 = add_f32x2(t2, nmagic);
    const uint64_t f2 = fma_f32x2(n2, m1, x2);   // x - n
    uint64_t p2 = fma_f32x2(f2, pack_f32x2(0.05517167f, 0.05517167f), pack_f32x2(0.24261113f, 0.24261113f));
    p2 = fma_f32x2(p2, f2, pack_f32x2(0.69326097f, 0.69326097f));
    p2 = fma_f32x2(p2, f2, pack_f32x2(0.99992806f, 0.99992806f));
    float p0, p1, t0, t1;
    unpack_f32x2(p2, p0, p1);
    unpack_f32x2(t2, t0, t1);
    e0 = __int_as_float(__float_as_int(p0) + (__float_as_int(t0) << 23));
    e1 = __int_as_float(__float_as_int(p1) + (__float_as_int(t1) << 23));
}

struct TcAttnParams {
    int B, H, Nq;
    int kv_begin, kv_end;
    int T;            // KV tile-steps per item
    int qblk;         // queries per item: 384 (three softmax warpgroups)
    int kt;           // KV tokens per tile-step: 128, or 64 for the double-buffered kernel
    int qblocks;      // ceil(Nq / qblk)
    // Band-aligned stream-K.  Items are ordered query-block-major: item = qb * BH + hb (hb = b * H + h), so that "band" qb
    // is the flat space BH x T of the K/V streams of every (frame, head).  Every full band is cut into n_full equal
    // contiguous ranges, the last band (whose last warpgroups may be idle: cheaper steps) into n_last, one range per CTA:
    // CTA c of band 0 and CTA c of band 1 then walk the SAME K/V tiles at the same time, so each tile comes from DRAM
    // once and from L2 for the other bands (the (frame, head)-major order of round 1 streamed K/V from DRAM once per
    // query block: 3.0x the algorithmic bytes).  n_full : n_last follows the measured step costs (w_full : w_last).
    int BH;           // B * H
    int n_full, n_last;
    int S_max;        // partial slots per item
    float* part_o;    // [items*S_max][qblk][32]
    float* part_lse;  // [items*S_max][qblk]   (log2 domain)
    // key padding mask (attention.py:76-90): bit i of mask_bits[b * T + j] = key kv_begin + 64 j + i of frame b is
    // attended (and < kv_end); nullptr = no mask.  Packed from the byte mask by pack_key_mask_kernel.
    const unsigned long long* mask_bits;
    // static softmax shift: max |q|^2 per (frame, head) [B*H] and max |k|^2 per (frame, head) at
    // k_norm2[b * kn_bstride + h] (written by the projection GEMMs' epilogues); nullptr = online softmax everywhere
    const float* q_norm2;
    const float* k_norm2;
    long long kn_bstride;
    int* unsafe_flags; // [gridDim.x] written by the static kernel (1 = this CTA's range holds items left to the online kernel)
    long long* trace; // debug: clock64 event trace of CTA 0 (three-warpgroup kernel), nullptr = off
};
constexpr int TRACE_STEPS = 96;
#ifdef CMT_ATTN_TRACE
#define CMT_TRACE(wg_, step_, k_)                                                          \
    do {                                                                                   \
        if (p.trace != nullptr && blockIdx.x == 0 && (step_) < TRACE_STEPS)                \
            p.trace[(static_cast<int>(wg_) * TRACE_STEPS + static_cast<int>(step_)) * 16 + (k_)] = clock64(); \
    } while (0)
#else
#define CMT_TRACE(wg_, step_, k_) do { } while (0)
#endif

// First global step (x = item * T + step) of CTA c; c == G gives the end of the space.
__device__ __forceinline__ long long range_start(const TcAttnParams& p, long long c, long long G) {
    const long long S = static_cast<long long>(p.BH) * p.T;
    const long long full_ctas = static_cast<long long>(p.qblocks - 1) * p.n_full;
    if (c >= G) return p.qblocks * S;
    if (c < full_ctas) {
        const long long band = c / p.n_full, local = c - band * p.n_full;
        return band * S + (local * S) / p.n_full;
    }
    return static_cast<long long>(p.qblocks - 1) * S + ((c - full_ctas) * S) / p.n_last;
}
// The CTA whose range contains global step x.
__device__ __forceinline__ int cta_of(const TcAttnParams& p, long long x, long long /*G*/) {
    const long long S = static_cast<long long>(p.BH) * p.T;
    const long long band = x / S, off = x - band * S;
    const long long n = band < p.qblocks - 1 ? p.n_full : p.n_last;
    return static_cast<int>(band * p.n_full + ((off + 1) * n - 1) / S);
}

// ------------------------------------------------------------------------------------------------
// Kernel layout ("db": double-buffered scores).  The event traces of the first schedules (tools/attn_trace.py)
// showed that what keeps the MUFU pipe from saturating is the round trip P stored -> issuer wakes -> PV + next S MMA
// -> softmax wakes (~900 cycles even with a back-to-back issuer) sitting inside every warpgroup's chain.
// Here the KV tile is 64 tokens and every warpgroup owns TWO score buffers, so the scores of step j+1
// (and j+2's, once PV(j) is issued) are already in TMEM while step j is being exponentiated: the
// softmax warps never wait for the tensor pipe in steady state.
//   TMEM: S_i,b at [128 i + 64 b, +64), P_i,b over the first 32 columns of S_i,b, O_i at [384 + 32 i, +32).
//   barriers per warpgroup: s_full[b], p_full[b] (b = step & 1), pv_done (for the rare O rescale, which
//   must not race the previous step's PV), o_full.
//   512 threads: warps 0-11 softmax (one query row per thread, 64 scores in registers), 12 TMA + TMEM
//   allocation, 13-15 one MMA issuer per warpgroup.  No setmaxnreg: 128 registers per thread are enough
//   for 64-column tiles.

// One thread = one 64-key tile of one frame: byte mask -> bit mask, tail beyond kv_end cleared.
__global__ void pack_key_mask_kernel(const unsigned char* keep, unsigned long long* bits, int B, int N_kv, int kv_begin,
                                     int kv_end, int T) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(B) * T) return;
    const int b = static_cast<int>(idx / T), j = static_cast<int>(idx - static_cast<long long>(b) * T);
    const int t0 = kv_begin + j * 64;
    unsigned long long m = 0;
    for (int i = 0; i < 64; ++i) {
        const int t = t0 + i;
        if (t < kv_end && keep[static_cast<long long>(b) * N_kv + t] != 0) m |= 1ull << i;
    }
    bits[idx] = m;
}

namespace attndb {
constexpr int NWG = 3;                  // softmax warpgroups (one 128-row Q tile each)
constexpr int QBLK = NWG * 128;
constexpr int KT = 64;
constexpr int NK = 8, NV = 8;
constexpr int Q_BYTES = 128 * 32 * 2;   // 8 KB per Q tile
constexpr int KV_BYTES = 64 * 32 * 2;   // 4 KB per K tile / V^T tile
// MMA issuer warps.  tools/attn_trace.py (per-warp stamps) shows that the softmax warps which share an SM
// sub-partition with an issuer warp take longer per step than the others, and that the slowest warp of a
// warpgroup sets the period (P needs all four warps).  One issuer per warpgroup spreads that cost over three
// sub-partitions, and the issuers sleep in hardware on their P waits (try_wait with a suspend hint) instead of
// polling: their wake-up latency hides under the double-buffered scores, their issue slots do not.
// Measured (B=8, 56 400 tokens, us per launch): 1 polling issuer 1058, 1 sleeping 1056, 3 polling 992, 3 sleeping 983.
// The TMA producer waits sleep as well; only the softmax warps' wait on their scores polls (mbar_wait).
constexpr int NISS = 3;                                // MMA issuer warps (warpgroup i is served by issuer i % NISS)
constexpr int THREADS = NWG * 128 + 32 + NISS * 32;   // softmax warps, TMA warp, issuer warps
constexpr int OFF_Q = 0;
constexpr int OFF_K = OFF_Q + NWG * Q_BYTES;
constexpr int OFF_V = OFF_K + NK * KV_BYTES;
constexpr int OFF_BAR = OFF_V + NV * KV_BYTES;
constexpr int SMEM_BYTES = OFF_BAR + 1024 + 1024;
constexpr uint32_t COL_O = 384;
constexpr float RESCALE_THRESHOLD = 8.0f;
// With the scores double-buffered and the packed FADD2 softmax, the steady-state step sits within ~7 % of the
// MUFU bound (16 ex2 / clk / SM), so moving exponentials to the FMA pipes pays: pairs i with i % DB_POLY ==
// DB_POLY - 1 of every 16-pair chunk use the packed cubic (ex2_poly_pair).  Measured (B=8, 56 400 tokens, same
// box): off 1100 us, 1/16 1110, 1/8 1056, 1/6 1029, 1/5 1077, 1/4 1106, 1/3 1140, 1/2 1190; with the three sleeping
// issuers (below): off 1041, i%8 969, i%6 958, i%5 946 (shipped: 6 of 32 pairs), i%4 976, i%3 1033.
constexpr int DB_POLY = 5;
// Static softmax shift (see the softmax warps below): items whose Cauchy-Schwarz score bound is at most STATIC_LIMIT
// skip the row maximum and the rescale machinery; their freed ALU / issue slots take more polynomial exponentials.
// Measured with a fixed shift (B=8, 56 400 tokens): online i%5 946 us; static i%5 896, i%4 892, i%3 865.
constexpr int ST_POLY = 3;
// The lone active warp of a tail tile (see lone_warp below).  Measured (B=8, static kernel): every second pair
// polynomial 806 us, all pairs 913.
constexpr int LONE_POLY = 2;
constexpr float STATIC_LIMIT = 60.0f;
// pair i of a 16-pair chunk is polynomial when i % period == period - 1 (period 0: none)
constexpr uint32_t poly_mask(int period) {
    uint32_t m = 0;
    for (int i = 0; i < 16; ++i)
        if (period > 0 && i % period == period - 1) m |= 1u << i;
    return m;
}
constexpr uint32_t ST_MASK = poly_mask(ST_POLY);
constexpr uint32_t DB_MASK = poly_mask(DB_POLY);
constexpr uint32_t LONE_MASK = poly_mask(LONE_POLY);
}  // namespace attndb

// kMask: key padding mask variant (the unmasked instantiation carries none of its code: even an untaken mask
// branch in the softmax loop cost 12 % on the 128-register budget).
// kStatic: static-shift variant.  When the caller supplies the operand norm maxima, BOTH instantiations are launched
// back to back over the same ranges: <kStatic = true> processes the items whose score bound is at most
// STATIC_LIMIT and records per CTA whether it skipped any item; <false> processes exactly those (its CTAs return at
// once when their flag is clear).  Keeping the two softmax loops in separate kernels matters for the same reason as
// kMask: sharing a kernel cost the online loop 8 %.
template <bool kMask, bool kStatic>
__global__ void __launch_bounds__(attndb::THREADS, 1)
tc_attn_db_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_k,
                  const __grid_constant__ CUtensorMap tma_v, const TcAttnParams p) {
    using namespace attndb;
    pdl_trigger();
    if (!kStatic && p.q_norm2 != nullptr) {
        pdl_wait();                                    // the flags are the static kernel's output
        if (p.unsafe_flags[blockIdx.x] == 0) return;   // the static kernel took everything
    }
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
    uint64_t* q_full = bars + 0;
    uint64_t* q_empty = bars + 1;
    uint64_t* k_full = bars + 2;             // [NK]
    uint64_t* k_empty = k_full + NK;         // [NK]
    uint64_t* v_full = k_empty + NK;         // [NV]
    uint64_t* v_empty = v_full + NV;         // [NV]
    uint64_t* s_full = v_empty + NV;         // [NWG][2]
    uint64_t* p_full = s_full + 2 * NWG;     // [NWG][2]
    uint64_t* pv_done = p_full + 2 * NWG;    // [NWG]
    uint64_t* o_full = pv_done + NWG;        // [NWG]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + NWG);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // provably warp-uniform
    const int lane = threadIdx.x & 31;
    constexpr int W_TMA = NWG * 4, W_MMA = W_TMA + 1;   // issuers: W_MMA .. W_MMA + NISS - 1

    if (warp == W_MMA && lane == 0) {
        tma_prefetch_desc(&tma_q);
        tma_prefetch_desc(&tma_k);
        tma_prefetch_desc(&tma_v);
        mbar_init(q_full, 1);
        mbar_init(q_empty, NISS);   // every issuer releases the Q / K / V stages
        for (int s = 0; s < NK; ++s) { mbar_init(&k_full[s], 1); mbar_init(&k_empty[s], NISS); }
        for (int s = 0; s < NV; ++s) { mbar_init(&v_full[s], 1); mbar_init(&v_empty[s], NISS); }
        for (int i = 0; i < NWG; ++i) {
            mbar_init(&s_full[2 * i], 1);
            mbar_init(&s_full[2 * i + 1], 1);
            mbar_init(&p_full[2 * i], 128);
            mbar_init(&p_full[2 * i + 1], 128);
            mbar_init(&pv_done[i], 1);
            mbar_init(&o_full[i], 1);
        }
        fence_barrier_init();
    }
    if (warp == W_TMA) tmem_alloc(tmem_slot, 512);
    pdl_wait();   // barrier init / TMEM allocation / descriptor prefetch overlapped the predecessor's tail
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    const long long t_start = p.trace != nullptr ? clock64() : 0;
    const long long G = gridDim.x;
    const long long pos_begin = range_start(p, blockIdx.x, G);
    const long long pos_end = range_start(p, blockIdx.x + 1, G);
    // Which items are this instantiation's?  Without norms: everything goes to the online kernel.  With norms: the item's
    // Cauchy-Schwarz score bound |q||k| (norms of the fp32 projection outputs; + 2^-7 covers the two bf16 roundings the
    // MMA operands went through) decides.  Every role evaluates the same predicate, so skipped segments touch no barrier.
    auto mine = [&](int item) -> bool {
        if (p.q_norm2 == nullptr) return !kStatic;
        const int hb = item % p.BH;   // b * H + h
        const float bound = sqrtf(__ldg(p.q_norm2 + hb) * __ldg(p.k_norm2 + static_cast<long long>(hb / p.H) * p.kn_bstride + hb % p.H)) * 1.0079f + 1e-3f;
        return (bound <= STATIC_LIMIT) == kStatic;
    };

    if (warp == W_TMA) {
        // ----------------------------- TMA producer -----------------------------
        const bool leader = elect_one();
        uint32_t kc = 0, vc = 0, seg = 0;
        int skipped = 0;
        for (long long pos = pos_begin; pos < pos_end;) {
            const int item = static_cast<int>(pos / p.T);
            const int j0 = static_cast<int>(pos - static_cast<long long>(item) * p.T);
            const int n = static_cast<int>(min(static_cast<long long>(p.T - j0), pos_end - pos));
            if (!mine(item)) { pos += n; skipped = 1; continue; }
            const int qb = item / p.BH;
            const int h = (item % p.BH) % p.H;
            const int b = (item % p.BH) / p.H;
            int nact = (p.Nq - qb * QBLK + 127) >> 7;
            nact = nact > NWG ? NWG : nact;
            mbar_wait_sleep(q_empty, (seg & 1) ^ 1);
            if (leader) {
                mbar_arrive_expect_tx(q_full, nact * Q_BYTES);
                for (int i = 0; i < nact; ++i)
                    tma_load_4d(smem + OFF_Q + i * Q_BYTES, &tma_q, q_full, 0, qb * QBLK + i * 128, h, b);
            }
            // K runs two steps ahead of V: the issuer needs K(j+2) when it retires step j
            const int tok_base = p.kv_begin + j0 * KT;
            for (int jj = 0; jj < n + 2; ++jj) {
                if (jj < n) {
                    const uint32_t ks = kc % NK;
                    mbar_wait_sleep(&k_empty[ks], ((kc / NK) & 1) ^ 1);
                    if (leader) {
                        mbar_arrive_expect_tx(&k_full[ks], KV_BYTES);
                        tma_load_4d(smem + OFF_K + ks * KV_BYTES, &tma_k, &k_full[ks], 0, tok_base + jj * KT, h, b);
                    }
                    ++kc;
                }
                if (jj >= 2) {
                    const uint32_t vs = vc % NV;
                    mbar_wait_sleep(&v_empty[vs], ((vc / NV) & 1) ^ 1);
                    if (leader) {
                        mbar_arrive_expect_tx(&v_full[vs], KV_BYTES);
                        tma_load_4d(smem + OFF_V + vs * KV_BYTES, &tma_v, &v_full[vs], tok_base + (jj - 2) * KT, 0, h, b);
                    }
                    ++vc;
                }
            }
            pos += n;
            ++seg;
        }
        // tell the online kernel whether this CTA's range holds items the static kernel left to it
        if (kStatic && leader && p.unsafe_flags != nullptr) p.unsafe_flags[blockIdx.x] = skipped;
    } else if (warp >= W_MMA && warp < W_MMA + NISS) {
        // ------------- MMA issuers: warp W_MMA + ii serves the warpgroups i with i % NISS == ii -------------
        const int ii = warp - W_MMA;
        const bool leader = elect_one();
        constexpr uint32_t idesc_s = make_idesc_bf16(128, KT);
        constexpr uint32_t idesc_o = make_idesc_bf16(128, 32);
        const uint32_t sq = smem_u32(smem + OFF_Q);
        uint32_t kc = 0, vc = 0, seg = 0;
        uint32_t g[NWG];                       // steps retired per warpgroup (buffer = g & 1, parity = (g >> 1) & 1)
#pragma unroll
        for (int i = 0; i < NWG; ++i) g[i] = 0;
        for (long long pos = pos_begin; pos < pos_end;) {
            const int item = static_cast<int>(pos / p.T);
            const int j0 = static_cast<int>(pos - static_cast<long long>(item) * p.T);
            const int n = static_cast<int>(min(static_cast<long long>(p.T - j0), pos_end - pos));
            if (!mine(item)) { pos += n; continue; }
            const int qb = item / p.BH;
            int nact = (p.Nq - qb * QBLK + 127) >> 7;   // warpgroups with queries; the others only release stages
            nact = nact > NWG ? NWG : nact;
            mbar_wait_sleep(q_full, seg & 1);
            // prologue: scores of steps 0 and 1 into the two buffers
            for (int pre = 0; pre < 2 && pre < n; ++pre) {
                const uint32_t ks = kc % NK;
                mbar_wait_sleep(&k_full[ks], (kc / NK) & 1);
                tc_fence_after();
                if (leader) {
                    const uint64_t kdesc = make_kmajor_desc(smem_u32(smem + OFF_K + ks * KV_BYTES), 64);
#pragma unroll
                    for (int i = 0; i < NWG; ++i) {
                        if ((i % NISS) == ii && i < nact) {
                            const uint32_t bsel = (g[i] + pre) & 1;
                            const uint64_t qdesc = make_kmajor_desc(sq + i * Q_BYTES, 64);
                            tc_mma_ss(tmem_base + i * 128 + bsel * 64, qdesc, kdesc, idesc_s, 0);
                            tc_mma_ss(tmem_base + i * 128 + bsel * 64, qdesc + 2, kdesc + 2, idesc_s, 1);
                            tc_commit(&s_full[2 * i + bsel]);
                        }
                    }
                    tc_commit(&k_empty[ks]);
                    if (pre + 1 == n) tc_commit(q_empty);
                }
                __syncwarp();
                ++kc;
            }
            for (int jj = 0; jj < n; ++jj) {
                const bool has2 = (jj + 2 < n);
                const uint32_t vs = vc % NV;
                const uint32_t ks = kc % NK;
                if (leader) CMT_TRACE(ii, g[ii], 6);
                mbar_wait_sleep(&v_full[vs], (vc / NV) & 1);
                if (has2) mbar_wait_sleep(&k_full[ks], (kc / NK) & 1);
                if (leader) CMT_TRACE(ii, g[ii], 7);
                const uint64_t vdesc = make_kmajor_desc(smem_u32(smem + OFF_V + vs * KV_BYTES), 128);
                const uint64_t kdesc = make_kmajor_desc(smem_u32(smem + OFF_K + ks * KV_BYTES), 64);
#pragma unroll
                for (int i = 0; i < NWG; ++i) {
                    if ((i % NISS) == ii && i < nact) {
                        const uint32_t bsel = g[i] & 1;
                        if (leader) CMT_TRACE(i, g[i], 11);
                        mbar_wait_sleep(&p_full[2 * i + bsel], (g[i] >> 1) & 1);
                        tc_fence_after();
                        if (leader) {
                            CMT_TRACE(i, g[i], 4);
                            const uint32_t t_sp = tmem_base + i * 128 + bsel * 64;
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk)
                                tc_mma_ts(tmem_base + COL_O + i * 32, t_sp + kk * 8, vdesc + ((kk * 32) >> 4), idesc_o,
                                          (jj > 0 || kk > 0) ? 1u : 0u);
                            if (jj + 1 == n) tc_commit(&o_full[i]);
                            else tc_commit(&pv_done[i]);
                            if (has2) {
                                const uint64_t qdesc = make_kmajor_desc(sq + i * Q_BYTES, 64);
                                tc_mma_ss(t_sp, qdesc, kdesc, idesc_s, 0);
                                tc_mma_ss(t_sp, qdesc + 2, kdesc + 2, idesc_s, 1);
                                tc_commit(&s_full[2 * i + bsel]);
                            }
                            CMT_TRACE(i, g[i], 5);
                        }
                        __syncwarp();
                        ++g[i];
                    }
                }
                if (leader) {
                    tc_commit(&v_empty[vs]);
                    if (has2) {
                        tc_commit(&k_empty[ks]);
                        if (jj + 3 == n) tc_commit(q_empty);
                    }
                }
                __syncwarp();
                ++vc;
                if (has2) ++kc;
            }
            pos += n;
            ++seg;
        }
    } else {
        // --------------------------- softmax warpgroups ---------------------------
        const int wg = warp >> 2;                       // Q tile of the item
        const int r = (warp & 3) * 32 + lane;           // row inside the 128-row tile == TMEM lane
        const uint32_t lane_base = static_cast<uint32_t>((warp & 3) * 32) << 16;
        const uint32_t t_s = tmem_base + lane_base + wg * 128;   // + 64 * buffer
        const uint32_t t_o = tmem_base + lane_base + COL_O + wg * 32;
        uint64_t* my_s_full = s_full + 2 * wg;
        uint64_t* my_p_full = p_full + 2 * wg;
        const bool tracer = (threadIdx.x & 127) == 0;
        (void)tracer;
        uint32_t g = 0, seg = 0, pv_base = 0;   // pv_base: pv_done phases of the earlier segments (n - 1 each)
        for (long long pos = pos_begin; pos < pos_end;) {
            const int item = static_cast<int>(pos / p.T);
            const int j0 = static_cast<int>(pos - static_cast<long long>(item) * p.T);
            const int n = static_cast<int>(min(static_cast<long long>(p.T - j0), pos_end - pos));
            const int qb = item / p.BH;
            pos += n;
            if (!mine(item)) continue;
            if (qb * QBLK + wg * 128 >= p.Nq) continue;     // this warpgroup's tile is past the last query
            if (qb * QBLK + wg * 128 + (warp & 3) * 32 >= p.Nq) {
                // all 32 rows of this warp are past the last query (900 queries: three warps of the eighth tile):
                // keep the barrier protocol in step, skip the exponentials -- the MUFU pipe is the bound
                for (int jj = 0; jj < n; ++jj, ++g) {
                    mbar_wait(&my_s_full[g & 1], (g >> 1) & 1);
                    mbar_arrive(&my_p_full[g & 1]);
                }
                mbar_wait(&o_full[wg], seg & 1);
                ++seg;
                pv_base += n - 1;
                continue;
            }
            const int hb = item % p.BH;                     // b * H + h
            const unsigned long long* mask_row = kMask ? p.mask_bits + static_cast<long long>(hb / p.H) * p.T : nullptr;
            float m = -INFINITY, l = 0.0f;

            // One KV step of this thread's row.
            auto step = [&](auto poly_tag, int jj) {
                // bit i of PMASK: pair i of each 16-pair chunk takes its two exponentials through the packed cubic on the
                // FMA pipes instead of the MUFU
                constexpr uint32_t PMASK = decltype(poly_tag)::value;
                const uint32_t bsel = g & 1;
                const uint32_t t_sb = t_s + bsel * 64;
                mbar_wait(&my_s_full[bsel], (g >> 1) & 1);
                if (tracer) CMT_TRACE(wg, g, 0);
                tc_fence_after();
                uint32_t s[2][32];
                tmem_ld32(t_sb + 0, s[0]);
                tmem_ld32(t_sb + 32, s[1]);
                tc_wait_ld();
                if (tracer) CMT_TRACE(wg, g, 1);
                const int valid = p.kv_end - (p.kv_begin + (j0 + jj) * KT);
                if (kMask) {
                    // padded keys (and the tail past kv_end, folded into the bit mask) score -inf
                    const unsigned long long mb = __ldg(mask_row + j0 + jj);
                    const uint32_t mlo = static_cast<uint32_t>(mb), mhi = static_cast<uint32_t>(mb >> 32);
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        if (!((mlo >> i) & 1u)) s[0][i] = 0xff800000u;
                        if (!((mhi >> i) & 1u)) s[1][i] = 0xff800000u;
                    }
                } else if (valid < KT) {
                    // keys past kv_end: -inf, or -126 on the static path (2^-126 against weights >= 2^-60 is nothing,
                    // and the polynomial exponentials there run without their underflow clamp)
                    const uint32_t gone = kStatic ? 0xc2fc0000u : 0xff800000u;
#pragma unroll
                    for (int c = 0; c < 2; ++c)
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if (c * 32 + i >= valid) s[c][i] = gone;
                }
                if (!kStatic) {
                    float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        mx0 = fmaxf(mx0, __uint_as_float(s[0][i]));
                        mx1 = fmaxf(mx1, __uint_as_float(s[0][16 + i]));
                        mx2 = fmaxf(mx2, __uint_as_float(s[1][i]));
                        mx3 = fmaxf(mx3, __uint_as_float(s[1][16 + i]));
                    }
                    const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
                    if (jj == 0) {
                        // O_i is overwritten by the first PV of the segment: nothing to rescale.  A first tile whose
                        // keys are all padding has mx = -inf: keep m finite so that x - m stays -inf (weight 0).
                        m = kMask ? fmaxf(mx, -1e30f) : mx;
                    } else {
                        const bool need = (mx - m) > RESCALE_THRESHOLD;
                        if (__any_sync(0xffffffffu, need)) {
                            // PV(step - 1) may still be accumulating into O_i: wait for it before touching O_i
                            mbar_wait(&pv_done[wg], (pv_base + jj - 1) & 1);
                            tc_fence_after();
                            const float m_new = need ? mx : m;
                            const float alpha = ex2_approx(m - m_new);
                            l *= alpha;
                            uint32_t o[32];
                            tmem_ld32(t_o, o);
                            tc_wait_ld();
#pragma unroll
                            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
                            tmem_st32(t_o, o);
                            m = m_new;
                        }
                    }
                }
                if (tracer) CMT_TRACE(wg, g, 2);
                // x - m and the row sums as packed fp32 pairs (FADD2): half the issue slots of scalar FADDs.
                // One PAIR of exponentials in POLY runs on the FMA pipes (packed cubic) instead of the MUFU; without
                // the row-max work there are issue slots for more of them.
                const uint64_t neg_m2 = pack_f32x2(-m, -m);
                uint64_t l2 = pack_f32x2(0.f, 0.f);
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    uint32_t pk[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        uint64_t x2 = pack_f32x2(__uint_as_float(s[c][2 * i]), __uint_as_float(s[c][2 * i + 1]));
                        if (!kStatic) x2 = add_f32x2(x2, neg_m2);   // static: |s| <= 60, 2^s needs no shift at all
                        float e0, e1;
                        if ((PMASK >> i) & 1u) {
                            ex2_poly_pair<(!kStatic || kMask)>(x2, e0, e1);
                        } else {
                            float x0, x1;
                            unpack_f32x2(x2, x0, x1);
                            e0 = ex2_approx(x0);
                            e1 = ex2_approx(x1);
                        }
                        l2 = add_f32x2(l2, pack_f32x2(e0, e1));
                        pk[i] = pack_bf16x2(e0, e1);
                    }
                    tmem_st16(t_sb + c * 16, pk);
                }
                float l0, l1;
                unpack_f32x2(l2, l0, l1);
                l += l0 + l1;
                tc_wait_st();
                if (lane == 0) CMT_TRACE(wg, g, (warp & 3) == 0 ? 3 : 7 + (warp & 3));
                tc_fence_before();
                mbar_arrive(&my_p_full[bsel]);
                ++g;
            };

            // static variant: every score of the item lies in [-STATIC_LIMIT, STATIC_LIMIT] (see `mine`), so the weights
            // 2^s are normal numbers as they are: the softmax is shift-invariant, hence no row maximum, no subtraction
            // and no rescale of O; the partial's LSE is just log2 of the sum (m = 0).
            if (kStatic) m = 0.0f;
            // A tile with at most 32 queries (the 4-query tail of 900 = 7 * 128 + 4) has ONE active warp, and that warp
            // shares its sub-partition's MUFU with the full tile next door: the pass is then bound by that one
            // sub-partition (trace: 957 of 1165 cycles per step in the shared warp).  The lone warp therefore takes every
            // second pair of exponentials (LONE_POLY) through the polynomial on the otherwise idle FMA pipes and leaves
            // more of the MUFU to its neighbour.
            const bool lone_warp = p.Nq - (qb * QBLK + wg * 128) <= 32;
            // A software-pipelined static loop over the two 32-column halves measured slower (DESIGN.md §3, round 2).
            if (lone_warp) {
                for (int jj = 0; jj < n; ++jj) step(std::integral_constant<uint32_t, LONE_MASK>{}, jj);
            } else {
                for (int jj = 0; jj < n; ++jj) step(std::integral_constant<uint32_t, (kStatic ? ST_MASK : DB_MASK)>{}, jj);
            }
            // segment epilogue: normalised partial + log2-sum-exp into the workspace
            mbar_wait(&o_full[wg], seg & 1);
            ++seg;
            pv_base += n - 1;
            tc_fence_after();
            uint32_t o[32];
            tmem_ld32(t_o, o);
            tc_wait_ld();
            const int slot = item * p.S_max + (static_cast<int>(blockIdx.x) - cta_of(p, static_cast<long long>(item) * p.T, G));
            const long long prow = static_cast<long long>(slot) * QBLK + wg * 128 + r;
            const float inv = l > 0.0f ? 1.0f / l : 0.0f;   // l == 0: every key of the segment was padding
            float4* dst = reinterpret_cast<float4*>(p.part_o + prow * 32);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                dst[i] = make_float4(__uint_as_float(o[4 * i]) * inv, __uint_as_float(o[4 * i + 1]) * inv,
                                     __uint_as_float(o[4 * i + 2]) * inv, __uint_as_float(o[4 * i + 3]) * inv);
            p.part_lse[prow] = m + log2f(l);
            tc_fence_before();
        }
    }

    tc_fence_before();
    __syncthreads();
    if (p.trace != nullptr && threadIdx.x == 0) p.trace[3 * TRACE_STEPS * 16 + blockIdx.x] = clock64() - t_start;
    if (warp == W_TMA) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}


// Merge the per-CTA segments of each item.  One block = 32 rows of one item, one thread = (row, 4 output dims); the
// item's segment count (two 64-bit divisions) is computed once per block, not per thread (17 -> ~5 us per launch).
template <bool kBf16>
__global__ void __launch_bounds__(256) tc_attn_merge_kernel(TcAttnParams p, long long G, void* o,
                                                            float* lse) {
    __shared__ int nseg_s;
    pdl_trigger();
    pdl_wait();
    const int QB = p.qblk;
    const int chunks = QB / 32;                       // blocks per item
    const int item = blockIdx.x / chunks;
    const int rr = (blockIdx.x - item * chunks) * 32 + (threadIdx.x >> 3);
    const int q4 = threadIdx.x & 7;
    const int qb = item / p.BH;
    const int row = qb * QB + rr;
    if (qb * QB + (rr & ~31) >= p.Nq) return;         // the whole block is padding (block-uniform)
    if (threadIdx.x == 0) {
        const long long x0 = static_cast<long long>(item) * p.T;
        nseg_s = cta_of(p, x0 + p.T - 1, G) - cta_of(p, x0, G) + 1;
    }
    __syncthreads();
    if (row >= p.Nq) return;
    const int nseg = nseg_s;
    const int h = (item % p.BH) % p.H;
    const int b = (item % p.BH) / p.H;
    float mx = -INFINITY;
    for (int s = 0; s < nseg; ++s)
        mx = fmaxf(mx, p.part_lse[(static_cast<long long>(item) * p.S_max + s) * QB + rr]);
    float den = 0.f;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < nseg; ++s) {
        const long long prow = (static_cast<long long>(item) * p.S_max + s) * QB + rr;
        const float w = (mx == -INFINITY) ? 0.f : exp2f(p.part_lse[prow] - mx);   // -inf: no attended key at all
        den += w;
        const float4 x = reinterpret_cast<const float4*>(p.part_o + prow * 32)[q4];
        acc.x = fmaf(w, x.x, acc.x);
        acc.y = fmaf(w, x.y, acc.y);
        acc.z = fmaf(w, x.z, acc.z);
        acc.w = fmaf(w, x.w, acc.w);
    }
    const float inv = den > 0.f ? 1.0f / den : 0.f;
    acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
    const long long oidx = ((static_cast<long long>(b) * p.Nq + row) * p.H + h) * 8 + q4;  // float4 units
    if (kBf16) {
        uint2 w;
        w.x = pack_bf16x2(acc.x, acc.y);
        w.y = pack_bf16x2(acc.z, acc.w);
        reinterpret_cast<uint2*>(o)[oidx] = w;
    } else {
        reinterpret_cast<float4*>(o)[oidx] = acc;
    }
    if (lse != nullptr && q4 == 0)
        lse[(static_cast<long long>(b) * p.H + h) * p.Nq + row] = (mx + log2f(den)) * 0.6931471805599453f;
}

// Work plan.  G = number of weighted ranges = CTAs.
// (An "independent warpgroup" variant -- one K/V stream per warpgroup, items of 128 queries, 3 ranges per CTA -- was
// built and measured in round 1: parity-green but 1108 vs 973 us.  A 4-query tail tile still loads one SM
// sub-partition with three active warps, so it costs a full tile; see DESIGN.md.)
// static_shift: the call carries operand norms (the static-shift kernel runs the ranges): its full step is cheaper, so
// the chain-bound last query block weighs relatively more... measured optimum 10:7 against 4:3 for the online kernel
// (us per launch, B=8: static 842 @10:7 vs 858 @4:3; online 951 @4:3 vs 961 @10:7).
static void attn_plan(int B, int H, int Nq, int n_tok, int sms, bool static_shift, TcAttnParams* p, int* grid,
                      long long* slots_out) {
    p->qblk = attndb::QBLK;
    p->kt = attndb::KT;
    p->qblocks = (Nq + p->qblk - 1) / p->qblk;
    p->T = (n_tok + p->kt - 1) / p->kt;
    p->BH = B * H;
    const int rows_last = Nq - (p->qblocks - 1) * p->qblk;
    // with every warpgroup active a step is MUFU-bound; with an idle warpgroup it is bound by one warpgroup's
    // own chain, ~3/4 of that
    constexpr long long ST_WFULL = 10, ST_WLAST = 7;   // static-shift kernel
    constexpr long long ON_WFULL = 4, ON_WLAST = 3;    // online kernel
    const long long w_full = static_shift ? ST_WFULL : ON_WFULL;
    const long long w_last = (rows_last + 127) / 128 < attndb::NWG ? (static_shift ? ST_WLAST : ON_WLAST) : w_full;
    const long long S = static_cast<long long>(p->BH) * p->T;   // steps of one band
    const int nbf = p->qblocks - 1;                              // full bands
    long long n_full = 0, n_last = sms;
    if (nbf > 0) {
        n_full = (sms * w_full + (w_full * nbf + w_last) / 2) / (w_full * nbf + w_last);   // CTAs per band ~ its share of the time
        if (n_full * nbf > sms - 1) n_full = (sms - 1) / nbf;
        if (n_full < 1) n_full = 1;
        n_last = sms - n_full * nbf;
        if (n_last < 1) n_last = 1;
    }
    if (n_full > S) n_full = S;   // no empty ranges
    if (n_last > S) n_last = S;
    p->n_full = static_cast<int>(n_full);
    p->n_last = static_cast<int>(n_last);
    const long long ctas = n_full * nbf + n_last;
    const long long G = ctas;
    long long len_min = S / n_last;
    if (nbf > 0 && S / n_full < len_min) len_min = S / n_full;
    if (len_min < 1) len_min = 1;
    p->S_max = static_cast<int>((p->T - 1) / len_min + 2);
    *grid = static_cast<int>(ctas);
    *slots_out = G;
}

// Debug hook: device buffer of 3 * TRACE_STEPS * 16 + 148 int64.  Every CTA of tc_attn_db_kernel writes its total
// cycle count into the last 148 entries (gives the SM clock under load); with -DCMT_ATTN_TRACE
// (`make EXTRA=-DCMT_ATTN_TRACE`) CTA 0 also fills the per-step clock64 stamps (tools/attn_trace.py).
// nullptr switches it off.
static long long* g_trace_buf[64] = {};   // per device; written only by the diagnostic entry below
int tc_attn_set_timing_buffer(long long* dev_buf) { g_trace_buf[current_device()] = dev_buf; return CMT_OK; }

size_t tc_attn_workspace_bytes(int B, int H, int Nq, int n_kv_tokens) {
    if (B <= 0 || H <= 0 || Nq <= 0 || n_kv_tokens <= 0) return 0;
    TcAttnParams p{}, p2{};
    int grid;
    long long G;
    attn_plan(B, H, Nq, n_kv_tokens, device_sm_count(), false, &p, &grid, &G);
    attn_plan(B, H, Nq, n_kv_tokens, device_sm_count(), true, &p2, &grid, &G);
    if (p2.S_max > p.S_max) p.S_max = p2.S_max;   // either plan fits
    const size_t slots = static_cast<size_t>(B) * H * p.qblocks * p.S_max;
    // partials + alignment + the packed key mask (used only when a key_padding_mask is given) + per-CTA flags
    return slots * p.qblk * 33 * sizeof(float) + 256 + static_cast<size_t>(B) * p.T * 8 + 8 + static_cast<size_t>(grid) * 4 + 16;
}

int launch_tc_attn(const AttnArgs& a, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    const int n_tok = a.kv_end - a.kv_begin;
    CMT_CHECK_ARG(n_tok > 0, "cmt_cross_attn_fwd: empty token range");
    CMT_CHECK_ARG(a.q_ld % 8 == 0 && a.v_ld % 8 == 0 && a.k_bstride % 8 == 0 && a.k_hstride % 8 == 0 &&
                      a.v_bstride % 8 == 0 && a.v_hstride % 8 == 0,
                  "cmt_cross_attn_fwd(bf16): strides must be multiples of 8 elements");
    CMT_CHECK_ARG(((reinterpret_cast<uintptr_t>(a.q) | reinterpret_cast<uintptr_t>(a.k) |
                    reinterpret_cast<uintptr_t>(a.vt) | reinterpret_cast<uintptr_t>(a.o)) & 15) == 0,
                  "cmt_cross_attn_fwd(bf16): pointers must be 16-byte aligned");
    TcAttnParams p{};
    int grid;
    long long G;
    attn_plan(a.B, a.H, a.Nq, n_tok, device_sm_count(), a.q_norm2 != nullptr && a.k_norm2 != nullptr, &p, &grid, &G);
    p.B = a.B;
    p.H = a.H;
    p.Nq = a.Nq;
    p.kv_begin = a.kv_begin;
    p.kv_end = a.kv_end;
    const size_t need = tc_attn_workspace_bytes(a.B, a.H, a.Nq, n_tok);
    if (workspace == nullptr || workspace_bytes < need) {
        set_error("cmt_cross_attn_fwd: workspace too small (%zu < %zu)", workspace_bytes, need);
        return CMT_ERR_WORKSPACE;
    }
    const size_t slots = static_cast<size_t>(a.B) * a.H * p.qblocks * p.S_max;
    uintptr_t wsp = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255);
    p.part_o = reinterpret_cast<float*>(wsp);
    p.part_lse = p.part_o + slots * p.qblk * 32;
    p.trace = g_trace_buf[current_device()];
    p.q_norm2 = (a.q_norm2 != nullptr && a.k_norm2 != nullptr) ? a.q_norm2 : nullptr;
    p.k_norm2 = a.k_norm2;
    p.kn_bstride = a.kn_bstride;
    p.mask_bits = nullptr;
    uintptr_t tail = (reinterpret_cast<uintptr_t>(p.part_lse + slots * p.qblk) + 7) & ~uintptr_t(7);
    if (a.key_keep != nullptr) {
        unsigned long long* bits = reinterpret_cast<unsigned long long*>(tail);
        const long long n = static_cast<long long>(a.B) * p.T;
        pack_key_mask_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, stream>>>(a.key_keep, bits, a.B, a.N_kv, a.kv_begin,
                                                                                a.kv_end, p.T);
        CMT_LAUNCH_CHECK("cmt_cross_attn_fwd(mask)");
        p.mask_bits = bits;
    }
    p.unsafe_flags = reinterpret_cast<int*>(tail + static_cast<size_t>(a.B) * p.T * 8 + 8);

    static DeviceOnce attr_once;
    int attr_dev;
    if (attr_once.need(&attr_dev)) {
        const void* fns[4] = {reinterpret_cast<const void*>(&tc_attn_db_kernel<false, false>),
                              reinterpret_cast<const void*>(&tc_attn_db_kernel<false, true>),
                              reinterpret_cast<const void*>(&tc_attn_db_kernel<true, false>),
                              reinterpret_cast<const void*>(&tc_attn_db_kernel<true, true>)};
        for (const void* f : fns) {
            cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, attndb::SMEM_BYTES);
            if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(tc_attn_db)");
        }
        attr_once.mark(attr_dev);
    }
    CUtensorMap tq, tk, tv;
    {
        uint64_t dims[4] = {32, static_cast<uint64_t>(a.Nq), static_cast<uint64_t>(a.H), static_cast<uint64_t>(a.B)};
        uint64_t strides[3] = {static_cast<uint64_t>(a.q_ld) * 2, 64, static_cast<uint64_t>(a.Nq) * a.q_ld * 2};
        uint32_t box[4] = {32, 128, 1, 1};
        int rc = encode_tma_bf16(&tq, a.q, 4, dims, strides, box, 64);
        if (rc) return rc;
    }
    {
        uint64_t dims[4] = {32, static_cast<uint64_t>(a.kv_end), static_cast<uint64_t>(a.H), static_cast<uint64_t>(a.B)};
        uint64_t strides[3] = {64, static_cast<uint64_t>(a.k_hstride) * 2, static_cast<uint64_t>(a.k_bstride) * 2};
        uint32_t box[4] = {32, static_cast<uint32_t>(p.kt), 1, 1};
        int rc = encode_tma_bf16(&tk, a.k, 4, dims, strides, box, 64);
        if (rc) return rc;
    }
    {
        uint64_t dims[4] = {static_cast<uint64_t>(a.kv_end), 32, static_cast<uint64_t>(a.H), static_cast<uint64_t>(a.B)};
        uint64_t strides[3] = {static_cast<uint64_t>(a.v_ld) * 2, static_cast<uint64_t>(a.v_hstride) * 2,
                               static_cast<uint64_t>(a.v_bstride) * 2};
        uint32_t box[4] = {64, 32, 1, 1};
        int rc = encode_tma_bf16(&tv, a.vt, 4, dims, strides, box, 128);
        if (rc) return rc;
    }
    const bool masked = p.mask_bits != nullptr;
    if (p.q_norm2 != nullptr) {
        // static-shift kernel first (items with a score bound <= STATIC_LIMIT), then the online kernel for the rest
        cudaError_t e = masked ? launch_pdl(tc_attn_db_kernel<true, true>, dim3(grid), dim3(attndb::THREADS), attndb::SMEM_BYTES, stream, tq, tk, tv, p)
                               : launch_pdl(tc_attn_db_kernel<false, true>, dim3(grid), dim3(attndb::THREADS), attndb::SMEM_BYTES, stream, tq, tk, tv, p);
        if (e != cudaSuccess) return cuda_fail(e, "cmt_cross_attn_fwd(tcgen05, static shift) launch");
        CMT_LAUNCH_CHECK("cmt_cross_attn_fwd(tcgen05, static shift)");
    }
    {
        cudaError_t e = masked ? launch_pdl(tc_attn_db_kernel<true, false>, dim3(grid), dim3(attndb::THREADS), attndb::SMEM_BYTES, stream, tq, tk, tv, p)
                               : launch_pdl(tc_attn_db_kernel<false, false>, dim3(grid), dim3(attndb::THREADS), attndb::SMEM_BYTES, stream, tq, tk, tv, p);
        if (e != cudaSuccess) return cuda_fail(e, "cmt_cross_attn_fwd(tcgen05) launch");
    }
    CMT_LAUNCH_CHECK("cmt_cross_attn_fwd(tcgen05)");
    const long long mblocks = static_cast<long long>(a.B) * a.H * p.qblocks * (p.qblk / 32);
    CMT_CHECK_ARG(mblocks < (1ll << 31), "cmt_cross_attn_fwd: too many merge blocks");
    if (a.o_bf16)
        launch_pdl(tc_attn_merge_kernel<true>, dim3(static_cast<int>(mblocks)), dim3(256), 0, stream, p, G, a.o, a.lse);
    else
        launch_pdl(tc_attn_merge_kernel<false>, dim3(static_cast<int>(mblocks)), dim3(256), 0, stream, p, G, a.o, a.lse);
    CMT_LAUNCH_CHECK("cmt_cross_attn_fwd(merge)");
    return CMT_OK;
}

}  // namespace cmt
