// Shared device/host helpers for libcmtcoop_b200 (sm_100a only).
// PTX wrappers for mbarrier / TMA / tcgen05 are written by hand against the PTX ISA;
// nothing from CUTLASS/CuTe is included in the product path.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstdlib>
#include <stdint.h>
#include <cstdio>

#include "../../include/cmtcoop_b200.h"

namespace cmt {

// ---------------------------------------------------------------------------
// error plumbing (no exceptions cross the C ABI)
// ---------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define CMT_CHECK_ARG(cond, ...)                    \
    do {                                            \
        if (!(cond)) {                              \
            ::cmt::set_error(__VA_ARGS__);          \
            return CMT_ERR_BAD_ARG;                 \
        }                                           \
    } while (0)

#define CMT_LAUNCH_CHECK(what)                                   \
    do {                                                         \
        cudaError_t e__ = cudaGetLastError();                    \
        if (e__ != cudaSuccess) return ::cmt::cuda_fail(e__, what); \
    } while (0)

int device_sm_count();
int require_sm100();
int current_device();   // cudaGetDevice clamped to [0, 64)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a per-device (per-context) setting: remember, thread-safely,
// which devices of this process already have it.  Usage:
//     static DeviceOnce once;  int dev;
//     if (once.need(&dev)) { ...cudaFuncSetAttribute...; once.mark(dev); }
// Two threads racing on the same device both set the (idempotent) attribute; nothing else is shared.
struct DeviceOnce {
    unsigned long long done = 0;   // bit d = device d configured (accessed with atomics)
    bool need(int* dev) {
        *dev = current_device();
        return ((__atomic_load_n(&done, __ATOMIC_ACQUIRE) >> *dev) & 1ull) == 0;
    }
    void mark(int dev) { __atomic_fetch_or(&done, 1ull << dev, __ATOMIC_RELEASE); }
};

// Driver entry point for cuTensorMapEncodeTiled, fetched once through the runtime
// (no link-time dependency on libcuda).
// dtype CMT_F32 | CMT_BF16 | CMT_F16, strides_bytes: rank - 1 entries, swizzle_bytes 0 (none) | 32 | 64 | 128
int encode_tma(CUtensorMap* map, const void* base, int dtype, int rank, const uint64_t* dims,
               const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes);

// ---------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// Two values rounded to the 16-bit compute dtype kLp (CMT_F16, else bf16) in one word, `lo` in the low half.
template <int kLp>
__device__ __forceinline__ uint32_t pack_lp2(float lo, float hi) {
    return kLp == CMT_F16 ? pack_f16x2(lo, hi) : pack_bf16x2(lo, hi);
}
// One value of the 16-bit dtype kLp (CMT_F16, else bf16): element i of `base`.
template <int kLp>
__device__ __forceinline__ void store_lp(void* base, long long i, float v) {
    if (kLp == CMT_F16) reinterpret_cast<__half*>(base)[i] = __float2half_rn(v);
    else reinterpret_cast<__nv_bfloat16*>(base)[i] = __float2bfloat16_rn(v);
}
template <int kLp>
__device__ __forceinline__ float load_lp(const void* base, long long i) {
    if (kLp == CMT_F16) return __half2float(reinterpret_cast<const __half*>(base)[i]);
    return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[i]);
}

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Packed fp32 pairs (sm_100 FADD2 / FFMA2): two lanes of work per issue slot.
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

// ------------------- programmatic dependent launch (PDL) -------------------
// A kernel launched with launch_pdl() may begin (scheduling, barrier init, TMEM allocation, descriptor prefetch) while
// its stream predecessor is still draining; pdl_wait() blocks until the predecessor grid has completed and its
// memory is visible, so it must precede every access to data a predecessor may write or still read.  Kernels call
// pdl_trigger() first thing so that their own successor can be scheduled early.  Without the launch attribute both are
// no-ops.  CMT_PDL=0 in the environment turns the attribute off.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

inline bool pdl_enabled() {
    static const bool on = [] {
        const char* e = getenv("CMT_PDL");
        return !(e != nullptr && e[0] == '0');
    }();
    return on;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ------------------------------ mbarrier ----------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
// Plain try_wait.  Also tried: try_wait with a suspend-time hint, 3 % slower on the attention kernel (slower wake-up),
// and test_wait (pure spin).
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// A protocol bug must surface as a launch failure, never as a hung GPU: every wait is bounded
// (try_wait itself suspends for a HW-defined interval, so the bound is tens of seconds).
constexpr uint32_t SPIN_LIMIT = 1u << 24;
#ifdef CMT_TRAP_REPORT
// debug builds: before trapping, record which barrier timed out into a HOST-mapped buffer (it survives the dead context):
// cmt_dbg_host[0] = record count, then 4 words per record: blockIdx | warp << 16, barrier smem offset, parity, line.
// Out of line, so that the wait loops compile as they do with the plain trap.
static __device__ unsigned long long* cmt_dbg_host = nullptr;
static __device__ __noinline__ void cmt_wait_timeout(uint32_t bar_off, uint32_t parity, int line) {
    if ((threadIdx.x & 31) == 0 && cmt_dbg_host != nullptr) {
        const unsigned long long k = atomicAdd(cmt_dbg_host, 1ull);
        if (k < 500) {
            cmt_dbg_host[1 + 4 * k] = blockIdx.x | (static_cast<unsigned long long>(threadIdx.x >> 5) << 16);
            cmt_dbg_host[2 + 4 * k] = bar_off;
            cmt_dbg_host[3 + 4 * k] = parity;
            cmt_dbg_host[4 + 4 * k] = line;
        }
        __threadfence_system();
    }
    __trap();
}
#define CMT_WAIT_TIMEOUT(bar, parity) cmt_wait_timeout(smem_u32(bar) & 0xffff, parity, __LINE__)
#else
#define CMT_WAIT_TIMEOUT(bar, parity) __trap()   // surfaces as cudaErrorLaunchFailure
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > SPIN_LIMIT) CMT_WAIT_TIMEOUT(bar, parity);
    }
}
// Latency-tolerant waiters (producers, issuers that run a buffer ahead): let the hardware suspend the warp
// instead of re-polling, so that the probes do not compete with the softmax warps for issue / MIO slots.
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u)
            : "memory");
        if (ok) break;
        if (++spins > SPIN_LIMIT) CMT_WAIT_TIMEOUT(bar, parity);
    }
}

// -------------------------------- TMA --------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)),
        "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)),
        "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// smem -> global tensor store (bulk async group), used by the GEMM epilogue
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* smem_src, int c0, int c1,
                                             int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
        ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------ tcgen05 ------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(smem_result)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_wait_ld() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_wait_st() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// commit: the mbarrier receives one arrival when every tcgen05.mma issued so far by
// this thread has completed (implies fence::before_thread_sync).
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                     smem_u32(bar))
                 : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, bf16 inputs, fp32 accumulate.
__device__ __forceinline__ void tc_mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A operand read from tensor memory (bf16 pairs packed into 32-bit columns).
__device__ __forceinline__ void tc_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread (thread = lane).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
          "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
          "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
          "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
    return v;
}
__device__ __forceinline__ void tmem_st1(uint32_t taddr, uint32_t v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(v) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]),
        "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]),
        "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]),
        "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]),
        "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]),
        "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
        "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}

// Shared-memory matrix descriptor for a K-major bf16 operand laid out by TMA with a
// 64B or 128B swizzle: rows are `swizzle` bytes long, 8-row groups are contiguous, groups
// are `8*swizzle` bytes apart (SBO).  Bits: [0,14) addr>>4, [16,30) LBO>>4 (ignored for
// swizzled K-major, set to 1), [32,46) SBO>>4, [46,48) version=1, [61,64) layout type.
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr, int swizzle_bytes) {
    const uint64_t layout = (swizzle_bytes == 128) ? 2ull : (swizzle_bytes == 64 ? 4ull : 6ull);
    const uint64_t sbo = static_cast<uint64_t>(8 * swizzle_bytes) >> 4;
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= 1ull << 16;
    d |= sbo << 32;
    d |= 1ull << 46;
    d |= layout << 61;
    return d;
}

// Instruction descriptor: kind::f16, D=fp32, both operands K-major; A=B=bf16 (a/b format 1), or fp16 (format 0).
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, bool fp16) {
    return (1u << 4) | (fp16 ? 0u : (1u << 7) | (1u << 10)) | (static_cast<uint32_t>(N >> 3) << 17) |
           (static_cast<uint32_t>(M >> 4) << 24);
}

template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

}  // namespace cmt
