// cmt_bbox_topk_decode: MultiTaskBBoxCoder.decode_single for every frame of a batch in one launch
// (multi_task_bbox_coder.py:46-141, util.py:37-68, z shift of cmt_head.py:912).
//
// One 1024-thread CTA per frame:
//   0. with a node mask, a frame none of whose nodes is present writes the "nothing kept" state (count 0, zero boxes
//      and scores, label and top-k index -1) and returns;
//   1. score = 1 / (1 + expf(-logit)) of every (query, class) into shared memory as an order-preserving uint32 key
//      (NaN -> one key above +inf, as torch ranks it);
//   2. radix select, four 8-bit digits from the top, finds the K-th largest key; warp-aggregated shared-memory
//      histograms (scores in [0, 1] put nearly every key in one or two bins of the first digit);
//   3. one pass collects every key above it and, through an ordered block scan, the lowest flat indices of the tie
//      group at it;
//   4. a bitonic sort of the <= 1024 (key, ~index) pairs gives descending score, ties by ascending flat index
//      (= torch.sort(descending=True, stable=True));
//   5. one thread per slot gathers and denormalises its box and applies the centre-range / score mask;
//   6. a block scan compacts the kept slots; the rest is zero with label -1.
// Arithmetic is the eager path's: expf / atan2f without fast-math, and the z shift rounds its product before the
// subtraction, so every output value is the one torch computes on the same device.
#include "kernels.cuh"

namespace cmt {

static constexpr int DEC_THREADS = 1024;

struct DecodeTask {
    const float* cls;      // [B, Nq, n_cls]
    const float* center;   // [B, Nq, 2]
    const float* height;   // [B, Nq, 1]
    const float* dim;      // [B, Nq, 3]
    const float* rot;      // [B, Nq, 2]
    const float* vel;      // [B, Nq, 2]
    int n_cls;
};

struct DecodeParams {
    DecodeTask task[CMT_BOX_DECODE_MAX_TASKS];
    int class_begin[CMT_BOX_DECODE_MAX_TASKS + 1];   // first concatenated class of each task
    int T, Nq, C, N, K, P;                            // P: K rounded up to a power of two (sort width)
    float pcr[6];
    float thr;
    int use_thr, bottom_center;
    float* boxes;
    float* scores;
    long long* labels;
    int* count;
    long long* topk_index;
    const uint8_t* node_valid;   // [n_nodes, B] or nullptr: a frame none of whose nodes delivered keeps nothing
    int n_nodes;
};

// torch's CUDA sigmoid for fp32: one / (one + std::exp(-a))
static __device__ __forceinline__ float sigmoid_ref(float x) { return 1.0f / (1.0f + expf(-x)); }

static __device__ __forceinline__ uint32_t order_key(float s) {
    uint32_t u = __float_as_uint(s);
    if (s != s) u = 0x7fffffffu;   // every NaN: sign cleared, one value, above +inf
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

static __device__ __forceinline__ int task_of(const DecodeParams& p, int c) {
    int t = 0;
    while (t + 1 < p.T && c >= p.class_begin[t + 1]) ++t;
    return t;
}

// Inclusive scan of v over the block's 1024 threads; *total = sum over the block.  Every thread must call it.
static __device__ __forceinline__ uint32_t block_scan(uint32_t v, uint32_t* warp_sums, uint32_t* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = warp_sums[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        warp_sums[lane] = w;
    }
    __syncthreads();
    const uint32_t r = x + (warp > 0 ? warp_sums[warp - 1] : 0u);
    *total = warp_sums[31];
    __syncthreads();   // warp_sums may be reused by the next call
    return r;
}

// The node-mask check and the empty-frame store, out of line: inlined, they raise the kernel from 37 to 40 registers.
static __device__ __noinline__ bool frame_present(const DecodeParams& p, int b) {
    bool any = false;
    for (int i = 0; i < p.n_nodes; ++i) any |= p.node_valid[static_cast<long long>(i) * gridDim.x + b] != 0;
    return any;
}
static __device__ __noinline__ void write_empty_frame(const DecodeParams& p, int b, int tid) {
    if (tid < p.K) {
        const long long o = static_cast<long long>(b) * p.K + tid;
        for (int j = 0; j < 9; ++j) p.boxes[o * 9 + j] = 0.0f;
        p.scores[o] = 0.0f;
        p.labels[o] = -1;
        p.topk_index[o] = -1;
    }
    if (tid == 0) p.count[b] = 0;
}

__global__ void __launch_bounds__(DEC_THREADS, 1) bbox_topk_decode_kernel(const __grid_constant__ DecodeParams p) {
    extern __shared__ __align__(16) unsigned char dsm[];
    unsigned long long* cand = reinterpret_cast<unsigned long long*>(dsm);         // [P] (key << 32) | ~index
    uint32_t* keys = reinterpret_cast<uint32_t*>(dsm + sizeof(unsigned long long) * p.P);   // [N]
    __shared__ uint32_t hist[256];
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t s_digit, s_above, s_nsel;

    const int tid = threadIdx.x, lane = tid & 31;
    const int b = blockIdx.x;
    const int N = p.N, C = p.C, K = p.K;

    // 0. a frame none of whose nodes delivered
    if (p.node_valid != nullptr && !frame_present(p, b)) {
        write_empty_frame(p, b, tid);
        return;
    }

    // 1. keys
    for (int n = tid; n < N; n += DEC_THREADS) {
        const int q = n / C, c = n - q * C;
        const int t = task_of(p, c);
        const DecodeTask& tk = p.task[t];
        const float x = tk.cls[(static_cast<long long>(b) * p.Nq + q) * tk.n_cls + (c - p.class_begin[t])];
        keys[n] = order_key(sigmoid_ref(x));
    }

    // 2. radix select of the K-th largest key: after digit d, `prefix` holds its top digits and `remaining` is its rank
    //    among the keys that share them
    uint32_t prefix = 0, pmask = 0, remaining = static_cast<uint32_t>(K);
    for (int shift = 24; shift >= 0; shift -= 8) {
        if (tid < 256) hist[tid] = 0;
        __syncthreads();   // also orders step 1's stores before the first histogram
        for (int base = 0; base < N; base += DEC_THREADS) {
            const int n = base + tid;
            uint32_t bin = 256;
            if (n < N) {
                const uint32_t k = keys[n];
                if ((k & pmask) == prefix) bin = (k >> shift) & 255u;
            }
            const uint32_t peers = __match_any_sync(0xffffffffu, bin);
            if (bin < 256 && lane == __ffs(peers) - 1) atomicAdd(&hist[bin], static_cast<uint32_t>(__popc(peers)));
        }
        __syncthreads();
        // thread i < 256 looks at digit 255 - i: cum = keys with this digit or a larger one
        const uint32_t h = tid < 256 ? hist[255 - tid] : 0u;
        uint32_t total;
        const uint32_t cum = block_scan(h, warp_sums, &total);
        if (tid < 256 && cum >= remaining && cum - h < remaining) {
            s_digit = 255u - tid;
            s_above = cum - h;
        }
        __syncthreads();
        prefix |= s_digit << shift;
        pmask |= 255u << shift;
        remaining -= s_above;
        __syncthreads();   // s_digit / s_above / hist are rewritten by the next digit
    }
    const uint32_t kth = prefix;   // the K-th largest key; `remaining` (>= 1) of its ties are taken

    // 3. candidates: every key above kth, and the `remaining` lowest flat indices of the keys equal to it
    if (tid == 0) s_nsel = 0;
    uint32_t eq_seen = 0;
    __syncthreads();
    for (int base = 0; base < N; base += DEC_THREADS) {
        const int n = base + tid;
        const uint32_t k = n < N ? keys[n] : 0u;
        const bool gt = n < N && k > kth;
        const bool eq = n < N && k == kth;
        uint32_t n_eq;
        const uint32_t rank = block_scan(eq ? 1u : 0u, warp_sums, &n_eq);   // inclusive: 1 for the first tie here
        if (gt || (eq && eq_seen + rank <= remaining)) {
            const uint32_t pos = atomicAdd(&s_nsel, 1u);
            cand[pos] = (static_cast<unsigned long long>(k) << 32) | static_cast<uint32_t>(~static_cast<uint32_t>(n));
        }
        eq_seen += n_eq;
    }
    // padding sorts last: no real entry is 0 (the smallest key, of -inf, is 0x007fffff)
    for (int i = K + tid; i < p.P; i += DEC_THREADS) cand[i] = 0ull;

    // 4. bitonic sort, descending
    for (int size = 2; size <= p.P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            const int i = tid, j = tid ^ stride;
            if (i < p.P && j > i) {
                const unsigned long long a = cand[i], c2 = cand[j];
                const bool desc = (i & size) == 0;
                if ((a < c2) == desc) {
                    cand[i] = c2;
                    cand[j] = a;
                }
            }
        }
    }
    __syncthreads();

    // 5. one thread per slot: gather, denormalise, mask
    float box[9];
    float score = 0.0f;
    long long label = -1;
    bool keep = false;
    if (tid < K) {
        const uint32_t n = ~static_cast<uint32_t>(cand[tid]);
        const int q = static_cast<int>(n) / C, c = static_cast<int>(n) - q * C;
        const int t = task_of(p, c);
        const DecodeTask& tk = p.task[t];
        const long long row = static_cast<long long>(b) * p.Nq + q;
        score = sigmoid_ref(tk.cls[row * tk.n_cls + (c - p.class_begin[t])]);
        label = c;
        box[0] = tk.center[row * 2];
        box[1] = tk.center[row * 2 + 1];
        box[2] = tk.height[row];
        box[3] = expf(tk.dim[row * 3]);
        box[4] = expf(tk.dim[row * 3 + 1]);
        box[5] = expf(tk.dim[row * 3 + 2]);
        box[6] = atan2f(tk.rot[row * 2], tk.rot[row * 2 + 1]);
        box[7] = tk.vel[row * 2];
        box[8] = tk.vel[row * 2 + 1];
        keep = box[0] >= p.pcr[0] && box[1] >= p.pcr[1] && box[2] >= p.pcr[2] &&
               box[0] <= p.pcr[3] && box[1] <= p.pcr[4] && box[2] <= p.pcr[5];
        if (p.use_thr) keep = keep && score > p.thr;
        if (p.bottom_center) box[2] = __fsub_rn(box[2], __fmul_rn(box[5], 0.5f));
        p.topk_index[static_cast<long long>(b) * K + tid] = n;
    }

    // 6. compaction in score order
    uint32_t n_keep;
    const uint32_t pos = block_scan(keep ? 1u : 0u, warp_sums, &n_keep);
    const long long out0 = static_cast<long long>(b) * K;
    if (keep) {
        const long long o = out0 + pos - 1;
#pragma unroll
        for (int j = 0; j < 9; ++j) p.boxes[o * 9 + j] = box[j];
        p.scores[o] = score;
        p.labels[o] = label;
    }
    if (tid >= static_cast<int>(n_keep) && tid < K) {
        const long long o = out0 + tid;
#pragma unroll
        for (int j = 0; j < 9; ++j) p.boxes[o * 9 + j] = 0.0f;
        p.scores[o] = 0.0f;
        p.labels[o] = -1;
    }
    if (tid == 0) p.count[b] = static_cast<int>(n_keep);
}

int launch_bbox_topk_decode(const float* const* task_ptrs, const int* task_classes, int T, int B, int Nq, int num_classes,
                            int max_num, const float* post_center_range, float score_threshold, int use_score_threshold,
                            int bottom_center, float* boxes, float* scores, long long* labels, int* count,
                            long long* topk_index, const uint8_t* node_valid, int n_nodes, cudaStream_t stream) {
    CMT_CHECK_ARG(task_ptrs && task_classes && post_center_range, "cmt_bbox_topk_decode: null host array");
    CMT_CHECK_ARG(boxes && scores && labels && count && topk_index, "cmt_bbox_topk_decode: null output");
    CMT_CHECK_ARG(node_valid == nullptr || n_nodes >= 1, "cmt_bbox_topk_decode: node_valid needs n_nodes >= 1 (got %d)",
                  n_nodes);
    CMT_CHECK_ARG(T >= 1 && T <= CMT_BOX_DECODE_MAX_TASKS, "cmt_bbox_topk_decode: %d tasks (1..%d supported)", T,
                  CMT_BOX_DECODE_MAX_TASKS);
    CMT_CHECK_ARG(B >= 1 && Nq >= 1, "cmt_bbox_topk_decode: bad shape B=%d Nq=%d", B, Nq);
    DecodeParams p{};
    long long sum_c = 0;
    for (int t = 0; t < T; ++t) {
        CMT_CHECK_ARG(task_classes[t] >= 1, "cmt_bbox_topk_decode: task %d has %d classes", t, task_classes[t]);
        for (int j = 0; j < 6; ++j)
            CMT_CHECK_ARG(task_ptrs[6 * t + j] != nullptr, "cmt_bbox_topk_decode: null tensor %d of task %d", j, t);
        p.task[t] = DecodeTask{task_ptrs[6 * t], task_ptrs[6 * t + 1], task_ptrs[6 * t + 2], task_ptrs[6 * t + 3],
                               task_ptrs[6 * t + 4], task_ptrs[6 * t + 5], task_classes[t]};
        p.class_begin[t] = static_cast<int>(sum_c);
        sum_c += task_classes[t];
    }
    CMT_CHECK_ARG(sum_c == num_classes, "cmt_bbox_topk_decode: num_classes %d != sum of the tasks' classes %lld",
                  num_classes, sum_c);
    const long long N = static_cast<long long>(Nq) * sum_c;
    CMT_CHECK_ARG(N <= CMT_BOX_DECODE_MAX_CANDIDATES,
                  "cmt_bbox_topk_decode: Nq * num_classes = %lld exceeds %d (the scores of a frame live in shared memory)",
                  N, CMT_BOX_DECODE_MAX_CANDIDATES);
    CMT_CHECK_ARG(max_num >= 1 && max_num <= CMT_BOX_DECODE_MAX_K && max_num <= N,
                  "cmt_bbox_topk_decode: max_num %d must be in [1, min(%d, Nq * num_classes = %lld)]", max_num,
                  CMT_BOX_DECODE_MAX_K, N);
    p.class_begin[T] = static_cast<int>(sum_c);
    p.T = T;
    p.Nq = Nq;
    p.C = num_classes;
    p.N = static_cast<int>(N);
    p.K = max_num;
    p.P = 1;
    while (p.P < max_num) p.P <<= 1;
    for (int i = 0; i < 6; ++i) p.pcr[i] = post_center_range[i];
    p.thr = score_threshold;
    p.use_thr = use_score_threshold ? 1 : 0;
    p.bottom_center = bottom_center ? 1 : 0;
    p.boxes = boxes;
    p.scores = scores;
    p.labels = labels;
    p.count = count;
    p.topk_index = topk_index;
    p.node_valid = node_valid;
    p.n_nodes = n_nodes;
    const size_t smem = sizeof(unsigned long long) * p.P + sizeof(uint32_t) * static_cast<size_t>(N);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(bbox_topk_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(smem));
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(bbox_topk_decode)");
    }
    bbox_topk_decode_kernel<<<B, DEC_THREADS, smem, stream>>>(p);
    CMT_LAUNCH_CHECK("cmt_bbox_topk_decode");
    return CMT_OK;
}

}  // namespace cmt
