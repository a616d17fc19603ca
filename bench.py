#!/usr/bin/env python
"""bench.py -- CmtTransformer+PE forward throughput (frames/s), the metric BASELINE.json names.

    python bench.py --gpus N --steps K --warmup W [--workload nusc|coop_lidar|coop_fusion|lidar128] [--batch B]
    python bench.py --impl reference ...      # the reference's CPU path (oracle port), same metric/config; one frame
                                              # per step, 1.65 s per step at nusc on 16 host cores of a B200 box
    python bench.py ... --dump-outputs DIR    # + the task-head outputs of the last timed step as DIR/<name>.npy

A "step" is one forward of the hot path over one batch of synthetic frames: camera-ray PE, BEV PE,
query embeddings, token gather, all-layer K/V projection, the 6-layer decoder (cross-attention on the
tcgen05 flash kernel) and the task heads -- i.e. CmtHead.forward_single from the post-shared_conv BEV
map and the neck's image features (SURVEY.md 8(d) scope).  Default workload: BASELINE.json configs[2]/[4]
shape, nuScenes multimodal (6 cams 40x100 tokens + 180x180 BEV = 56 400 K/V tokens, 900 queries, 6 layers,
d=256, bf16), 8 frames per GPU; frames shard across GPUs with no data-path collective (weak scaling).

One JSON line on stdout (rank 0).  `value` = device-timed throughput with inputs resident in HBM;
`e2e` = the same forward through the public head API from pinned HOST buffers (H2D + D2H in the timed
region); `roofline` is for the dominant kernel (tc_attn_db_kernel); `cpu_baseline` is the CPU oracle on a
bounded sample.  Only the cpu_baseline / --impl reference legs touch oracle/.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from cmtcoop_b200 import synth  # noqa: E402

METRIC = "CmtTransformer+PE fwd frames/sec"
WORKLOADS = {
    # name: (head kind, bev_hw, n_views, description)
    "nusc": ("CmtHead", 180, 6, "CMT nuScenes multimodal: 6 cams 1600x640 stride-16 (6x40x100 tokens) + 180x180 BEV, "
                                "900 queries, 6 layers, d=256 (BASELINE configs[2]/[4])"),
    "coop_lidar": ("CmtLidarHeadCoop", 180, 0, "CMTCoop-L TUMTraf cooperative LiDAR-only: 2 nodes x 180x180 BEV "
                                               "(BASELINE configs[1])"),
    "coop_fusion": ("CmtHeadCoop", 180, 0, "CMTCoop TUMTraf cooperative multimodal: vehicle 1 cam + infrastructure "
                                           "3 cams + 2 LiDAR BEV maps (BASELINE configs[3])"),
    "lidar128": ("CmtLidarHead", 128, 0, "CMT-L LiDAR-only 128x128 BEV (BASELINE configs[0])"),
}


# dram__bytes_read.sum + dram__bytes_write.sum of tc_attn_db_kernel per launch from the committed ncu --set full
# capture (profiles/r2_attn_static_ncu_raw.csv, the static-shift instantiation the bench runs: 850.2 MB read + 11.1 MB
# written at B=8), per frame.  K+V of one layer are 57.8 MB per frame; with the band-aligned partition the first two query
# blocks of a (frame, head) share one pass over K/V through L2 and the third streams them again: 1.86x the algorithmic
# bytes (round 1: 3.0x).
NCU_DRAM_BYTES_PER_FRAME = {"nusc": (850.232832e6 + 11.066368e6) / 8}


def build_case(workload, B, seed=0, in_channels=256):
    kind, bev_hw, n_views, _ = WORKLOADS[workload]
    cfg = synth.head_cfg(kind, num_query=900, num_layers=6, grid=8 * bev_hw)
    cfg["_apply_shared_conv"] = False
    # hot-path scope: the BEV input is the post-shared_conv map (256 channels); in_channels=512: the raw map
    inputs = synth.make_inputs(kind, B=B, bev_hw=bev_hw, n_views=max(n_views, 1), img_hw=(40, 100),
                               in_channels=in_channels, seed=seed)
    return kind, cfg, inputs


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


DUMP_MAX_BYTES = 64 * 10**6   # files written by --dump-outputs, .npy headers included


def host_copy(rets):
    """forward_single's result (one dict per task of [layers, frames, queries, channels] tensors) as fp32 CPU tensors."""
    return [{n: t.detach().float().cpu() for n, t in task.items()} for task in rets]


def dump_outputs(out_dir, rets):
    """Writes every task-head tensor of `rets` as out_dir/task<t>.<name>.npy (float32).  The inputs are seeded, so two
    builds run with the same arguments can be compared file by file.  Only the first frames that fit in
    DUMP_MAX_BYTES are written (every tensor keeps the same frames)."""
    arrays = {f"task{t}.{n}": v for t, task in enumerate(rets) for n, v in task.items()}
    frames = next(iter(arrays.values())).shape[1]
    per_frame = sum(v[:, :1].numel() * 4 for v in arrays.values())
    keep = max(1, min(frames, (DUMP_MAX_BYTES - 256 * len(arrays)) // per_frame))   # an .npy header is <= 256 bytes here
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v[:, :keep].numpy())


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled every 100 ms during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return dict(sm_mhz=med, sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons))


# ---------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference's CPU implementation of the path (oracle port: the verbatim reference needs mmcv/mmdet,
    absent on the box), fp32, nn.MultiheadAttention-style attention, all host threads, one frame per step."""
    if rank != 0:
        return
    from oracle import cmt_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    kind, cfg, inputs = build_case(args.workload, 1)
    from cmtcoop_b200.plugin import build_head
    head = build_head({k: v for k, v in cfg.items() if not k.startswith("_")})
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in
          synth.synth_state_dict({k: tuple(v.shape) for k, v in head.state_dict().items()}).items()}
    del head
    times = []
    with torch.no_grad():
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            rets, _ = O.head_forward(sd, cfg, inputs)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
    per = float(np.mean(times))
    val = 1.0 / per
    line = dict(metric=METRIC, value=val, unit="frames/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=per * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload=WORKLOADS[args.workload][3], frames_per_step=1, precision="fp32",
                            implementation="oracle port of the reference CPU path (nn.MultiheadAttention math)"),
                cpu_baseline=dict(value=val, unit="frames/s", cores=torch.get_num_threads(), kind="port",
                                  sample="1 frame per step"),
                e2e=dict(value=val, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, host_copy(rets))
    print(json.dumps(line), flush=True)


def cpu_baseline_sample(workload):
    """Bounded CPU sample for the default line: ONE frame of the same workload through the oracle."""
    from oracle import cmt_oracle as O
    from cmtcoop_b200.plugin import build_head
    prev_threads = torch.get_num_threads()
    torch.set_num_threads(os.cpu_count() or 1)
    kind, cfg, inputs = build_case(workload, 1)
    head = build_head({k: v for k, v in cfg.items() if not k.startswith("_")})
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in
          synth.synth_state_dict({k: tuple(v.shape) for k, v in head.state_dict().items()}).items()}
    del head
    iters = 6   # ~10 s of host work on the box's cores
    with torch.no_grad():
        O.head_forward(sd, cfg, inputs)   # untimed warm-up (thread pool, allocator)
        t0 = time.perf_counter()
        for _ in range(iters):
            O.head_forward(sd, cfg, inputs)
        dt = (time.perf_counter() - t0) / iters
    cores = torch.get_num_threads()
    torch.set_num_threads(prev_threads)
    return dict(value=1.0 / dt, unit="frames/s", cores=cores, kind="port",
                sample=f"1 frame of the same workload per iteration, 1 warm-up + {iters} timed iterations "
                       f"({dt:.2f} s each), fp32, all host threads")


# ---------------------------------------------------------------------------------------------
FEAT_DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}
# ops.profile_events tags timed per launch inside the eager timed region (CUDA events on the launching stream)
KERNEL_TAGS = ("cross_attn", "ray_pe", "gather_tokens", "k_proj", "v_proj", "rv_pe_mlp.0", "rv_pe_mlp.2")


def frame0_inputs(inputs, B, coop, feat_dtype):
    """Frame 0 of the step's batch as an oracle input dict.  Features are the values the GPU path received
    (rounded to the hand-over dtype), as fp32 numpy."""
    out = dict(img_metas=inputs["img_metas"][:1])
    for k, v in inputs.items():
        if isinstance(v, np.ndarray):
            per = v.shape[0] // B
            t = torch.from_numpy(v[:per]).to(feat_dtype).float()
            out[k] = t.numpy()
        elif k != "img_metas":
            out[k] = v
    return out


def parity_check(cfg, inputs, B, coop, feat_dtype, head, rets):
    """Frame 0 of the timed workload against the CPU oracle (outside every timed region)."""
    from oracle import cmt_oracle as O
    prev_threads = torch.get_num_threads()
    torch.set_num_threads(os.cpu_count() or 1)
    sd = {k: v.detach().float().cpu() for k, v in head.state_dict().items()}
    with torch.no_grad():
        want, _ = O.head_forward(sd, cfg, frame0_inputs(inputs, B, coop, feat_dtype))
    # back to the launcher's thread count (torchrun: OMP_NUM_THREADS=1): a 24-thread intra-op pool left behind turns
    # every small host-side tensor op of the serving loop into an oversubscribed OpenMP region (e2e 8.6 -> 42 ms per step)
    torch.set_num_threads(prev_threads)
    per = {n: O.rel_l2(rets[0][n][:, :1].float().cpu(), want[0][n]) for n in want[0]}
    worst = max(per.values())
    shp = {n: list(want[0][n].shape) for n in ("cls_logits", "center")}
    return dict(rel_l2=worst, per_output=per, tolerance=1e-2, ok=bool(worst < 1e-2),
                checked_shape=f"frame 0 of the timed batch, all 6 decoder layers: cls_logits {shp['cls_logits']}, "
                              f"center {shp['center']} (+ height, dim, rot, vel) vs the fp32 CPU oracle on the same inputs")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="nusc", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=8, help="frames per GPU per step")
    ap.add_argument("--feat-dtype", default="bf16", choices=sorted(FEAT_DTYPES),
                    help="dtype in which the neck's feature maps are handed over (host buffers of the e2e leg, resident "
                         "buffers of the device leg); the gather kernel rounds fp32 features to bf16 on arrival, so the "
                         "outputs are bit-identical for fp32 and bf16 hand-over")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the frame-0 oracle comparison (about 2 s of host work)")
    ap.add_argument("--no-cuda-graph", action="store_true", help="time eager launches instead of CUDA-graph replay")
    ap.add_argument("--kv-split-graph", action="store_true",
                    help="with --kv-split: capture the forward INCLUDING the per-layer NCCL all-gathers in a CUDA graph")
    ap.add_argument("--no-shared-conv-leg", action="store_true", help="skip the second scope (step including shared_conv)")
    ap.add_argument("--kv-split-peer", action="store_true",
                    help="with --kv-split: per-layer exchange + merge as ONE kernel over peer memory (NVLink loads) instead of "
                         "NCCL all-gather + merge")
    ap.add_argument("--kv-split", action="store_true",
                    help="BASELINE configs[4] variant: every rank sees the SAME frames and attends 1/N of the K/V tokens; "
                         "one NCCL all-gather of (O, LSE) per decoder layer + log-sum-exp merge (strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the task-head outputs of the last timed step (rank 0) as DIR/<name>.npy, float32, "
                         "at most 64 MB (the first frames of the batch that fit)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        args.warmup = min(args.warmup, 1)
        run_reference(args, rank, world)
        return

    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    import torch.distributed as dist
    from cmtcoop_b200 import ops
    from cmtcoop_b200.plugin import build_head, fused_decoder
    from cmtcoop_b200.runtime import GraphedForward, PipelinedRunner, numa_local_to_gpu

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch
    fdt = FEAT_DTYPES[args.feat_dtype]
    kv_split = args.kv_split and world > 1
    if kv_split and not (args.kv_split_graph or args.kv_split_peer):
        args.no_cuda_graph = True   # default: the per-layer NCCL all-gather stays outside graph capture (the peer-memory
                                    # exchange is an ordinary kernel and replays from the graph like the rest)
    kind, cfg, inputs = build_case(args.workload, B, seed=0 if kv_split else rank)
    head = build_head({k: v for k, v in cfg.items() if not k.startswith("_")})
    synth.load_synth_weights(head, 0)
    head = head.to(dev).eval().set_precision("bf16")
    head.apply_shared_conv = False
    if kv_split:
        head.transformer.enable_kv_split(peer_memory=args.kv_split_peer)
    coop = kind.endswith("Coop")
    feat_keys = [k for k, v in inputs.items() if isinstance(v, np.ndarray)]
    with numa_local_to_gpu(local_rank) as numa:
        # pinned staging buffers first-touched on the GPU's own NUMA node
        host = {k: torch.from_numpy(inputs[k]).to(fdt).pin_memory() for k in feat_keys}
    resident = {k: v.to(dev) for k, v in host.items()}
    metas = inputs["img_metas"]

    def forward(feats, m=None):
        g = feats.get
        m = metas if m is None else m
        if coop:
            return head.forward_single(g("vehicle_pts_feats"), g("infrastructure_pts_feats"), g("vehicle_img_feats"),
                                       g("infrastructure_img_feats"), m)
        return head.forward_single(g("pts_feats"), g("img_feats"), m)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps between a barrier+sync on both sides, CUDA events on the launching stream; max over ranks.
        Returns the time and what the last step returned."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    with torch.no_grad():
        # ---- device-resident throughput ----
        for _ in range(args.warmup):
            rets = forward(resident)
        # diagnostic pass, OUTSIDE the timed region: per-CTA clock64 totals of the attention kernel (one 8-byte store per
        # CTA) with the event time of the same launch give the SM clock the kernel really ran at -- NVML keeps reporting
        # the maximum clock while the kernel runs power-limited, and the MUFU-floor analysis in DESIGN.md is in cycles
        import ctypes
        from cmtcoop_b200 import _lib
        lib = _lib.load()
        tbuf = torch.zeros(3 * 96 * 16 + 148, dtype=torch.int64, device=dev)
        lib.cmt_debug_attn_timing(ctypes.c_void_p(tbuf.data_ptr()))
        ops.profile_events("cross_attn", True)
        forward(resident)
        diag_ms = ops.profile_events("cross_attn", False)
        lib.cmt_debug_attn_timing(ctypes.c_void_p(0))
        cyc = float(tbuf[3 * 96 * 16:].max().item())   # the last cross-attention launch of the pass
        sm_clock_ghz = cyc / (diag_ms[-1] * 1e-3) / 1e9 if diag_ms and cyc > 0 else None
        # which instantiation do the attention items take?  (static shift iff the operand-norm score bound <= 60)
        static_frac = None
        if fused_decoder.last_norms is not None:
            qn2, kn2 = fused_decoder.last_norms
            kn2 = torch.cat(list(kn2)) if isinstance(kn2, (list, tuple)) else kn2
            bound = torch.sqrt(qn2 * kn2.permute(1, 0, 2)) * 1.0079 + 1e-3
            static_frac = float((bound <= 60.0).float().mean().item())

        sampler = ClockSampler(local_rank)
        sampler.start()
        n0 = ops.launch_count()
        for t in KERNEL_TAGS:
            ops.profile_events(t, True)
        ms_eager, last = timed(lambda: forward(resident), args.steps)
        per_launch = {t: ops.profile_events(t, False) for t in KERNEL_TAGS}
        attn_ms = per_launch["cross_attn"]
        launches = ops.launch_count() - n0
        ms = ms_eager
        # the online-softmax instantiation on the same workload (what a checkpoint with peaky logits would run):
        # per-launch device time only, not part of `value`
        ops.FORCE_ONLINE_SOFTMAX = True
        for _ in range(2):
            forward(resident)
        ops.profile_events("cross_attn", True)
        for _ in range(3):
            forward(resident)
        online_ms = ops.profile_events("cross_attn", False)
        ops.FORCE_ONLINE_SOFTMAX = False
        rets = forward(resident)
        if not args.no_cuda_graph:
            # same forward, same kernels, replayed from a CUDA graph (public API: cmtcoop_b200.runtime.GraphedForward):
            # the eager run above keeps the per-launch kernel timings for the roofline
            graphed = GraphedForward(head, metas, resident, adopt_inputs=True)
            for _ in range(3):
                rets = graphed()
            ms, last = timed(lambda: graphed(), args.steps)
        # what the last timed step returned, copied before a later replay of the graph overwrites it in place
        last = host_copy(last) if args.dump_outputs and rank == 0 else None
        clocks = sampler.stop()
        torch.cuda.synchronize()
        parity = None
        if rank == 0 and not args.no_parity:
            parity = parity_check(cfg, inputs, B, coop, fdt, head, rets)
        barrier()   # rank 0 spent seconds in the CPU oracle: nobody starts a forward whose exchange it would keep waiting

        # ---- end to end: pinned host inputs -> H2D -> forward -> D2H of every task-head tensor ----
        # public serving API: cmtcoop_b200.runtime.PipelinedRunner double-buffers the H2D of step i+1 and
        # the D2H of step i-1 under the compute of step i; every byte still moves inside the timed region
        runner = PipelinedRunner(head, metas, host, dev, use_cuda_graph=not args.no_cuda_graph)
        runner.run([host] * 3)
        torch.cuda.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        runner.run([host] * args.steps)
        e1.record()
        barrier()
        ms_t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
        ms_e2e = float(ms_t.item())
        h2d, d2h = runner.h2d_bytes, runner.d2h_bytes

        # ---- second scope: the same step INCLUDING shared_conv (3x3 conv 512->256 + BN + ReLU on the raw BEV map,
        # cmt_head.py:280-287,481) as the tcgen05 implicit GEMM that writes the BEV tokens ----
        with_conv = None
        if any("pts_feats" in k for k in feat_keys) and not kv_split and not args.no_shared_conv_leg:
            kind2, _, inputs2 = build_case(args.workload, B, seed=rank, in_channels=512)
            res2 = {k: torch.from_numpy(inputs2[k]).to(fdt).to(dev) for k in feat_keys}
            metas2 = inputs2["img_metas"]
            head.apply_shared_conv = True
            for _ in range(3):
                rets2 = forward(res2, metas2)
            tags2 = ("shared_conv", "nchw_to_padded_nhwc")
            for t in tags2:
                ops.profile_events(t, True)
            # with a graph timing after it, this eager pass only feeds the per-launch kernel profile: 5 steps suffice
            eager_steps = args.steps if args.no_cuda_graph else 5
            ms2, _ = timed(lambda: forward(res2, metas2), eager_steps)
            per2 = {t: ops.profile_events(t, False) for t in tags2}
            if not args.no_cuda_graph:
                graphed2 = GraphedForward(head, metas2, res2, adopt_inputs=True)
                for _ in range(3):
                    rets2 = graphed2()
                ms2, _ = timed(lambda: graphed2(), args.steps)
            torch.cuda.synchronize()
            par2 = None
            if rank == 0 and not args.no_parity:
                cfg2 = dict(cfg)
                cfg2["_apply_shared_conv"] = True
                par2 = parity_check(cfg2, inputs2, B, coop, fdt, head, rets2)
            head.apply_shared_conv = False
            n_conv = len(per2["shared_conv"]) // eager_steps if per2["shared_conv"] else 0   # launches per step (coop: one per node)
            conv_ms = float(np.mean(per2["shared_conv"])) if per2["shared_conv"] else None
            bev = inputs2[[k for k in feat_keys if "pts_feats" in k][0]]
            conv_flops = 2.0 * B * bev.shape[2] * bev.shape[3] * 256 * 9 * 512
            with_conv = dict(value=B * world * args.steps / (ms2 * 1e-3), unit="frames/s", ms_per_step=ms2 / args.steps,
                             scope="forward_single from the RAW BEV map (512 channels) + image features: shared_conv included",
                             parity=par2,
                             shared_conv_kernel=dict(kernel="tc_gemm_kernel, 9-tap implicit GEMM + token epilogue", avg_launch_ms=conv_ms,
                                                     launches_per_step=n_conv,
                                                     achieved=(conv_flops / (conv_ms * 1e-3) / 1e12) if conv_ms else None, unit="TFLOP/s",
                                                     frac=(conv_flops / (conv_ms * 1e-3) / 1e12 / peaks()["bf16_tflops_sustained"]) if conv_ms else None,
                                                     algorithmic_flops_per_launch=conv_flops,
                                                     layout_kernel_ms=float(np.mean(per2["nchw_to_padded_nhwc"])) if per2["nchw_to_padded_nhwc"] else None))
            del res2

    frames = B * (1 if kv_split else world) * args.steps
    value = frames / (ms * 1e-3)
    pk = peaks()

    def node_tokens(prefix):
        n_b = n_i = 0
        p, i = inputs.get(prefix + "pts_feats"), inputs.get(prefix + "img_feats")
        if p is not None:
            n_b = p.shape[2] * p.shape[3]
        if i is not None:
            n_i = (i.shape[0] // B) * i.shape[2] * i.shape[3]
        return n_b, n_i

    nodes = [node_tokens("vehicle_"), node_tokens("infrastructure_")] if coop else [node_tokens("")]
    N_kv = float(np.mean([a + b for a, b in nodes]))  # one attention launch per node per layer
    N_img = float(np.mean([b for _, b in nodes]))
    N_kv_rank = N_kv
    if kv_split:
        from cmtcoop_b200 import parallel
        lo, hi = parallel.kv_split_range(int(N_kv), rank, world)
        N_kv_rank = float(hi - lo)   # each rank attends its own share of the tokens
    # roofline of the dominant kernel (tc_attn_db_kernel): algorithmic flops 4*Nq*N_kv*C per frame per layer
    flops_per_launch = 4.0 * 900 * N_kv_rank * 256 * B
    attn_avg_ms = float(np.mean(attn_ms)) if attn_ms else None
    roof = None
    kernels = []
    fsz = torch.empty((), dtype=fdt).element_size()
    if attn_avg_ms:
        achieved = flops_per_launch / (attn_avg_ms * 1e-3) / 1e12
        exps = 900.0 * N_kv_rank * 8 * B            # one exponential per (query, key, head)
        poly = (1.0 / 3.0) if (static_frac or 0) > 0.5 else 0.2   # share of the exponentials on the FMA pipes (ST_POLY / DB_POLY)
        clk = sm_clock_ghz or 1.9
        floor_ms = exps * (1.0 - poly) / (16.0 * 148 * clk * 1e9) * 1e3
        online_avg = float(np.mean(online_ms)) if online_ms else None
        roof = dict(bound="tensor", kernel="tc_attn_db_kernel<static shift> (+ online-kernel early exit + merge)",
                    achieved=achieved, peak=pk["bf16_tflops_sustained"], unit="TFLOP/s",
                    frac=achieved / pk["bf16_tflops_sustained"],
                    traffic=NCU_DRAM_BYTES_PER_FRAME.get(args.workload, 0) * B or None,
                    traffic_source="profiles/ ncu --set full capture of this kernel at this shape (not measured in this run)",
                    peak_source=pk["source"] + " sustained bf16 (kernel timed inside the step)",
                    launches_timed=len(attn_ms), avg_launch_ms=attn_avg_ms,
                    sm_clock_ghz_under_kernel=sm_clock_ghz,
                    share_of_step=attn_avg_ms * len(attn_ms) / ms_eager,
                    algorithmic_flops_per_launch=flops_per_launch,
                    static_item_fraction=static_frac,
                    online_kernel=dict(avg_launch_ms=online_avg,
                                       frac=(flops_per_launch / (online_avg * 1e-3) / 1e12 / pk["bf16_tflops_sustained"]) if online_avg else None,
                                       note="same workload with the operand-norm bound ignored: every item on the online-softmax "
                                            "instantiation (what a checkpoint with a score bound > 60 runs)"),
                    exp_roofline=dict(exponentials_per_launch=exps, mufu_ex2_per_clk_per_sm=16, sms=148,
                                      polynomial_share=poly, sm_clock_ghz=clk, floor_ms=floor_ms,
                                      frac=floor_ms / attn_avg_ms,
                                      note="time the MUFU pipe alone needs for the exponentials not taken by the FMA-pipe "
                                           "polynomial, over the measured launch time: at d_head = 32 the softmax pipe, not the "
                                           "tensor pipe, is the first wall (128 MMA flops per exponential)"))

        def kline(tag, kernel, bound, work, unit_peak, note=None):
            t = per_launch.get(tag) or []
            if not t:
                return
            avg = float(np.mean(t))
            ach = work / (avg * 1e-3) / (1e9 if bound == "hbm" else 1e12)
            kernels.append(dict(kernel=kernel, tag=tag, bound=bound, avg_launch_ms=avg, launches_timed=len(t), achieved=ach,
                                peak=unit_peak, unit="GB/s" if bound == "hbm" else "TFLOP/s", frac=ach / unit_peak,
                                algorithmic_work_per_launch=work, share_of_step=avg * len(t) / ms_eager, **({"note": note} if note else {})))

        n_nodes = len(nodes)
        hb, tp = pk["hbm_gbs"], pk["bf16_tflops_sustained"]
        # under the KV-token split every token-shaped kernel works on the rank's rows only
        n_bev_tok = N_kv - N_img
        img_rank = float(N_img)
        bev_rank = float(n_bev_tok)
        if kv_split:
            img_rank = float(max(0, hi - max(lo, int(n_bev_tok))))
            bev_rank = float(max(0, min(hi, int(n_bev_tok)) - lo))
        kline("ray_pe", "ray_pe_kernel (K1)", "hbm", B * img_rank * 192 * 2.0, hb,
              note="at 8 frames the 74 MB output is L2-resident and the launch is ~20 us; profiles/ holds the 64-frame run")
        kline("gather_tokens", "gather_tokens_kernel (K4)", "hbm",
              B * N_kv_rank * 256 * fsz + B * img_rank * 256 * 4 + bev_rank * 256 * 4 + 2 * B * N_kv_rank * 256 * 2, hb)
        kline("k_proj", "tc_gemm_kernel K projection, all layers", "tensor", 2.0 * B * N_kv_rank * 256 * 1536, tp)
        kline("v_proj", "tc_gemm_kernel V^T projection, all layers", "tensor", 2.0 * B * N_kv_rank * 256 * 1536, tp)
        kline("rv_pe_mlp.0", "tc_gemm_kernel rv-PE MLP layer 1", "tensor", 2.0 * B * img_rank * 192 * 1024, tp)
        kline("rv_pe_mlp.2", "tc_gemm_kernel rv-PE MLP layer 2", "tensor", 2.0 * B * img_rank * 1024 * 256, tp)
        del n_nodes

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            cpu = cpu_baseline_sample(args.workload)
        line = dict(metric=METRIC, value=value, unit="frames/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong" if kv_split else "weak",
                    vs_baseline=None,
                    dtype="bf16", data="synthetic",
                    config=dict(workload=WORKLOADS[args.workload][3], frames_per_gpu=B,
                                global_batch=B if kv_split else B * world,
                                parallelism=((f"K/V tokens split x{world}: queries replicated, (O, LSE) records exchanged and "
                                              "merged per decoder layer by one kernel over peer memory (NVLink loads, no NCCL "
                                              "call on the data path)" if args.kv_split_peer else
                                              f"K/V tokens split x{world}: queries replicated, one NCCL all-gather of "
                                              "(O, LSE) per decoder layer + LSE merge") if kv_split else
                                             f"frame sharding x{world}, no data-path collective"),
                                feature_dtype=args.feat_dtype,
                                l2="inputs (%.0f MB per step) exceed the 126 MB L2" % (h2d / 1e6),
                                scope="forward_single from post-shared_conv BEV map + image features to task-head outputs",
                                cuda_graph=not args.no_cuda_graph, eager_ms_per_step=ms_eager / args.steps,
                                pinned_host_numa_cpus=(f"{numa.cpus[0]}-{numa.cpus[-1]} ({len(numa.cpus)})" if numa.cpus else None)),
                    clocks=clocks, gpu_launches=launches,
                    e2e=dict(value=frames / (ms_e2e * 1e-3), unit="frames/s", h2d_bytes_per_step=h2d,
                             d2h_bytes_per_step=d2h, ms_per_step=ms_e2e / args.steps),
                    parity=parity, roofline=roof, roofline_kernels=kernels, with_shared_conv=with_conv, cpu_baseline=cpu)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
        print(json.dumps(line), flush=True)
        if parity is not None and not parity["ok"]:
            print(f"bench.py: PARITY FAILED: frame 0 rel-L2 {parity['rel_l2']:.3e} > 1e-2", file=sys.stderr, flush=True)
    if world > 1:
        # graphs that captured NCCL work must be gone before the process group is torn down
        graphed = graphed2 = runner = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
