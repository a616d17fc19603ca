"""Serving-loop helper: run a head over a stream of HOST batches with the host->device copy of batch
i+1 and the device->host copy of result i-1 overlapped with the compute of batch i.

The hot path itself never synchronises (every kernel is stream-ordered), so overlapping is a matter of
three CUDA streams and double buffering:

    copy-in stream : pinned host features -> device buffer[i % 2]
    compute stream : head.forward_single(device buffer[i % 2]) -> task-head tensors
    copy-out stream: task-head tensors (or, with outputs="boxes", the batched box decode) -> pinned host result[i % 2]

This is plumbing (torch streams / events), not a kernel; it is what bench.py's end-to-end number uses.

`GraphedForward` captures one forward (about a hundred launches, a third of them a few microseconds long) into a CUDA
graph for a fixed batch shape and calibration and replays it: no per-launch host work, back-to-back kernel issue.
"""
from __future__ import annotations

import os

import torch


class numa_local_to_gpu:
    """Context manager: while active, the calling thread runs on the CPU cores NVML reports as local to GPU
    `device_index`, so pinned host buffers allocated (first touched) inside land on that GPU's NUMA node -- with 4 or 8
    ranks streaming features at PCIe rate, remote-node staging buffers are what a dual-socket host runs out of first.
    Restores the previous affinity on exit; a no-op when NVML or sched_setaffinity are unavailable."""

    def __init__(self, device_index: int):
        self.index = device_index
        self.prev = None
        self.cpus = None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            n_words = (os.cpu_count() + 63) // 64
            words = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
            cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
            allowed = os.sched_getaffinity(0)
            cpus &= allowed
            if cpus and cpus != allowed:
                self.prev = allowed
                os.sched_setaffinity(0, cpus)
                self.cpus = sorted(cpus)
        except Exception:
            self.prev = None
        return self

    def __exit__(self, *exc):
        if self.prev is not None:
            try:
                os.sched_setaffinity(0, self.prev)
            except Exception:
                pass
        return False


def _head_forward(head, coop, inputs, metas, decode_boxes):
    """head.forward_single on an inputs dict (feature tensors, plus "node_valid" for the cooperative heads or
    "sensor_valid" for the single-node heads), followed by the batched box decode with decode_boxes."""
    g = inputs.get
    if coop:
        if g("sensor_valid") is not None:
            raise ValueError("sensor_valid is an input of the single-node heads only (the cooperative heads take node_valid)")
        mask = g("node_valid")
        rets = head.forward_single(g("vehicle_pts_feats"), g("infrastructure_pts_feats"), g("vehicle_img_feats"),
                                   g("infrastructure_img_feats"), metas, node_valid=mask)
    else:
        if g("node_valid") is not None:
            raise ValueError("node_valid is an input of the cooperative heads only")
        mask = g("sensor_valid")
        rets = head.forward_single(g("pts_feats"), g("img_feats"), metas, sensor_valid=mask)
    if decode_boxes:
        return rets, head.get_bboxes_batched([[r] for r in rets], metas, node_valid=mask)
    return rets


class PipelinedRunner:
    def __init__(self, head, img_metas, example_inputs: dict, device, use_cuda_graph: bool = False,
                 keep_results: bool = True, partial_upload=None, outputs: str = "heads"):
        """example_inputs: {name: pinned CPU tensor} with the feature tensors `forward_single` takes
        (pts_feats / img_feats, or the four vehicle_/infrastructure_ entries for the coop heads); fp32, bf16 or
        fp16 -- the gather kernel rounds every feature to the compute dtype on arrival, so 16-bit features halve
        the PCIe traffic without changing a single output bit in bf16 mode.  A cooperative head may also take
        "node_valid", a pinned torch.bool [2, B] mask of the nodes that delivered each frame, and a single-node head
        "sensor_valid", a pinned torch.bool [S, B] mask of the sensors that delivered each frame (forward_single); it is
        copied in with every batch like the features and, with outputs="boxes", also reaches the decode.
        use_cuda_graph: replay one captured forward per device input slot instead of launching eagerly.
        keep_results: `run` returns every batch's outputs as ordinary CPU tensors (copied out of the two pinned
        staging buffers before those are reused); False keeps only the staging buffers (results of the last two
        batches), for callers that consume results through `on_result`.
        partial_upload: under the KV-token split a rank reads only the map rows that hold its tokens, so only those
        rows are copied to the device (a few strided cudaMemcpy2DAsync per tensor, parallel.token_rows_copy_plan); the rest of
        the device buffers is never read.  None = do so whenever the split is enabled on a non-cooperative head.
        outputs: what each batch hands back.  "heads": the task-head outputs of every decoder layer (the list of per-task
        dicts forward_single returns).  "boxes": the detections, head.get_bboxes_batched of those outputs, computed on
        the device after the forward (inside the graph with use_cuda_graph) -- only that fixed-shape dict
        {boxes, scores, labels, count, topk_index} is copied back (detector_glue.batched_to_results makes per-frame
        results of it)."""
        if outputs not in ("heads", "boxes"):
            raise ValueError(f'outputs must be "heads" or "boxes", got {outputs!r}')
        self.outputs = outputs
        self.head = head
        self.metas = img_metas
        self.dev = torch.device(device)
        self.coop = type(head).__name__.endswith("Coop")
        self.keys = [k for k, v in example_inputs.items() if v is not None]
        self.dbuf = [{k: torch.empty_like(example_inputs[k], device=self.dev) for k in self.keys} for _ in range(2)]
        self.hout = [None, None]                                   # per slot: list (tasks) of {name: pinned tensor}
        self.keep_results = keep_results
        self.s_in = torch.cuda.Stream(self.dev)
        self.s_out = torch.cuda.Stream(self.dev)
        self.ev_in = [torch.cuda.Event() for _ in range(2)]       # copy-in of slot done
        self.ev_free = [torch.cuda.Event() for _ in range(2)]     # compute finished reading slot
        self.ev_done = [torch.cuda.Event() for _ in range(2)]     # compute of slot done
        self.ev_out = [torch.cuda.Event() for _ in range(2)]      # copy-out of slot done
        self._primed = [False, False]
        self.h2d_bytes = int(sum(example_inputs[k].numel() * example_inputs[k].element_size() for k in self.keys))
        self.d2h_bytes = 0
        self.graphs = None
        self.copy_plan = None
        tr = getattr(head, "transformer", None)
        if partial_upload is None:
            partial_upload = (tr is not None and getattr(tr, "kv_split_group", None) is not None and not self.coop
                              and set(self.keys) <= {"pts_feats", "img_feats"})
        if partial_upload:
            self._plan_partial_upload(example_inputs)
        if use_cuda_graph:
            for slot in range(2):     # the graphs read the slot buffers in place: give them defined contents first
                for k in self.keys:
                    self.dbuf[slot][k].copy_(example_inputs[k], non_blocking=True)
            torch.cuda.current_stream(self.dev).synchronize()
            self.graphs = [GraphedForward(head, img_metas, self.dbuf[slot], adopt_inputs=True,
                                          decode_boxes=outputs == "boxes") for slot in range(2)]

    def _forward(self, feats):
        return _head_forward(self.head, self.coop, feats, self.metas, self.outputs == "boxes")

    def _payload(self, staging):
        """What a batch hands out: the per-task list of head outputs, or the box dict."""
        return staging[0] if self.outputs == "boxes" else staging

    def _plan_partial_upload(self, example_inputs):
        """Rectangles of the feature maps this rank's tokens live in (KV-token split)."""
        import ctypes

        from . import parallel
        pts, img = example_inputs.get("pts_feats"), example_inputs.get("img_feats")
        B = pts.shape[0] if pts is not None else len(self.metas)
        n_kv = (pts.shape[2] * pts.shape[3] if pts is not None else 0) + \
               ((img.shape[0] // B) * img.shape[2] * img.shape[3] if img is not None else 0)
        lo, hi = self.head.transformer.kv_token_range(n_kv)
        halo = 1 if (getattr(self.head, "apply_shared_conv", True) and getattr(self.head, "shared_conv", None) is not None) else 0
        plan = parallel.token_rows_copy_plan(None if pts is None else tuple(pts.shape), None if img is None else tuple(img.shape),
                                             B, lo, hi, halo)
        self.copy_plan = {"pts_feats": plan["pts"], "img_feats": plan["img"]}
        self._plan_key = (n_kv, lo, hi)
        self._cudart = ctypes.CDLL("libcudart.so.12")      # the runtime torch has loaded
        self._cudart.cudaMemcpy2DAsync.restype = ctypes.c_int
        self._cudart.cudaMemcpy2DAsync.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t,
                                                   ctypes.c_size_t, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]
        self.h2d_bytes = int(sum(w * h * example_inputs[k].element_size() for k in self.keys for _, _, w, h in self.copy_plan[k]))

    def _enqueue_copy_in(self, slot, host_inputs):
        with torch.cuda.stream(self.s_in):
            if self._primed[slot]:
                self.s_in.wait_event(self.ev_free[slot])   # the previous user of this slot has consumed it
            if self.copy_plan is not None:
                n_kv, lo, hi = self._plan_key
                if self.head.transformer.kv_token_range(n_kv) != (lo, hi):
                    raise RuntimeError("PipelinedRunner: the KV-token split changed after the partial upload was planned; "
                                       "build a new runner")
            for k in self.keys:
                if self.copy_plan is None:
                    self.dbuf[slot][k].copy_(host_inputs[k], non_blocking=True)
                    continue
                src, dst = host_inputs[k], self.dbuf[slot][k]
                assert src.is_contiguous() and src.is_pinned() and src.shape == dst.shape and src.dtype == dst.dtype
                esz = src.element_size()
                for off, pitch, width, height in self.copy_plan[k]:
                    rc = self._cudart.cudaMemcpy2DAsync(dst.data_ptr() + off * esz, pitch * esz, src.data_ptr() + off * esz,
                                                        pitch * esz, width * esz, height, 1, self.s_in.cuda_stream)
                    if rc != 0:
                        raise RuntimeError(f"cudaMemcpy2DAsync failed with error {rc}")
            self.ev_in[slot].record(self.s_in)

    def _collect(self, slot):
        """Host copy of the staging buffers of `slot` once its device->host transfer has landed."""
        self.ev_out[slot].synchronize()
        return self._payload([{n: t.clone() for n, t in task.items()} for task in self.hout[slot]])

    @torch.no_grad()
    def run(self, host_batches, on_result=None):
        """host_batches: iterable of {name: pinned CPU tensor}.  Returns one entry per batch: the list (one dict per
        task) of head outputs as CPU tensors, or with outputs="boxes" the batched box-decode dict.  Every device->host
        copy has completed when this returns.
        on_result(i, staging): optional callback invoked with the pinned staging dicts of batch i right after its
        transfer completed (zero-copy consumers); with keep_results=False the returned list holds None for every
        batch but the last two, whose entries are the staging buffers themselves."""
        cur = torch.cuda.current_stream(self.dev)
        batches = list(host_batches)
        results = [None] * len(batches)
        if not batches:
            return results
        pending = [None, None]                                      # batch index whose outputs sit in the slot
        trace = os.environ.get("CMT_RUNNER_TRACE") == "1"           # host-side phase times of every step -> stderr
        if trace:
            import sys
            import time
            marks = []
        self._enqueue_copy_in(0, batches[0])
        for i, _ in enumerate(batches):
            slot = i & 1
            if trace:
                tm = [time.perf_counter()]
            if i + 1 < len(batches):
                self._enqueue_copy_in(slot ^ 1, batches[i + 1])     # overlaps this step's compute
            cur.wait_event(self.ev_in[slot])
            if trace:
                tm.append(time.perf_counter())
            if pending[slot] is not None:
                # the staging buffers of this slot still hold batch i-2: hand it out before they are overwritten
                j = pending[slot]
                if on_result is not None:
                    self.ev_out[slot].synchronize()
                    on_result(j, self._payload(self.hout[slot]))
                if self.keep_results:
                    results[j] = self._collect(slot)
                pending[slot] = None
            if trace:
                tm.append(time.perf_counter())
            if self._primed[slot]:
                # a graph's static outputs are overwritten by the slot's next replay, and the staging buffers by the
                # next copy-out: both wait for the copy-out of the slot's previous batch
                cur.wait_event(self.ev_out[slot])
            rets = self.graphs[slot]() if self.graphs is not None else self._forward(self.dbuf[slot])
            if self.outputs == "boxes":
                rets = [rets[1]]
            self.ev_free[slot].record(cur)
            self._primed[slot] = True
            if trace:
                tm.append(time.perf_counter())
            if self.hout[slot] is None:
                self.hout[slot] = [{n: torch.empty(t.shape, dtype=t.dtype).pin_memory() for n, t in task.items()}
                                   for task in rets]
                self.d2h_bytes = int(sum(t.numel() * t.element_size() for task in rets for t in task.values()))
            self.ev_done[slot].record(cur)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(self.ev_done[slot])
                for task, stage in zip(rets, self.hout[slot]):
                    for n, t in task.items():
                        t.record_stream(self.s_out)
                        stage[n].copy_(t, non_blocking=True)
                self.ev_out[slot].record(self.s_out)
            pending[slot] = i
            if trace:
                tm.append(time.perf_counter())
                marks.append([1e3 * (b - a) for a, b in zip(tm[:-1], tm[1:])])
        if trace:
            for i, m in enumerate(marks):
                print(f"runner step {i}: copy-in enqueue {m[0]:.2f} ms, collect {m[1]:.2f}, forward enqueue {m[2]:.2f}, copy-out enqueue {m[3]:.2f}",
                      file=sys.stderr, flush=True)
        self.s_out.synchronize()                                    # every device->host copy has landed
        self.s_in.synchronize()
        for slot in (0, 1):
            j = pending[slot]
            if j is None:
                continue
            if on_result is not None:
                on_result(j, self._payload(self.hout[slot]))
            results[j] = self._collect(slot) if self.keep_results else self._payload(self.hout[slot])
        return results


def _metas_key(img_metas):
    """Identity of the calibration the forward depends on (lidar2img of every view of every frame + pad shapes)."""
    import numpy as np
    out = []
    for m in img_metas:
        for k in sorted(m):
            if k.endswith("lidar2img"):
                out.append((k, np.asarray(m[k], dtype=np.float64).tobytes()))
            elif k.endswith("pad_shape"):
                out.append((k, repr(m[k])))
            elif k.endswith("calibration") and m[k] is not None:   # device tensors: the graph follows in-place updates
                out.append((k, tuple(int(t.data_ptr()) for t in m[k])))
    return tuple(out)


class GraphedForward:
    """CUDA-graph replay of `head.forward_single` for one input shape.

        g = GraphedForward(head, img_metas, {"pts_feats": x, "img_feats": x_img})   # device tensors
        rets = g(inputs)          # copies `inputs` into the graph's static buffers (unless they ARE those buffers), replays

    With decode_boxes=True the graph also holds `head.get_bboxes_batched` of the outputs, and a call returns
    (head outputs, boxes dict), both static outputs of the graph.

    For a cooperative head the inputs may include "node_valid" (torch.bool [2, B]), for a single-node head
    "sensor_valid" (torch.bool [S, B]; forward_single): like the features it lives in a static buffer that each call
    overwrites, so a new mask is one small copy and never a re-capture.

    The graph bakes in device addresses, so the inputs live in static buffers (`g.static_inputs`) and the outputs are
    overwritten by the next replay.  The calibration matrices enter the forward as device tensors uploaded once per
    distinct `img_metas` (CmtHead._matrices); a call with different calibration re-captures.
    """

    def __init__(self, head, img_metas, example_inputs: dict, warmup: int = 3, adopt_inputs: bool = False,
                 decode_boxes: bool = False):
        """adopt_inputs: use the given tensors themselves as the graph's static input buffers (no clone).
        decode_boxes: capture the batched box decode (head.get_bboxes_batched) after the forward."""
        self.head = head
        self.decode_boxes = decode_boxes
        self.coop = type(head).__name__.endswith("Coop")
        self.static_inputs = {k: (v if adopt_inputs else v.clone()) for k, v in example_inputs.items() if v is not None}
        self.graph = None
        self.static_outputs = None
        self._key = None
        self._capture(img_metas, warmup)

    def _forward(self, metas):
        return _head_forward(self.head, self.coop, self.static_inputs, metas, self.decode_boxes)

    @torch.no_grad()
    def _capture(self, img_metas, warmup):
        dev = next(iter(self.static_inputs.values())).device
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):          # warm-up off the capture: weight / PE / calibration caches, workspaces
            for _ in range(max(warmup, 1)):
                self._forward(img_metas)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.static_outputs = self._forward(img_metas)
        self._key = _metas_key(img_metas)

    @torch.no_grad()
    def __call__(self, inputs: dict = None, img_metas=None):
        if img_metas is not None and _metas_key(img_metas) != self._key:
            self._capture(img_metas, 1)
        if inputs is not None:
            for k, buf in self.static_inputs.items():
                src = inputs[k]
                if src.data_ptr() != buf.data_ptr():
                    buf.copy_(src, non_blocking=True)
        self.graph.replay()
        return self.static_outputs
