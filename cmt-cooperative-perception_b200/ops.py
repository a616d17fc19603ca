"""Torch-tensor front ends of the C-ABI operators (``include/cmtcoop_b200.h``).

PyTorch is used for device memory and the current stream only; every computation below runs in
``libcmtcoop_b200.so``.  All tensors must live on a CUDA (sm_100) device -- there is no CPU path.
"""
from __future__ import annotations

import ctypes
import math

import torch

from . import _lib
from ._lib import (CMT_BF16, CMT_BF16_SIMT, CMT_F16, CMT_F32, GEMM_BIAS_PER_ROW, GEMM_FORCE_SIMT, GEMM_RELU,
                   GEMM_TRANSPOSE_OUT)

HEAD_DIM = 32
LOG2E = 1.4426950408889634

_launches = 0  # kernels launched through this module (bench.py reports it as gpu_launches)


def launch_count() -> int:
    return _launches


def _count(n=1):
    global _launches
    _launches += n


_profile = {}  # op name -> list of (start, end) CUDA events recorded on the launching stream


def profile_events(name: str, enable: bool):
    """bench.py hook: time every launch of op `name` with CUDA events on the stream it is launched on.
    Enabling starts a fresh list; disabling synchronises and returns the per-launch durations in ms."""
    if enable:
        _profile[name] = []
        return None
    pairs = _profile.pop(name, [])
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in pairs]


class _timed:
    """Records a CUDA-event pair around the launches of one op on the launching stream when bench.py asked for
    that tag (profile_events); otherwise free."""

    def __init__(self, tag, ref):
        self.ev = _profile.get(tag) if tag is not None and _profile else None
        self.ref = ref

    def __enter__(self):
        if self.ev is not None:
            self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.e0.record(torch.cuda.current_stream(self.ref.device))
        return self

    def __exit__(self, *exc):
        if self.ev is not None:
            self.e1.record(torch.cuda.current_stream(self.ref.device))
            self.ev.append((self.e0, self.e1))
        return False


# bench.py switch: ignore the operand-norm maxima so that every attention item takes the online-softmax kernel
# (what a checkpoint with peaky logits, score bound > 60, would run); never set by the library itself
FORCE_ONLINE_SOFTMAX = False


# The compute precisions of the modules (`set_precision`): 'bf16' and 'fp16' run the tcgen05 kernels with 16-bit operands,
# 'fp32' the fp32 CUDA-core verification kernels.  The task heads stay fp32-grade in every precision.
PRECISIONS = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}


def compute_dtype(precision: str) -> torch.dtype:
    """The torch dtype of a precision name; an unknown name raises ValueError."""
    try:
        return PRECISIONS[precision]
    except KeyError:
        raise ValueError(f"unknown precision {precision!r} (one of {', '.join(PRECISIONS)})") from None


def _dt(dtype) -> int:
    if dtype == torch.float32:
        return CMT_F32
    if dtype == torch.bfloat16:
        return CMT_BF16
    if dtype == torch.float16:
        return CMT_F16
    raise TypeError(f"unsupported dtype {dtype} (fp32, bf16 or fp16 only)")


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream(t):
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _cuda(t, name, dtype=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.CmtLibraryError(f"{name} must be a CUDA tensor: libcmtcoop_b200 has no CPU fallback")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


def check_node_valid(node_valid, B, device, n_nodes=2, name="node_valid"):
    """Host-side checks of a per-frame node mask: a torch.bool tensor [n_nodes, B] on `device` (n_nodes=None: any
    n_nodes >= 1).  Row n, column b is True when node n delivered frame b.  The values are never read here, so the check
    costs no device synchronisation.  Returns the mask, contiguous.  `name` is the argument named in the errors (the
    single-node heads' per-sensor mask, `sensor_valid`, has the same layout)."""
    if not isinstance(node_valid, torch.Tensor):
        raise TypeError(f"{name} must be a torch.bool tensor, got {type(node_valid).__name__}")
    if node_valid.dtype != torch.bool:
        raise TypeError(f"{name} must be torch.bool, got {node_valid.dtype}")
    rows = n_nodes if n_nodes is not None else (node_valid.shape[0] if node_valid.dim() == 2 else -1)
    if node_valid.dim() != 2 or rows < 1 or tuple(node_valid.shape) != (rows, B):
        want = f"[{n_nodes}, {B}]" if n_nodes is not None else f"[n_nodes, {B}]"
        raise ValueError(f"{name} must be {want}, got {list(node_valid.shape)}")
    if node_valid.device != torch.device(device):
        raise ValueError(f"{name} must live on {torch.device(device)} (the features' device), got {node_valid.device}")
    return node_valid.contiguous()


def _mask_bytes(mask, B, device, rows, name):
    """A checked bool mask [rows, B] as the uint8 device array the kernels read (a view: bool is one 0/1 byte)."""
    return check_node_valid(mask, B, device, n_nodes=rows, name=name).view(torch.uint8)


def _pc(pc_range):
    return (ctypes.c_float * 6)(*[float(v) for v in pc_range])


# ------------------------------------------------------------------------------------------
def ray_pe(img2lidar, H, W, depth_num, pad_h, pad_w, pc_range, out_dtype=torch.bfloat16):
    """K1 (cmt_head.py:417-432). img2lidar [n_cam,4,4] fp32 -> [n_cam,H,W,depth_num*3]."""
    m = _cuda(img2lidar, "img2lidar", torch.float32)
    n_cam = m.shape[0]
    out = torch.empty((n_cam, H, W, depth_num * 3), dtype=out_dtype, device=m.device)
    lib = _lib.load()
    with torch.cuda.device(m.device), _timed("ray_pe", m):
        rc = lib.cmt_ray_pe(_ptr(m), _ptr(out), n_cam, H, W, depth_num, float(pad_h), float(pad_w),
                            ctypes.cast(_pc(pc_range), ctypes.c_void_p), _dt(out_dtype), _stream(m))
    _lib.check(rc, "cmt_ray_pe")
    _count()
    return out


def ray_query_pe(ref, lidar2img, img2lidar, depth_num, pad_h, pad_w, pc_range, out_dtype=torch.bfloat16):
    """K1b (cmt_head.py:439-464). ref [B,Nq,3], matrices [B,V,4,4] -> feat [B,V,Nq,D*3], mask [B,V,Nq]."""
    ref = _cuda(ref, "ref", torch.float32)
    l2i = _cuda(lidar2img, "lidar2img", torch.float32)
    i2l = _cuda(img2lidar, "img2lidar", torch.float32)
    B, Nq, _ = ref.shape
    V = l2i.shape[1]
    out = torch.empty((B, V, Nq, depth_num * 3), dtype=out_dtype, device=ref.device)
    mask = torch.empty((B, V, Nq), dtype=torch.float32, device=ref.device)
    lib = _lib.load()
    with torch.cuda.device(ref.device):
        rc = lib.cmt_ray_query_pe(_ptr(ref), _ptr(l2i), _ptr(i2l), _ptr(out), _ptr(mask), B, V, Nq, depth_num,
                                  float(pad_h), float(pad_w), ctypes.cast(_pc(pc_range), ctypes.c_void_p),
                                  _dt(out_dtype), _stream(ref))
    _lib.check(rc, "cmt_ray_query_pe")
    _count()
    return out, mask


def masked_view_sum(emb, mask, base=None, view_valid=None):
    """base + (emb * mask[..., None]).sum(1)  (cmt_head.py:466, :492). emb [B,V,Nq,C] -> [B,Nq,C] fp32.
    base: optional fp32 [B,Nq,C] or [Nq,C] (shared by every frame) added after the view sum.
    view_valid: optional torch.bool [V, B] on emb's device; a view that is False for frame b is left out of its sum (its
    embedding, NaN included, is not read), the others are summed in the same order."""
    emb = _cuda(emb, "emb")
    mask = _cuda(mask, "mask", torch.float32)
    B, V, Nq, C = emb.shape
    out = torch.empty((B, Nq, C), dtype=torch.float32, device=emb.device)
    bstride = 0
    if base is not None:
        base = _cuda(base, "base", torch.float32)
        assert base.shape in ((B, Nq, C), (Nq, C))
        bstride = Nq * C if base.dim() == 3 else 0
    if view_valid is not None:
        view_valid = _mask_bytes(view_valid, B, emb.device, V, "view_valid")
    lib = _lib.load()
    with torch.cuda.device(emb.device):
        rc = lib.cmt_masked_view_sum(_ptr(emb), _ptr(mask), _ptr(base), bstride, _ptr(out), B, V, Nq, C, _dt(emb.dtype),
                                     _stream(emb), _ptr(view_valid))
    _lib.check(rc, "cmt_masked_view_sum")
    _count()
    return out


def pos2embed(pos, num_pos_feats=128, out_dtype=torch.bfloat16):
    """pos2embed (cmt_head.py:40-50). pos [...,>=2] fp32 -> [..., 2*num_pos_feats]."""
    pos = _cuda(pos.contiguous(), "pos", torch.float32)
    lead = pos.shape[:-1]
    stride = pos.shape[-1]
    N = int(math.prod(lead))
    out = torch.empty((*lead, 2 * num_pos_feats), dtype=out_dtype, device=pos.device)
    lib = _lib.load()
    with torch.cuda.device(pos.device):
        rc = lib.cmt_pos2embed(_ptr(pos), _ptr(out), N, stride, num_pos_feats, _dt(out_dtype), _stream(pos))
    _lib.check(rc, "cmt_pos2embed")
    _count()
    return out


_FEAT_DTYPES = {torch.float32: CMT_F32, torch.bfloat16: CMT_BF16, torch.float16: CMT_F16}


def gather_tokens(x_bev, x_img, bev_pos, rv_pos, B, V, out_dtype=torch.bfloat16, tok_range=None, n_bev_reserved=0,
                  out=None, rv_rows=None, sensor_valid=None):
    """K4 (cmt_transformer.py:105-110 + petr_transformer.py:296-299).
    x_bev [B,C,Hb,Wb] | None, x_img [B*V,C,h,w] | None (fp32, bf16 or fp16 -- both the same dtype),
    bev_pos [N_bev,C], rv_pos [B*V*h*w, C] (any leading shape) fp32 -> xk = mem+pos, xv = mem, both
    [B,N_kv,C]; with tok_range=(lo, hi) only those tokens of the concatenated axis: [B,hi-lo,C].
    sensor_valid: optional torch.bool [S, B] on the features' device, one row per sensor in token order (the BEV map
    first when there are BEV tokens, then the V cameras); the tokens of an absent (sensor, frame) become zero rows of
    xk and xv, whatever its features and position encoding hold."""
    ref = x_bev if x_bev is not None else x_img
    dev = ref.device
    C = ref.shape[1]
    fdt = ref.dtype
    if fdt not in _FEAT_DTYPES:
        raise TypeError(f"feature maps must be fp32, bf16 or fp16, got {fdt}")
    n_bev = 0
    n_img = 0
    if x_bev is not None:
        x_bev = _cuda(x_bev, "x_bev", fdt)
        bev_pos = _cuda(bev_pos, "bev_pos", torch.float32)
        n_bev = x_bev.shape[2] * x_bev.shape[3]
        assert x_bev.shape[0] == B and bev_pos.numel() == n_bev * C
    if x_img is not None:
        x_img = _cuda(x_img, "x_img", fdt)
        rv_pos = _cuda(rv_pos, "rv_pos", torch.float32)
        n_img = x_img.shape[2] * x_img.shape[3]
        assert x_img.shape[0] == B * V
        assert rv_pos.numel() == (B * V * n_img * C if rv_rows is None else B * (rv_rows[1] - rv_rows[0]) * C)
    else:
        V = 0
    if x_bev is None:
        n_bev = n_bev_reserved
    N_kv = n_bev + V * n_img
    if sensor_valid is not None:
        sensor_valid = _mask_bytes(sensor_valid, B, dev, (1 if n_bev > 0 else 0) + V, "sensor_valid")
    lo, hi = (0, N_kv) if tok_range is None else tok_range
    if out is not None:
        xk, xv = out
        assert xk.shape == (B, hi - lo, C) and xv.shape == xk.shape and xk.dtype == out_dtype and xk.is_contiguous()
    else:
        xk = torch.empty((B, hi - lo, C), dtype=out_dtype, device=dev)
        xv = torch.empty((B, hi - lo, C), dtype=out_dtype, device=dev)
    if hi <= lo:
        return xk, xv   # empty share of the token axis: nothing to launch
    lib = _lib.load()
    with torch.cuda.device(dev), _timed("gather_tokens", ref):
        rc = lib.cmt_gather_tokens(_ptr(x_bev), _ptr(x_img), _ptr(bev_pos), _ptr(rv_pos), _ptr(xk), _ptr(xv),
                                   B, C, n_bev, V, n_img, lo, hi, 0 if rv_rows is None else rv_rows[0],
                                   0 if rv_rows is None else rv_rows[1] - rv_rows[0], _FEAT_DTYPES[fdt], _dt(out_dtype),
                                   _stream(ref), _ptr(sensor_valid))
    _lib.check(rc, "cmt_gather_tokens")
    _count()
    return xk, xv


def sensor_key_keep(sensor_valid, B, n_bev, V, n_img):
    """The cross-attention's key mask from a per-sensor mask (cmt_sensor_key_keep): sensor_valid torch.bool [S, B]
    (S = (n_bev > 0) + V, as in gather_tokens) -> torch.bool [B, n_bev + V*n_img], True where the token's sensor
    delivered the frame (cross_attn's key_keep)."""
    S = (1 if n_bev > 0 else 0) + V
    if not isinstance(sensor_valid, torch.Tensor) or not sensor_valid.is_cuda:
        raise _lib.CmtLibraryError("sensor_valid must be a CUDA tensor: libcmtcoop_b200 has no CPU fallback")
    mask = _mask_bytes(sensor_valid, B, sensor_valid.device, S, "sensor_valid")
    keep = torch.empty((B, n_bev + V * n_img), dtype=torch.bool, device=mask.device)
    lib = _lib.load()
    with torch.cuda.device(mask.device):
        rc = lib.cmt_sensor_key_keep(_ptr(mask), _ptr(keep), B, n_bev, V, n_img, _stream(mask))
    _lib.check(rc, "cmt_sensor_key_keep")
    _count()
    return keep


def conv_guard_rows(W):
    """Guard rows before and after each frame of the padded channel-last operand (>= W + 3, kept a multiple of 8)."""
    return (W + 3 + 7) // 8 * 8


def nchw_to_padded_nhwc(x, out=None, dtype=torch.bfloat16, frame_valid=None):
    """[B,C,H,W] (fp32|bf16|fp16) -> zero-padded channel-last rows [B, 2*guard + (H+2)*(W+2), C] in `dtype` (bf16 or fp16)
    (cmt_nchw_to_padded_nhwc).  `out` (zero-initialised once, then reusable: only interior rows are written) is allocated
    when None.  frame_valid: optional torch.bool [B] on x's device; the interior rows of a False frame are written as
    zeros (its input is not read)."""
    x = _cuda(x, "x")
    if x.dtype not in _FEAT_DTYPES:
        raise TypeError(f"feature maps must be fp32, bf16 or fp16, got {x.dtype}")
    B, C, H, W = x.shape
    guard = conv_guard_rows(W)
    rows = 2 * guard + (H + 2) * (W + 2)
    if dtype not in (torch.bfloat16, torch.float16):
        raise TypeError(f"nchw_to_padded_nhwc: output dtype must be bf16 or fp16, got {dtype}")
    if out is None:
        out = torch.zeros((B, rows, C), dtype=dtype, device=x.device)
    assert out.shape == (B, rows, C) and out.dtype == dtype and out.is_contiguous()
    if frame_valid is not None:
        frame_valid = _mask_bytes(frame_valid.reshape(1, -1), B, x.device, 1, "frame_valid")
    lib = _lib.load()
    with torch.cuda.device(x.device), _timed("nchw_to_padded_nhwc", x):
        rc = lib.cmt_nchw_to_padded_nhwc(_ptr(x), _ptr(out), B, C, H, W, guard, _FEAT_DTYPES[x.dtype], _stream(x), _dt(dtype),
                                         _ptr(frame_valid))
    _lib.check(rc, "cmt_nchw_to_padded_nhwc")
    _count()
    return out


def shared_conv_tokens(xp, w, bias, bev_pos, xk, xv, H, W, tok_range=None):
    """3x3 conv + folded BN + ReLU as an implicit GEMM writing the BEV token rows of xk / xv (cmt_shared_conv_tokens).
    xp [B,rows,Cin] from nchw_to_padded_nhwc; w [Cout, 9*Cin] tap-major with the BN scale folded in; bias [Cout] fp32;
    bev_pos [H*W,Cout] fp32; xk, xv [B,n_rows,Cout] whose first (hi-lo) rows receive tokens [lo,hi) (default all).
    xp, w, xk and xv share one dtype, bf16 or fp16."""
    xp = _cuda(xp, "xp")
    if xp.dtype not in (torch.bfloat16, torch.float16):
        raise TypeError(f"shared_conv_tokens: operands must be bf16 or fp16, got {xp.dtype}")
    w = _cuda(w, "w", xp.dtype)
    bias = _cuda(bias, "bias", torch.float32)
    bev_pos = _cuda(bev_pos, "bev_pos", torch.float32)
    xk = _cuda(xk, "xk", xp.dtype)
    xv = _cuda(xv, "xv", xp.dtype)
    B, rows, Cin = xp.shape
    Cout = w.shape[0]
    guard = conv_guard_rows(W)
    assert rows == 2 * guard + (H + 2) * (W + 2) and w.shape[1] == 9 * Cin and bev_pos.numel() == H * W * Cout
    lo, hi = (0, H * W) if tok_range is None else tok_range
    assert xk.shape[0] == B and xk.shape[2] == Cout and xk.shape[1] >= hi - lo and xv.shape == xk.shape
    lib = _lib.load()
    with torch.cuda.device(xp.device), _timed("shared_conv", xp):
        rc = lib.cmt_shared_conv_tokens(_ptr(xp), _ptr(w), _ptr(bias), _ptr(bev_pos), _ptr(xk), _ptr(xv), B, Cin, Cout, H, W,
                                        guard, xk.shape[1] * Cout, lo, hi, _stream(xp), _dt(xp.dtype))
    _lib.check(rc, "cmt_shared_conv_tokens")
    _count()


def gemm_segmented(A, Bm, bias, C, M, N, seg_k, seg_acol, seg_shift, *, a_row_off, a_rows, a_cols, lda, ldb, ldc, batch=1,
                   strideA=0, strideB=0, b_batch_div=1, strideC=0, alpha=1.0, relu=False, tag=None):
    """cmt_gemm_segmented: C[z] = act((sum_s A_z[m + a_row_off + shift_s, acol_s : acol_s + seg_k] . B_zb[n, s*seg_k : ...] + bias) alpha)."""
    A = _cuda(A, "A", torch.bfloat16)
    Bm = _cuda(Bm, "B", torch.bfloat16)
    C = _cuda(C, "C")
    if bias is not None:
        bias = _cuda(bias, "bias", torch.float32)
    n_seg = len(seg_acol)
    assert len(seg_shift) == n_seg
    acol = (ctypes.c_int * n_seg)(*[int(v) for v in seg_acol])
    shift = (ctypes.c_int * n_seg)(*[int(v) for v in seg_shift])
    lib = _lib.load()
    with torch.cuda.device(A.device), _timed(tag, A):
        rc = lib.cmt_gemm_segmented(_ptr(A), _ptr(Bm), _ptr(bias), _ptr(C), M, N, n_seg, seg_k, ctypes.cast(acol, ctypes.c_void_p),
                                    ctypes.cast(shift, ctypes.c_void_p), a_row_off, a_rows, a_cols, lda, ldb, ldc, batch, strideA,
                                    strideB, b_batch_div, strideC, float(alpha), GEMM_RELU if relu else 0, _dt(C.dtype), _stream(A))
    _lib.check(rc, "cmt_gemm_segmented")
    _count()
    return C


def gemm(A, Bm, bias, C, M, N, K, *, lda, ldb, ldc, cb=None, cb_stride=0, batch=1, strideA=0, strideB=0,
         strideC=0, alpha=1.0, relu=False, bias_per_row=False, force_simt=False, transpose_out=False,
         norm2_max=None, tag=None):
    """Raw cmt_gemm_bias_act: C = act((A B^T + bias) * alpha) with column-block output addressing.
    norm2_max: optional zero-initialised fp32 [batch, N/32] receiving max |row block|^2 (16-bit tensor-core path)."""
    A = _cuda(A, "A")
    Bm = _cuda(Bm, "B", A.dtype)
    C = _cuda(C, "C")
    if bias is not None:
        bias = _cuda(bias, "bias", torch.float32)
    flags = ((GEMM_RELU if relu else 0) | (GEMM_BIAS_PER_ROW if bias_per_row else 0) |
             (GEMM_FORCE_SIMT if force_simt else 0) | (GEMM_TRANSPOSE_OUT if transpose_out else 0))
    lib = _lib.load()
    with torch.cuda.device(A.device), _timed(tag, A):
        rc = lib.cmt_gemm_bias_act(_ptr(A), _ptr(Bm), _ptr(bias), _ptr(C), M, N, K, lda, ldb, ldc,
                                   cb if cb is not None else max(N, 1), cb_stride, batch, strideA, strideB, strideC,
                                   float(alpha), flags, _dt(A.dtype), _dt(C.dtype), _ptr(norm2_max), _stream(A))
    _lib.check(rc, "cmt_gemm_bias_act")
    _count()
    return C


def linear(x, weight, bias=None, *, relu=False, alpha=1.0, out_dtype=None, force_simt=False, tag=None):
    """act((x @ weight.T + bias) * alpha) -- F.linear replacement. x [..., K], weight [N, K]."""
    K = x.shape[-1]
    N = weight.shape[0]
    x2 = x.reshape(-1, K)
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    M = x2.shape[0]
    out_dtype = out_dtype or x.dtype
    out = torch.empty((M, N), dtype=out_dtype, device=x.device)
    gemm(x2, weight, bias, out, M, N, K, lda=K, ldb=K, ldc=N, alpha=alpha, relu=relu, force_simt=force_simt, tag=tag)
    return out.reshape(*x.shape[:-1], N)


def project_queries(x, w, bias, H, alpha, norm2_max=None):
    """Q = (x @ w.T + bias) * alpha, [B,Nq,H*32] in x.dtype, one GEMM batch per frame.
    norm2_max: optional zero-initialised fp32 [B,H] receiving max_query |q|^2 per (frame, head) -- with the key
    maxima of project_keys it bounds every attention score of the (frame, head) (static softmax shift)."""
    B, Nq, C = x.shape
    NO = w.shape[0]
    assert NO == H * HEAD_DIM
    out = torch.empty((B, Nq, NO), dtype=x.dtype, device=x.device)
    gemm(x, w, bias, out, Nq, NO, C, lda=C, ldb=C, ldc=NO, batch=B, strideA=Nq * C, strideB=0, strideC=Nq * NO,
         alpha=alpha, norm2_max=norm2_max)
    return out


def project_keys(xk, w, bias, n_layers, H, out=None, norm2_max=None):
    """K = xk @ w.T + bias for all layers at once, written in the per-head attention layout.
    xk [B,N_kv,C]; w [n_layers*H*32, C]; -> [B, n_layers, H, N_kv, 32].
    norm2_max: optional zero-initialised fp32 [B, n_layers*H] receiving max_token |k|^2 per (frame, layer, head)."""
    B, N_kv, C = xk.shape
    NO = w.shape[0]
    assert NO == n_layers * H * HEAD_DIM
    if out is None:
        out = torch.empty((B, n_layers, H, N_kv, HEAD_DIM), dtype=xk.dtype, device=xk.device)
    gemm(xk, w, bias, out, N_kv, NO, C, lda=C, ldb=C, ldc=HEAD_DIM, cb=HEAD_DIM, cb_stride=N_kv * HEAD_DIM,
         batch=B, strideA=N_kv * C, strideB=0, strideC=n_layers * H * N_kv * HEAD_DIM, norm2_max=norm2_max,
         tag="k_proj" if n_layers > 1 else None)
    return out


def project_values_t(xv, w, bias, n_layers, H, out=None):
    """V^T = w @ xv^T + bias[:,None] for all layers, token-contiguous: [B, n_layers, H, 32, ld] with
    ld = N_kv rounded up to 8 (TMA row pitch must be a multiple of 16 bytes)."""
    B, N_kv, C = xv.shape
    NO = w.shape[0]
    assert NO == n_layers * H * HEAD_DIM
    ld = (N_kv + 7) // 8 * 8
    if out is None:
        out = torch.empty((B, n_layers, H, HEAD_DIM, ld), dtype=xv.dtype, device=xv.device)
    if xv.dtype != torch.float32:
        # tokens on the M side like the K projection (the CTA keeps its slice of W_v resident in shared memory and
        # streams token tiles), each [tokens, 32] head block stored transposed
        gemm(xv, w, bias, out, N_kv, NO, C, lda=C, ldb=C, ldc=ld, cb=HEAD_DIM, cb_stride=HEAD_DIM * ld, batch=B,
             strideA=N_kv * C, strideB=0, strideC=NO * ld, transpose_out=True, tag="v_proj" if n_layers > 1 else None)
    else:
        gemm(w, xv, bias, out, NO, N_kv, C, lda=C, ldb=C, ldc=ld, batch=B, strideA=0, strideB=N_kv * C,
             strideC=NO * ld, bias_per_row=True)
    return out


_ws_cache = {}


def _workspace(dev, nbytes):
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=dev)
        _ws_cache[key] = buf
    return buf


def cross_attn(q, k, vt, layer, *, kv_begin=0, kv_end=None, o_dtype=None, return_lse=False, simt=False,
               key_keep=None, q_norm2=None, k_norm2=None, tag="cross_attn", out=None, lse_out=None):
    """K3 (attention.py:46-92). q [B,Nq,H*32] pre-scaled by log2(e)/sqrt(32); k [B,L,H,N_kv,32];
    vt [B,L,H,32,ld]; attends tokens [kv_begin,kv_end) of layer `layer`. -> o [B,Nq,H*32] (, lse [B,H,Nq]).
    key_keep: optional [B,N_kv] bool/uint8, True = attend (the key_padding_mask of attention.py:76-90, whose
    unpad_input keeps the True entries); a contiguous bool mask is read in place (no conversion launch).
    q_norm2 [B,H] / k_norm2 [B,L,H] fp32 (from the projections' norm2_max): enables the static softmax shift.
    q, k, vt: bf16 or fp16 (tcgen05 kernel) or fp32 (CUDA-core kernel); o_dtype: fp32 or q's dtype."""
    q = _cuda(q, "q")
    k = _cuda(k, "k", q.dtype)
    vt = _cuda(vt, "vt", q.dtype)
    B, Nq, HD = q.shape
    H = HD // HEAD_DIM
    _, L, Hk, N_kv, _ = k.shape
    ld = vt.shape[-1]
    assert Hk == H and vt.shape[:4] == (B, L, H, HEAD_DIM)
    kv_end = N_kv if kv_end is None else kv_end
    o_dtype = o_dtype or q.dtype
    if out is not None:   # caller-provided output rows (a slice of a larger [frames, Nq, H*32] buffer)
        o = _cuda(out, "out", o_dtype)
        assert o.shape == (B, Nq, HD)
    else:
        o = torch.empty((B, Nq, HD), dtype=o_dtype, device=q.device)
    if lse_out is not None:
        lse = _cuda(lse_out, "lse_out", torch.float32)
        assert lse.shape == (B, H, Nq)
        return_lse = True
    else:
        lse = torch.empty((B, H, Nq), dtype=torch.float32, device=q.device) if return_lse else None
    esz = q.element_size()
    kp = ctypes.c_void_p(k.data_ptr() + layer * H * N_kv * HEAD_DIM * esz)
    vp = ctypes.c_void_p(vt.data_ptr() + layer * H * HEAD_DIM * ld * esz)
    lib = _lib.load()
    dt = _dt(q.dtype)
    if simt and dt == CMT_BF16:
        dt = CMT_BF16_SIMT
    elif simt and dt == CMT_F16:
        raise TypeError("cross_attn(simt=True): fp16 operands run on the tcgen05 kernel only")
    tc = dt in (CMT_BF16, CMT_F16)
    ws, ws_bytes = None, 0
    if tc:
        with torch.cuda.device(q.device):
            ws_bytes = int(lib.cmt_cross_attn_workspace_bytes(B, H, Nq, kv_end - kv_begin))
        ws = _workspace(q.device, ws_bytes)
    if key_keep is not None:
        key_keep = _cuda(key_keep, "key_keep")
        assert key_keep.shape == (B, N_kv), f"key_keep must be [B, N_kv] = {(B, N_kv)}, got {tuple(key_keep.shape)}"
        key_keep = key_keep.contiguous().view(torch.uint8) if key_keep.dtype == torch.bool else key_keep.to(torch.uint8).contiguous()
    qn = kn = None
    kn_stride = 0
    if q_norm2 is not None and k_norm2 is not None and tc and not FORCE_ONLINE_SOFTMAX:
        qn = _cuda(q_norm2, "q_norm2", torch.float32)
        k_norm2 = _cuda(k_norm2, "k_norm2", torch.float32)
        assert qn.shape == (B, H) and k_norm2.shape == (B, L, H)
        kn = ctypes.c_void_p(k_norm2.data_ptr() + layer * H * 4)
        kn_stride = L * H
    ev = _profile.get(tag)
    if ev is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    with torch.cuda.device(q.device):
        rc = lib.cmt_cross_attn_fwd(_ptr(q), kp, vp, _ptr(o), _ptr(lse), B, H, Nq, N_kv, kv_begin, kv_end, HD,
                                    L * H * N_kv * HEAD_DIM, N_kv * HEAD_DIM, L * H * HEAD_DIM * ld, HEAD_DIM * ld,
                                    ld, _ptr(key_keep), _ptr(qn), kn, kn_stride, dt, _dt(o_dtype), _ptr(ws), ws_bytes,
                                    _stream(q))
    if ev is not None:
        e1.record()
        ev.append((e0, e1))
    _lib.check(rc, "cmt_cross_attn_fwd")
    # tcgen05 path: [mask pack] + [static-shift kernel] + online kernel + merge
    _count((2 if tc else 1) + (1 if key_keep is not None and tc else 0) + (1 if qn is not None else 0))
    return (o, lse) if return_lse else o


def lse_merge(o_parts, lse_parts, o_dtype=torch.bfloat16, want_lse=True):
    """Merge G partial attention results: o_parts [G,B,Nq,H*32] fp32, lse_parts [G,B,H,Nq] fp32."""
    o_parts = _cuda(o_parts, "o_parts", torch.float32)
    lse_parts = _cuda(lse_parts, "lse_parts", torch.float32)
    G, B, Nq, HD = o_parts.shape
    H = HD // HEAD_DIM
    o = torch.empty((B, Nq, HD), dtype=o_dtype, device=o_parts.device)
    lse = torch.empty((B, H, Nq), dtype=torch.float32, device=o_parts.device) if want_lse else None
    lib = _lib.load()
    with torch.cuda.device(o_parts.device):
        rc = lib.cmt_lse_merge(_ptr(o_parts), _ptr(lse_parts), _ptr(o), _ptr(lse), G, B, H, Nq, 0, 0, _dt(o_dtype),
                               _stream(o_parts))
    _lib.check(rc, "cmt_lse_merge")
    _count()
    return o, lse


def packed_partial(B, Nq, H, device):
    """One (O | LSE) record: a flat fp32 buffer with views o [B,Nq,H*32] and lse [B,H,Nq] -- what a rank contributes to the
    single all-gather of a KV-token-split decoder layer."""
    n_o, n_l = B * Nq * H * HEAD_DIM, B * H * Nq
    buf = torch.empty((n_o + n_l,), dtype=torch.float32, device=device)
    return buf, buf[:n_o].view(B, Nq, H * HEAD_DIM), buf[n_o:].view(B, H, Nq)


def lse_merge_packed(parts, G, B, Nq, H, o_dtype=torch.bfloat16):
    """Merge the G packed (O | LSE) records of an all-gather: parts fp32 [G * (B*Nq*H*32 + B*H*Nq)] -> o [B,Nq,H*32]."""
    parts = _cuda(parts, "parts", torch.float32)
    n_o, n_l = B * Nq * H * HEAD_DIM, B * H * Nq
    assert parts.numel() == G * (n_o + n_l)
    o = torch.empty((B, Nq, H * HEAD_DIM), dtype=o_dtype, device=parts.device)
    lib = _lib.load()
    with torch.cuda.device(parts.device):
        rc = lib.cmt_lse_merge(_ptr(parts), ctypes.c_void_p(parts.data_ptr() + n_o * 4), _ptr(o), None, G, B, H, Nq, n_o + n_l,
                               n_o + n_l, _dt(o_dtype), _stream(parts))
    _lib.check(rc, "cmt_lse_merge")
    _count()
    return o


def lse_merge_peer(record_ptrs, ctx_ptrs, arrive_ptrs, state_ptr, rank, B, Nq, H, device, o_dtype=torch.bfloat16, scatter=-1):
    """Exchange + merge + redistribution of the KV-token split in one kernel over peer memory (cmt_lse_merge_peer):
    record_ptrs / ctx_ptrs / arrive_ptrs are the G ranks' device addresses (ints) of this exchange's packed record, of
    the context buffer and of the counters, all mapped into this process (parallel.PeerExchange).  Collective over the
    group; the merged context is in this rank's context buffer when the kernel has run.  scatter: 1 = each rank merges
    1/G of the rows and stores them to all ranks, 0 = each rank merges all rows for itself, -1 = by group size."""
    G = len(record_ptrs)
    assert len(arrive_ptrs) == G and len(ctx_ptrs) == G and 0 <= rank < G
    recs = (ctypes.c_void_p * G)(*record_ptrs)
    ctxs = (ctypes.c_void_p * G)(*ctx_ptrs)
    arrs = (ctypes.c_void_p * G)(*arrive_ptrs)
    lib = _lib.load()
    with torch.cuda.device(device):
        rc = lib.cmt_lse_merge_peer(recs, ctxs, arrs, ctypes.c_void_p(state_ptr), rank, G, B, H, Nq, _dt(o_dtype), int(scatter),
                                    ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream))
    _lib.check(rc, "cmt_lse_merge_peer")
    _count()


def coop_max(a, b):
    """max(nan_to_num(a), nan_to_num(b)) (cmt_head_coop.py:358,383-389)."""
    a = _cuda(a, "a", torch.float32)
    b = _cuda(b, "b", torch.float32)
    assert a.shape == b.shape
    out = torch.empty_like(a)
    lib = _lib.load()
    with torch.cuda.device(a.device):
        rc = lib.cmt_coop_max(_ptr(a), _ptr(b), _ptr(out), a.numel(), _stream(a))
    _lib.check(rc, "cmt_coop_max")
    _count()
    return out


def add_layernorm(x, r, gamma, beta, eps=1e-5, *, gamma2=None, beta2=None, y2=None, add=None, lp_dtype=None,
                  want_ylp=False, want_yadd=False, rows=None):
    """Fused residual add + LayerNorm (+ optional second LayerNorm, + low-precision copies of y and y+add).
    x, r, add: [..., 256] fp32.  Returns (y, y2, ylp, yadd) with None for outputs not requested."""
    x = _cuda(x, "x", torch.float32)
    C = x.shape[-1]
    flags = 0
    shape = x.shape
    if rows is not None:   # x is ONE row [C] shared by every row of the [*rows, C] output
        assert x.numel() == C and r is None
        flags = _lib.LN_X_ROW_BROADCAST
        shape = (*rows, C)
    M = int(math.prod(shape[:-1]))
    y = torch.empty(shape, dtype=torch.float32, device=x.device)
    if y2 is None and gamma2 is not None:
        y2 = torch.empty_like(y)
    lp_dtype = lp_dtype or torch.float32
    ylp = torch.empty(shape, dtype=lp_dtype, device=x.device) if want_ylp else None
    yadd = torch.empty(shape, dtype=lp_dtype, device=x.device) if want_yadd else None
    lib = _lib.load()
    with torch.cuda.device(x.device):
        rc = lib.cmt_add_layernorm(_ptr(x), _ptr(r), _ptr(gamma), _ptr(beta), float(eps), M, C, _ptr(y), _ptr(gamma2),
                                   _ptr(beta2), _ptr(y2), _ptr(add), _ptr(ylp), _ptr(yadd), _dt(lp_dtype), flags, _stream(x))
    _lib.check(rc, "cmt_add_layernorm")
    _count()
    return y, y2, ylp, yadd


def split3(a, b=None, want_merged=False, stacked_nodes=False, node_valid=None):
    """Three-term bf16 split of the stacked decoder outputs with nan_to_num (and the cooperative max over two stacks)
    fused in (cmt_split3_bf16).  a, b: [L,B,Nq,256] fp32 -> [L*B, Nq+2, 768] bf16 (, merged [L,B,Nq,256] fp32).
    stacked_nodes: `a` is [L,2B,Nq,256] holding the first node's frames then the second node's in every layer (one
    decoder pass over both nodes); the max is taken between frame b and frame B + b.
    node_valid: optional torch.bool [2, B] on a's device, row 0 for the first node (`a`, or the first half of the stack)
    and row 1 for the second; frame b takes the max with both nodes present, the present node's rows with one, and zero
    rows with none.  An absent node's rows are not read."""
    a = _cuda(a, "a", torch.float32)
    L, B, Nq, C = a.shape
    frames, lstride = 0, 0
    bptr = None
    if stacked_nodes:
        assert b is None and B % 2 == 0
        B //= 2
        frames, lstride = B, 2 * B * Nq
        bptr = ctypes.c_void_p(a.data_ptr() + B * Nq * C * 4)
    elif b is not None:
        b = _cuda(b, "b", torch.float32)
        assert b.shape == a.shape
        bptr = _ptr(b)
    if node_valid is not None:
        if bptr is None:
            raise ValueError("split3: node_valid needs a second node (b or stacked_nodes=True)")
        node_valid = check_node_valid(node_valid, B, a.device)
        if not stacked_nodes:   # dense layout, addressed per frame
            frames, lstride = B, B * Nq
    out = torch.empty((L * B, Nq + 2, 3 * C), dtype=torch.bfloat16, device=a.device)
    merged = torch.empty((L, B, Nq, C), dtype=torch.float32, device=a.device) if want_merged else None
    lib = _lib.load()
    with torch.cuda.device(a.device):
        rc = lib.cmt_split3_bf16(_ptr(a), bptr, _ptr(out), _ptr(merged), L * B, Nq, C, frames, lstride, _stream(a),
                                 _ptr(node_valid))
    _lib.check(rc, "cmt_split3_bf16")
    _count()
    return (out, merged) if want_merged else out


def task_head_tail(h, gamma, beta, w2, b2, eps, ksize=1, Nq=None, ref_logit=None, dec_comp=None, dec_scale=None,
                   dec_offset=None, head_couts=None):
    """sum_t ReLU(GroupLN(h[q+t-k/2]) * gamma + beta) . w2[:, t] + b2 for every (layer, row, output head) in one launch,
    plus the optional reference-point decode (cmt_head.py:116-150, :53-94, :501-513).  h [L,M,NH,64] fp32; gamma/beta
    [L,NH,64]; w2 [L,NH,CMAX,ksize,64]; b2 [L,NH,CMAX] -> [L,M,NH,CMAX] fp32, or with head_couts=[c_0, ...] a list of
    NH contiguous tensors [L,M,c_i] (views of one buffer: one device->host copy moves them all)."""
    h = _cuda(h, "h", torch.float32)
    L, M, NH, HC = h.shape
    CMAX = w2.shape[2]
    if w2.dim() == 4:
        w2 = w2.unsqueeze(3)
    args = [_cuda(t, n, torch.float32) for t, n in ((gamma, "gamma"), (beta, "beta"), (w2, "w2"), (b2, "b2"))]
    assert args[0].shape == (L, NH, HC) and args[1].shape == (L, NH, HC)
    assert args[2].shape == (L, NH, CMAX, ksize, HC) and args[3].shape == (L, NH, CMAX)
    Nq = M if Nq is None else Nq
    if ref_logit is not None:
        ref_logit = _cuda(ref_logit, "ref_logit", torch.float32)
        assert ref_logit.shape == (M, 3)
        dec_comp = _cuda(dec_comp, "dec_comp", torch.int32)
        dec_scale = _cuda(dec_scale, "dec_scale", torch.float32)
        dec_offset = _cuda(dec_offset, "dec_offset", torch.float32)
        assert dec_comp.numel() == NH * CMAX and dec_scale.numel() == NH * CMAX and dec_offset.numel() == NH * CMAX
    offs = couts = None
    if head_couts is not None:
        assert len(head_couts) == NH and NH <= 8
        sizes = [L * M * int(c) for c in head_couts]
        starts = [sum(sizes[:i]) for i in range(NH)]
        out = torch.empty((sum(sizes),), dtype=torch.float32, device=h.device)
        offs = (ctypes.c_int64 * NH)(*starts)
        couts = (ctypes.c_int * NH)(*[int(c) for c in head_couts])
    else:
        out = torch.empty((L, M, NH, CMAX), dtype=torch.float32, device=h.device)
    lib = _lib.load()
    with torch.cuda.device(h.device):
        rc = lib.cmt_task_head_tail(_ptr(h), *[_ptr(a) for a in args], _ptr(out), L, M, NH, HC, CMAX, float(eps), ksize, Nq,
                                    _ptr(ref_logit), _ptr(dec_comp), _ptr(dec_scale), _ptr(dec_offset),
                                    None if offs is None else ctypes.cast(offs, ctypes.c_void_p),
                                    None if couts is None else ctypes.cast(couts, ctypes.c_void_p), _stream(h))
    _lib.check(rc, "cmt_task_head_tail")
    _count()
    if head_couts is not None:
        return [out[s:s + n].view(L, M, int(c)) for s, n, c in zip(starts, sizes, head_couts)]
    return out


BOX_DECODE_FIELDS = ("cls_logits", "center", "height", "dim", "rot", "vel")
_BOX_DECODE_WIDTH = {"center": 2, "height": 1, "dim": 3, "rot": 2, "vel": 2}


def bbox_topk_decode(tasks, num_classes, max_num, post_center_range, score_threshold=None, bottom_center=False,
                     node_valid=None):
    """MultiTaskBBoxCoder.decode_single for every frame in one launch (cmt_bbox_topk_decode; multi_task_bbox_coder.py:46-141,
    util.py:37-68, with bottom_center the z shift of cmt_head.py:912).  tasks: one dict per task of its last decoder
    layer's fp32 outputs {cls_logits [B,Nq,C_t], center [B,Nq,2], height [B,Nq,1], dim [B,Nq,3], rot [B,Nq,2],
    vel [B,Nq,2]}.  score_threshold: applied (strict >) only when truthy, like the coder.  Returns the fixed-shape dict
    {boxes [B,K,9] fp32, scores [B,K] fp32, labels [B,K] int64, count [B] int32, topk_index [B,K] int64}: the kept
    detections of frame b are the first count[b] slots, in score order; the other slots are zero with label -1.
    node_valid: optional torch.bool [n_nodes, B] on the outputs' device; a frame none of whose nodes is present keeps
    nothing (count 0, every slot zero with label -1) and its topk_index is -1."""
    if not 1 <= len(tasks) <= 8:
        raise ValueError(f"bbox_topk_decode: {len(tasks)} tasks (1..8 supported)")
    B, Nq = tasks[0]["cls_logits"].shape[:2]
    ptrs, classes, keep = [], [], []
    for ti, d in enumerate(tasks):
        for name in BOX_DECODE_FIELDS:
            t = d[name]
            if not isinstance(t, torch.Tensor) or not t.is_cuda:
                raise _lib.CmtLibraryError(f"task {ti} {name} must be a CUDA tensor: libcmtcoop_b200 has no CPU fallback")
            if t.dtype != torch.float32:
                raise TypeError(f"task {ti} {name} must be torch.float32, got {t.dtype}")
            width = _BOX_DECODE_WIDTH.get(name, t.shape[-1])
            if t.dim() != 3 or tuple(t.shape) != (B, Nq, width) or t.device != tasks[0]["cls_logits"].device:
                raise ValueError(f"task {ti} {name}: expected [{B},{Nq},{width}] on {tasks[0]['cls_logits'].device}, "
                                 f"got {tuple(t.shape)} on {t.device}")
            t = t.contiguous()
            keep.append(t)
            ptrs.append(t.data_ptr())
        classes.append(int(d["cls_logits"].shape[-1]))
    if sum(classes) != num_classes:
        raise ValueError(f"bbox_topk_decode: num_classes {num_classes} != sum of the tasks' classes {sum(classes)}")
    if len(post_center_range) != 6:
        raise ValueError("post_center_range must have 6 entries")
    K = int(max_num)   # 1 <= K <= min(1024, Nq * num_classes), checked by the library
    dev = keep[0].device
    if node_valid is not None:
        node_valid = check_node_valid(node_valid, B, dev, n_nodes=None)
    out = dict(boxes=torch.empty((B, K, 9), dtype=torch.float32, device=dev),
               scores=torch.empty((B, K), dtype=torch.float32, device=dev),
               labels=torch.empty((B, K), dtype=torch.int64, device=dev),
               count=torch.empty((B,), dtype=torch.int32, device=dev),
               topk_index=torch.empty((B, K), dtype=torch.int64, device=dev))
    p_arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
    c_arr = (ctypes.c_int * len(classes))(*classes)
    lib = _lib.load()
    with torch.cuda.device(dev):
        rc = lib.cmt_bbox_topk_decode(ctypes.cast(p_arr, ctypes.c_void_p), ctypes.cast(c_arr, ctypes.c_void_p), len(tasks), B,
                                      Nq, int(num_classes), K, ctypes.cast(_pc(post_center_range), ctypes.c_void_p),
                                      float(score_threshold or 0.0), 1 if score_threshold else 0, 1 if bottom_center else 0,
                                      *[_ptr(out[n]) for n in ("boxes", "scores", "labels", "count", "topk_index")],
                                      _stream(keep[0]), _ptr(node_valid),
                                      0 if node_valid is None else node_valid.shape[0])
    _lib.check(rc, "cmt_bbox_topk_decode")
    _count()
    return out
