"""The fp16 compute precision (`set_precision('fp16')`): the tcgen05 GEMM and attention kernels with fp16 operands, the
kernels that round their outputs to fp16, shared_conv, and the six heads at the mini and BASELINE config shapes.

Tolerances are the bf16 tests' scaled to fp16's unit roundoff: a 16-bit output rounding is 2^-11 relative in fp16
against 2^-8 in bf16, so the bf16 bound 4e-3 becomes 5e-4.  The attention core is compared with the fp32 CUDA-core
kernel fed the same fp16-rounded operands, upcast (fp16 P: 2^-11 per weight, averaged over many keys).
End to end, fp16 must stay inside the 1e-2 rel-L2 budget and reach at most half the bf16 error measured on the same
inputs in the same test."""
import math
import os

import numpy as np
import pytest
import torch

from cmtcoop_b200 import ops, synth
from cmtcoop_b200.plugin import build_head, fused_decoder
from oracle import cmt_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NUSC = synth.NUSC_RANGE
NAMES = ("center", "height", "dim", "rot", "vel", "cls_logits")
TOL16 = 5e-4            # one fp16 rounding of an output
ATTN_TOL = 1e-3         # fp16 P against the fp32 CUDA-core kernel on the same operands
LSE_TOL = 1e-3          # the row sums are fp32 in both precisions: same bound as bf16


def _rel(a, b):
    return O.rel_l2(a.detach().cpu().double(), b.detach().cpu().double())


# ------------------------------------------------------------------------------------------ GEMM
GEMM_CASES = [
    # M, N, K, relu, bias, alpha
    (300, 256, 192, True, True, 1.0),
    (257, 256, 1024, False, True, 1.0),
    (900, 256, 256, False, True, 0.255),
    (129, 40, 64, False, False, 1.0),      # N % 32 != 0: masked stores
]


@pytest.mark.parametrize("M,N,K,relu,bias,alpha", GEMM_CASES)
def test_gemm_fp16_plain(M, N, K, relu, bias, alpha):
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g).half()
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).half()
    b = torch.randn(N, generator=g) if bias else None
    want = (a.double() @ w.double().t() + (b.double() if bias else 0)) * alpha
    if relu:
        want = want.clamp_min(0)
    kw = dict(relu=relu, alpha=alpha)
    got32 = ops.linear(a.to(DEV), w.to(DEV), None if b is None else b.to(DEV), out_dtype=torch.float32, **kw)
    got16 = ops.linear(a.to(DEV), w.to(DEV), None if b is None else b.to(DEV), **kw)
    torch.cuda.synchronize()
    assert got16.dtype == torch.float16
    assert _rel(got32, want) < 5e-6          # fp32 accumulation of exact fp16 products
    assert _rel(got16, want) < TOL16
    assert torch.equal(got16.cpu(), got32.cpu().half())   # the fp16 output is one rounding of the fp32 one


@pytest.mark.parametrize("M,N,K,batch,ldc,cb,cb_stride,strideC", [
    (200, 72, 128, 1, 80, None, 0, 0),                      # 256-bit chunks + ragged tail
    (150, 256, 64, 1, 260, None, 0, 0),                     # row pitch not a multiple of 32 bytes
    (170, 128, 64, 2, 32, 32, 170 * 32 + 4, 4 * (170 * 32 + 4)),   # column blocks, unaligned cb_stride
])
def test_gemm_fp16_output_layouts(M, N, K, batch, ldc, cb, cb_stride, strideC):
    g = torch.Generator().manual_seed(M + N + K + batch)
    a = torch.randn(batch, M, K, generator=g).half()
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).half()
    b = torch.randn(N, generator=g)
    want = (a.double() @ w.double().t() + b.double()) * 0.5
    cb = cb or N
    z, m, n = torch.meshgrid(torch.arange(batch), torch.arange(M), torch.arange(N), indexing="ij")
    idx = z * strideC + (n // cb) * cb_stride + m * ldc + n % cb
    size = int(idx.max()) + 1 + 8
    C = torch.full((size,), -7.0, dtype=torch.float16, device=DEV)
    ops.gemm(a.to(DEV), w.to(DEV), b.to(DEV), C, M, N, K, lda=K, ldb=K, ldc=ldc, cb=cb, cb_stride=cb_stride, batch=batch,
             strideA=M * K if batch > 1 else 0, strideC=strideC, alpha=0.5)
    torch.cuda.synchronize()
    out = C.cpu().float()
    assert _rel(out[idx], want) < TOL16
    untouched = torch.ones(size, dtype=torch.bool)
    untouched[idx.flatten()] = False
    assert bool((out[untouched] == -7.0).all())


def test_gemm_fp16_head_layouts_and_norm2_max():
    """Column-block K layout [B,L,H,N_kv,32], transposed V^T [B,L,H,32,ld] and the norm2_max epilogue, fp16 operands."""
    B, N_kv, C, L, H = 2, 333, 256, 2, 8
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, N_kv, C, generator=g).half()
    w = (torch.randn(L * H * 32, C, generator=g) / 16).half()
    b = torch.randn(L * H * 32, generator=g)
    want = x.double() @ w.double().t() + b.double()                           # [B,N_kv,L*H*32]
    kn2 = torch.zeros(B, L, H, device=DEV)
    k = ops.project_keys(x.to(DEV), w.to(DEV), b.to(DEV), L, H, norm2_max=kn2)
    assert k.dtype == torch.float16 and k.shape == (B, L, H, N_kv, 32)
    assert _rel(k.float(), want.view(B, N_kv, L, H, 32).permute(0, 2, 3, 1, 4)) < TOL16
    want_n2 = want.view(B, N_kv, L, H, 32).pow(2).sum(-1).amax(1)
    assert torch.allclose(kn2.cpu().double(), want_n2, rtol=1e-4)              # from the fp32 accumulators
    vt = ops.project_values_t(x.to(DEV), w.to(DEV), b.to(DEV), L, H)
    assert vt.dtype == torch.float16 and vt.shape[-1] == 336
    assert _rel(vt[..., :N_kv].float(), want.view(B, N_kv, L, H, 32).permute(0, 2, 3, 4, 1)) < TOL16
    qn2 = torch.zeros(B, H, device=DEV)
    q = ops.project_queries(x[:, :300].contiguous().to(DEV), w[:H * 32].contiguous().to(DEV), b[:H * 32].contiguous().to(DEV),
                            H, 0.5, norm2_max=qn2)
    want_q = (want[:, :300, :H * 32]) * 0.5
    assert _rel(q.float(), want_q) < TOL16
    assert torch.allclose(qn2.cpu().double(), want_q.view(B, 300, H, 32).pow(2).sum(-1).amax(1), rtol=1e-4)


def test_gemm_fp16_rejects_mixed_dtypes():
    from cmtcoop_b200 import _lib
    a = torch.zeros(64, 64, dtype=torch.float16, device=DEV)
    with pytest.raises(_lib.CmtLibraryError):   # fp16 operands, bf16 output
        ops.linear(a, a, out_dtype=torch.bfloat16)
    with pytest.raises(_lib.CmtLibraryError):   # fp16 operands on the CUDA-core kernel
        ops.linear(a, a, out_dtype=torch.float32, force_simt=True)


# ------------------------------------------------------------------------------------------ attention
def _attn_operands(B, Nq, N_kv, seed, q_scale=0.6, k_scale=1.0):
    g = torch.Generator().manual_seed(seed)
    q = (torch.randn(B, Nq, 8 * 32, generator=g) * q_scale).half()
    k = (torch.randn(B, 1, 8, N_kv, 32, generator=g) * k_scale).half()
    ld = (N_kv + 7) // 8 * 8
    vt = torch.zeros(B, 1, 8, 32, ld)
    vt[..., :N_kv] = torch.randn(B, 1, 8, 32, N_kv, generator=g)
    return q, k, vt.half()


def _norms(q, k):
    B, Nq, HD = q.shape
    qn = q.float().view(B, Nq, HD // 32, 32).pow(2).sum(-1).amax(1).contiguous()
    kn = k.float().pow(2).sum(-1).amax(-1).contiguous()
    return qn, kn


def _bound(qn, kn):
    return (qn * kn[:, 0]).sqrt() * 1.0079 + 1e-3


def _both(q, k, vt, **kw):
    """(fp16 tcgen05 result, fp32 CUDA-core result on the same operands upcast), each (o fp32, lse)."""
    d = lambda t: t.to(DEV)
    got = ops.cross_attn(d(q), d(k), d(vt), 0, o_dtype=torch.float32, return_lse=True, **kw)
    kw.pop("q_norm2", None)
    kw.pop("k_norm2", None)
    ref = ops.cross_attn(d(q).float(), d(k).float(), d(vt).float(), 0, o_dtype=torch.float32, return_lse=True, **kw)
    torch.cuda.synchronize()
    return got, ref


@pytest.mark.parametrize("B,Nq,N_kv,lo,hi", [
    (1, 900, 5000, 0, None),      # reference query count: 7 full tiles + a 4-row tail
    (2, 200, 4096, 1024, 3000),   # KV sub-range
    (1, 1, 130, 0, None),
])
@pytest.mark.parametrize("norms", [False, True])
def test_attention_fp16(B, Nq, N_kv, lo, hi, norms):
    hi = N_kv if hi is None else hi
    q, k, vt = _attn_operands(B, Nq, N_kv, Nq + N_kv)
    kw = dict(kv_begin=lo, kv_end=hi)
    if norms:
        qn, kn = _norms(q, k)
        kw.update(q_norm2=qn.to(DEV), k_norm2=kn.to(DEV))
    (o, lse), (o_ref, lse_ref) = _both(q, k, vt, **kw)
    assert _rel(o, o_ref) < ATTN_TOL
    assert float((lse - lse_ref).abs().max()) < LSE_TOL
    o16 = ops.cross_attn(q.to(DEV), k.to(DEV), vt.to(DEV), 0, o_dtype=torch.float16, **kw)
    torch.cuda.synchronize()
    assert o16.dtype == torch.float16 and torch.equal(o16, o.half())


def test_attention_fp16_static_limit_is_14():
    """One call holding (frame, head) items with a score bound <= 14 (the fp16 static kernel) and items with a bound in
    (14, 60] (the online kernel in fp16, where bf16 would take the static one), with and without a key mask."""
    B, Nq, N_kv = 2, 300, 3000
    q, k, vt = _attn_operands(B, Nq, N_kv, 23, q_scale=0.15)
    q[1] = (q[1].float() * 4.0).half()
    qn, kn = _norms(q, k)
    bound = _bound(qn, kn)
    assert float(bound[0].max()) <= 14.0
    assert float(bound[1].min()) > 14.0 and float(bound[1].max()) <= 60.0
    g = torch.Generator().manual_seed(4)
    keep = torch.rand(B, N_kv, generator=g) > 0.25
    keep[0, :130] = False
    for key_keep in (None, keep.to(DEV)):
        (o, lse), (o_ref, lse_ref) = _both(q, k, vt, key_keep=key_keep, q_norm2=qn.to(DEV), k_norm2=kn.to(DEV))
        assert _rel(o, o_ref) < ATTN_TOL, key_keep is not None
        assert float((lse - lse_ref).abs().max()) < LSE_TOL
        o_online = ops.cross_attn(q.to(DEV), k.to(DEV), vt.to(DEV), 0, o_dtype=torch.float32, key_keep=key_keep)
        torch.cuda.synchronize()
        assert _rel(o, o_online) < ATTN_TOL


@pytest.mark.parametrize("masked", [False, True])
def test_attention_fp16_scores_at_the_limit(masked):
    """Scores at exactly +-14 on the static kernel: one key at +14 (weight 2^14), every other key at -14 (2^-14, the
    smallest normal fp16).  Norms just inside the limit put every item on the static kernel.  No inf, no NaN, and the
    dominant key's value comes out."""
    B, Nq, N_kv, H = 1, 130, 700, 8
    q = torch.zeros(B, Nq, H * 32)
    q[..., 0::32] = 1.0
    k = torch.zeros(B, 1, H, N_kv, 32)
    k[..., 0] = -14.0
    k[..., 333, 0] = 14.0
    g = torch.Generator().manual_seed(3)
    vt = torch.randn(B, 1, H, 32, (N_kv + 7) // 8 * 8, generator=g)
    q, k, vt = q.half(), k.half(), vt.half()
    qn = torch.ones(B, H)
    kn = torch.full((B, 1, H), ((14.0 - 2e-3) / 1.0079) ** 2)
    assert float(_bound(qn, kn).max()) <= 14.0
    keep = None
    if masked:
        keep = torch.ones(B, N_kv, dtype=torch.bool)
        keep[:, 500:] = False
        keep = keep.to(DEV)
    (o, lse), (o_ref, lse_ref) = _both(q, k, vt, key_keep=keep, q_norm2=qn.to(DEV), k_norm2=kn.to(DEV))
    assert torch.isfinite(o).all() and torch.isfinite(lse).all()
    assert _rel(o, o_ref) < ATTN_TOL
    assert float((lse - lse_ref).abs().max()) < LSE_TOL
    v = vt[0, 0, :, :, 333].float().reshape(H * 32)
    assert torch.allclose(o[0].cpu(), v.expand(Nq, -1), rtol=2e-3, atol=2e-3)


def test_attention_fp16_no_attended_key():
    """A query with no attended key gets o = 0 and lse = -inf in fp16 as well: frame 0 has every key padded, frame 1
    has keys only outside the token range, frame 2 is ordinary."""
    B, Nq, N_kv, lo, hi = 3, 417, 1500, 600, 1337
    q, k, vt = _attn_operands(B, Nq, N_kv, 7, q_scale=0.15)   # score bound < 14: the norms select the static kernel
    g = torch.Generator().manual_seed(8)
    keep = torch.rand(B, N_kv, generator=g) > 0.3
    keep[0] = False
    keep[1, lo:hi] = False
    qn, kn = _norms(q, k)
    for norms in ({}, dict(q_norm2=qn.to(DEV), k_norm2=kn.to(DEV))):
        (o, lse), (o_ref, lse_ref) = _both(q, k, vt, key_keep=keep.to(DEV), kv_begin=lo, kv_end=hi, **norms)
        o, lse = o.cpu(), lse.cpu()
        assert torch.equal(o[:2], torch.zeros_like(o[:2]))
        assert bool(torch.isneginf(lse[:2]).all())
        assert _rel(o[2], o_ref[2]) < ATTN_TOL
        assert float((lse[2] - lse_ref[2].cpu()).abs().max()) < LSE_TOL


# ------------------------------------------------------------------------------------------ output rounding
def _mats(n, seed=0, pad_w=160.0, pad_h=96.0):
    rng = np.random.RandomState(seed)
    l2i = np.stack(synth.camera_matrices(n, rng, pad_w, pad_h))
    return l2i, np.linalg.inv(l2i).astype(np.float32)


@pytest.mark.parametrize("depth", [64, 24])   # 256-bit stores (D % 16 == 0) and 128-bit stores
def test_ray_pe_fp16(depth):
    _, i2l = _mats(3, 1)
    m = torch.from_numpy(i2l).to(DEV)
    got32 = ops.ray_pe(m, 6, 10, depth, 96.0, 160.0, NUSC, out_dtype=torch.float32)
    got16 = ops.ray_pe(m, 6, 10, depth, 96.0, 160.0, NUSC, out_dtype=torch.float16)
    assert got16.dtype == torch.float16 and torch.equal(got16, got32.half())


def test_ray_query_pe_pos2embed_and_view_sum_fp16():
    B, V, Nq = 2, 3, 77
    rng = np.random.RandomState(5)
    l2i = np.stack([np.stack(synth.camera_matrices(V, rng, 160.0, 96.0)) for _ in range(B)])
    l32, i32 = torch.from_numpy(l2i).float().to(DEV), torch.from_numpy(np.linalg.inv(l2i)).float().to(DEV)
    ref = torch.from_numpy(rng.uniform(0, 1, (B, Nq, 3)).astype(np.float32)).to(DEV)
    f32, m32 = ops.ray_query_pe(ref, l32, i32, 64, 96.0, 160.0, NUSC, out_dtype=torch.float32)
    f16, m16 = ops.ray_query_pe(ref, l32, i32, 64, 96.0, 160.0, NUSC, out_dtype=torch.float16)
    assert torch.equal(f16, f32.half()) and torch.equal(m16, m32)
    p32 = ops.pos2embed(ref, 128, out_dtype=torch.float32)
    p16 = ops.pos2embed(ref, 128, out_dtype=torch.float16)
    assert torch.equal(p16, p32.half())
    emb = torch.randn(B, V, Nq, 64, device=DEV).half()
    base = torch.randn(Nq, 64, device=DEV)
    assert torch.equal(ops.masked_view_sum(emb, m16, base=base), ops.masked_view_sum(emb.float(), m16, base=base))


def test_ray_query_pe_fp16_points_on_the_camera_plane():
    """Reference points on camera 0's plane (z = 0) project to |px| ~ 1e8: their lifted coordinates are far beyond fp16's
    range.  They are outside the view, so their features are written as zeros in every dtype; the rv-PE MLP and the view
    sum then stay finite in fp16, and the in-view points of camera 1 keep the oracle's features."""
    B, Nq = 1, 200
    rng = np.random.RandomState(9)
    plane = np.diag([800.0, 800.0, 1.0, 1.0])                     # s = (800 x, 800 y, z): z = 0 is the camera plane
    l2i = np.stack([plane, synth.camera_matrices(1, rng, 160.0, 96.0)[0]])[None]
    l32, i32 = torch.from_numpy(l2i).float(), torch.from_numpy(np.linalg.inv(l2i)).float()
    ref = torch.from_numpy(rng.uniform(0, 1, (B, Nq, 3)).astype(np.float32))
    ref[..., 2] = 0.625                                            # z = 0.625 * 8 - 5 = 0 exactly
    want, wmask = O.rv_query_feats(ref, l32, i32, 64, 96.0, 160.0, NUSC)
    assert not bool(wmask[0, 0].any()) and float(want[0, 0].abs().max()) > 65504.0   # the overflow this guards against
    feats = {dt: ops.ray_query_pe(ref.to(DEV), l32.to(DEV), i32.to(DEV), 64, 96.0, 160.0, NUSC, out_dtype=dt)
             for dt in (torch.float32, torch.bfloat16, torch.float16)}
    f32, m32 = feats[torch.float32]
    assert torch.equal(m32.cpu() > 0.5, wmask)
    for dt, (f, m) in feats.items():
        assert torch.equal(m, m32) and bool(torch.isfinite(f).all()), dt
        assert float(f[m == 0].abs().max()) == 0.0, dt
    sel = wmask.unsqueeze(-1).expand_as(want)
    assert int(wmask.sum()) > 0 and _rel(f32.cpu()[sel], want[sel]) < 1e-5
    f16 = feats[torch.float16][0]
    assert torch.equal(f16, f32.half())
    g = torch.Generator().manual_seed(2)
    w0 = (torch.randn(1024, 192, generator=g) / math.sqrt(192)).half().to(DEV)
    w1 = (torch.randn(256, 1024, generator=g) / 32).half().to(DEV)
    h = ops.linear(f16, w0, torch.zeros(1024, device=DEV), relu=True)
    emb = ops.linear(h, w1, torch.zeros(256, device=DEV), out_dtype=torch.float32)
    assert bool(torch.isfinite(ops.masked_view_sum(emb, m32)).all())


@pytest.mark.parametrize("fdt", [torch.float32, torch.float16])
def test_gather_tokens_fp16(fdt):
    B, C, V = 2, 256, 3
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, C, 9, 11, generator=g).to(fdt).to(DEV)
    xi = torch.randn(B * V, C, 5, 7, generator=g).to(fdt).to(DEV)
    bev_pos = torch.randn(99, C, generator=g).to(DEV)
    rv_pos = torch.randn(B * V, 5, 7, C, generator=g).to(DEV)
    n_kv = 99 + V * 35
    for rng in (None, (64, 99 + 17), (96, n_kv)):
        k32, v32 = ops.gather_tokens(x, xi, bev_pos, rv_pos, B, V, out_dtype=torch.float32, tok_range=rng)
        k16, v16 = ops.gather_tokens(x, xi, bev_pos, rv_pos, B, V, out_dtype=torch.float16, tok_range=rng)
        assert k16.dtype == torch.float16
        assert torch.equal(k16, k32.half()) and torch.equal(v16, v32.half())


def test_add_layernorm_fp16():
    M, C = 777, 256
    g = torch.Generator().manual_seed(2)
    x, r, add = (torch.randn(M, C, generator=g).to(DEV) for _ in range(3))
    gamma, beta = (torch.randn(C, generator=g).to(DEV) for _ in range(2))
    y, _, ylp, yadd = ops.add_layernorm(x, r, gamma, beta, 1e-5, add=add, lp_dtype=torch.float16, want_ylp=True, want_yadd=True)
    y32, _, ylp32, yadd32 = ops.add_layernorm(x, r, gamma, beta, 1e-5, add=add, lp_dtype=torch.float32, want_ylp=True,
                                              want_yadd=True)
    assert ylp.dtype == torch.float16 and torch.equal(y, y32)
    assert torch.equal(ylp, ylp32.half()) and torch.equal(yadd, yadd32.half())


def test_lse_merge_fp16():
    G, B, H, Nq = 3, 2, 8, 37
    g = torch.Generator().manual_seed(9)
    o = torch.randn(G, B, Nq, H * 32, generator=g).to(DEV)
    lse = (torch.randn(G, B, H, Nq, generator=g) * 3).to(DEV)
    lse[1, 0, 0, :5] = float("-inf")
    o32, l32 = ops.lse_merge(o, lse, o_dtype=torch.float32)
    o16, l16 = ops.lse_merge(o, lse, o_dtype=torch.float16)
    assert torch.equal(o16, o32.half()) and torch.equal(l16, l32)
    parts = torch.cat([torch.cat([o[i].reshape(-1), lse[i].reshape(-1)]) for i in range(G)])
    assert torch.equal(ops.lse_merge_packed(parts, G, B, Nq, H, o_dtype=torch.float16),
                       ops.lse_merge_packed(parts, G, B, Nq, H, o_dtype=torch.float32).half())


def _peer_run(G, B, Nq, H, o_dtype, scatter, seed):
    """G emulated ranks in ordinary memory of one GPU (parallel.PeerExchange's layout); returns every rank's context."""
    g = torch.Generator().manual_seed(seed)
    n_o, n_l = B * Nq * H * 32, B * H * Nq
    bufs = []
    for _ in range(G):
        buf = torch.zeros(n_o + n_l + n_o + 64, dtype=torch.float32, device=DEV)
        buf[:n_o] = torch.randn(n_o, generator=g).to(DEV)
        buf[n_o:n_o + n_l] = (torch.randn(n_l, generator=g) * 3).to(DEV)
        bufs.append(buf)
    bases = [b.data_ptr() for b in bufs]
    streams = [torch.cuda.Stream() for _ in range(G)]
    torch.cuda.synchronize()
    for r in range(G):
        with torch.cuda.stream(streams[r]):
            ops.lse_merge_peer(bases, [p + (n_o + n_l) * 4 for p in bases], [p + (2 * n_o + n_l) * 4 for p in bases],
                               bases[r] + (2 * n_o + n_l + 16) * 4, r, B, Nq, H, torch.device(DEV), o_dtype, scatter)
    torch.cuda.synchronize()
    esz = 2 if o_dtype != torch.float32 else 4
    return [b[n_o + n_l:2 * n_o + n_l].view(torch.uint8)[:n_o * esz].view(o_dtype).clone() for b in bufs]


def _check_peer(G, scatter):
    B, Nq, H = 2, 37, 8
    want = _peer_run(G, B, Nq, H, torch.float32, scatter, 11 + G)
    got = _peer_run(G, B, Nq, H, torch.float16, scatter, 11 + G)
    for r in range(G):
        assert torch.equal(got[r], want[r].half()), r


@pytest.mark.parametrize("scatter", [0, 1])
def test_lse_merge_peer_fp16_single_rank(scatter):
    _check_peer(1, scatter)


@pytest.mark.skipif(os.environ.get("CMT_TEST_PEER_EMULATION") != "1",
                    reason="opt-in: G kernels of one GPU wait for each other -- needs them co-resident; the real "
                           "multi-process check is tests/test_gpu_multi.py")
@pytest.mark.parametrize("G,scatter", [(2, 0), (3, 1)])
def test_lse_merge_peer_fp16_emulated_group(G, scatter):
    _check_peer(G, scatter)


# ------------------------------------------------------------------------------------------ shared_conv
@pytest.mark.parametrize("shape", [(2, 128, 64, 9, 11, torch.float32), (1, 64, 32, 5, 4, torch.float16),
                                   (1, 512, 256, 60, 60, torch.float16)])
def test_shared_conv_tokens_fp16(shape):
    import torch.nn.functional as F
    B, Cin, Cout, H, W, fdt = shape
    g = torch.Generator().manual_seed(H * W + Cin)
    x = torch.randn(B, Cin, H, W, generator=g).to(fdt)
    w = torch.randn(Cout, Cin, 3, 3, generator=g) * (2.0 / (9 * Cin)) ** 0.5
    bias = torch.randn(Cout, generator=g) * 0.1
    pos = torch.randn(H * W, Cout, generator=g)
    wt = w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).half()
    xr = x.half().double()
    wr = wt.double().view(Cout, 3, 3, Cin).permute(0, 3, 1, 2)
    want = F.relu(F.conv2d(xr, wr, bias.double(), padding=1)).flatten(2).transpose(1, 2)     # [B, H*W, Cout]
    d = lambda t: t.to(DEV)
    xp = ops.nchw_to_padded_nhwc(d(x), dtype=torch.float16)
    guard = ops.conv_guard_rows(W)
    inner = xp.cpu().float()[:, guard:guard + (H + 2) * (W + 2)].view(B, H + 2, W + 2, Cin)
    assert xp.dtype == torch.float16 and torch.equal(inner[:, 1:-1, 1:-1], x.half().float().permute(0, 2, 3, 1))
    xk = torch.full((B, H * W + 5, Cout), 7.0, dtype=torch.float16, device=DEV)
    xv = torch.full_like(xk, 7.0)
    ops.shared_conv_tokens(xp, d(wt), d(bias), d(pos), xk, xv, H, W)
    torch.cuda.synchronize()
    assert _rel(xv[:, :H * W].float(), want) < TOL16
    assert _rel(xk[:, :H * W].float(), want + pos.double()) < TOL16
    assert bool((xv[:, H * W:] == 7.0).all()) and bool((xk[:, H * W:] == 7.0).all())
    lo, hi = W + 3, H * W - 2 * W - 1
    xk2 = torch.zeros((B, hi - lo, Cout), dtype=torch.float16, device=DEV)
    xv2 = torch.zeros_like(xk2)
    ops.shared_conv_tokens(xp, d(wt), d(bias), d(pos), xk2, xv2, H, W, tok_range=(lo, hi))
    assert torch.equal(xv2, xv[:, lo:hi]) and torch.equal(xk2, xk[:, lo:hi])


# ------------------------------------------------------------------------------------------ heads
def _build(cfg, precision):
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    return head.to(DEV).eval().set_precision(precision)


def _feats(inputs):
    return {k: torch.from_numpy(v).to(DEV) for k, v in inputs.items() if isinstance(v, np.ndarray)}


def _forward(head, kind, f, metas):
    with torch.no_grad():
        if kind.endswith("Coop"):
            return head.forward_single(f.get("vehicle_pts_feats"), f.get("infrastructure_pts_feats"),
                                       f.get("vehicle_img_feats"), f.get("infrastructure_img_feats"), metas)
        return head.forward_single(f.get("pts_feats"), f.get("img_feats"), metas)


def _compare(rets, want, precision, cfg, errs):
    """rel-L2 of every output against the reference, and the tie-tolerant top-k of every frame's last layer."""
    errs[precision] = {n: O.rel_l2(rets[0][n].float().cpu(), want[n]) for n in NAMES}
    k = cfg["bbox_coder"]["max_num"]
    for i in range(rets[0]["cls_logits"].shape[1]):
        ours = rets[0]["cls_logits"][-1][i].float().cpu().sigmoid().flatten()
        ref = want["cls_logits"][-1][i].sigmoid().flatten()
        tau = 2 * float((ours - ref).abs().max()) + 1e-7
        assert tau < 3e-2, precision
        assert O.topk_tie_tolerant_equal(ours.topk(k).indices, ours, ref.topk(k).indices, ref, tau), precision


def _assert_fp16_gain(errs, what):
    print(f"{what}: " + "  ".join(f"{p} " + " ".join(f"{n}={v:.2e}" for n, v in e.items()) for p, e in errs.items()))
    for n in NAMES:
        assert errs["fp16"][n] < 1e-2, (what, n, errs)
        assert errs["fp16"][n] <= 0.5 * errs["bf16"][n], (what, n, errs)


@pytest.mark.parametrize("kind", synth.HEAD_KINDS)
def test_head_fp16_against_golden(kind, golden_dir):
    gold = np.load(os.path.join(golden_dir, f"{kind}_mini.npz"))
    cfg, inputs = synth.mini_case(kind)
    want = {n: torch.from_numpy(gold[f"task0.{n}"]) for n in NAMES}
    errs = {}
    for precision in ("bf16", "fp16"):
        head = _build(cfg, precision)
        rets = _forward(head, kind, _feats(inputs), inputs["img_metas"])
        _compare(rets, want, precision, cfg, errs)
    _assert_fp16_gain(errs, kind)


CONFIGS = {
    "c0_lidar128": ("CmtLidarHead", 1024, dict(B=2, bev_hw=128)),
    "c1_coop_lidar": ("CmtLidarHeadCoop", 1440, dict(B=1, bev_hw=180)),
    "c2_nusc": ("CmtHead", 1440, dict(B=2, bev_hw=180, n_views=6, img_hw=(40, 100))),
    "c3_coop_fusion": ("CmtHeadCoop", 1440, dict(B=1, bev_hw=180, img_hw=(40, 100), vehicle_views=1, infra_views=3)),
}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_baseline_config_fp16_against_oracle(name):
    """configs[0]-[3] at their full shapes against the CPU oracle, bf16 and fp16 on the same inputs; also reports how
    many attention items the fp16 static kernel took (fused_decoder.last_norms)."""
    kind, grid, kw = CONFIGS[name]
    cfg = synth.head_cfg(kind, num_query=900, num_layers=6, grid=grid)
    inputs = synth.make_inputs(kind, seed=11, **kw)
    errs, want = {}, None
    for precision in ("bf16", "fp16"):
        head = _build(cfg, precision)
        if want is None:
            sd = {k: v.detach().cpu() for k, v in head.state_dict().items()}
            torch.set_num_threads(max(torch.get_num_threads(), 8))
            want = O.head_forward(sd, cfg, inputs)[0][0]
        rets = _forward(head, kind, _feats(inputs), inputs["img_metas"])
        torch.cuda.synchronize()
        assert rets[0]["cls_logits"].shape[0] == 6 and rets[0]["cls_logits"].shape[2] == 900
        _compare(rets, want, precision, cfg, errs)
        if precision == "fp16" and fused_decoder.last_norms is not None:
            qn2, kn2 = fused_decoder.last_norms
            kn = torch.cat([c.permute(1, 0, 2) for c in kn2], 1)        # [L, frames, H]
            bound = (qn2 * kn).sqrt() * 1.0079 + 1e-3
            print(f"{name}: fp16 static-kernel items {float((bound <= 14.0).float().mean()):.3f}")
    _assert_fp16_gain(errs, name)


@pytest.mark.parametrize("kind", ["CmtHeadCoop", "CmtLidarHeadCoop"])
def test_coop_node_batching_fp16(kind):
    """Both nodes' frames in one decoder pass == two sequential passes in fp16.  Not bit for bit: the self-attention's
    stream-K ranges depend on the number of frames, so its partials are merged in another fp32 order."""
    cfg, inputs = synth.mini_case(kind)
    head = _build(cfg, "fp16")
    f, metas = _feats(inputs), inputs["img_metas"]
    head.batch_nodes = True
    one = _forward(head, kind, f, metas)
    head.batch_nodes = False
    two = _forward(head, kind, f, metas)
    for n in one[0]:
        assert _rel(one[0][n], two[0][n]) < 2e-3, n


@pytest.mark.parametrize("kind", ["CmtHead", "CmtLidarHeadCoop"])
def test_graph_replay_and_batched_decode_fp16(kind):
    """runtime.GraphedForward in fp16: the captured forward and box decode replay the eager ones bit for bit;
    get_bboxes_batched selects what the torch coder selects."""
    from cmtcoop_b200.runtime import GraphedForward
    cfg, inputs = synth.mini_case(kind)
    head = _build(cfg, "fp16")
    feats, metas = _feats(inputs), inputs["img_metas"]
    g = GraphedForward(head, metas, feats, decode_boxes=True)
    for f in (feats, {k: v * 0.5 + 0.1 for k, v in feats.items()}):
        want = _forward(head, kind, f, metas)
        want_boxes = head.get_bboxes_batched([[r] for r in want], metas)
        got, got_boxes = g(f)
        torch.cuda.synchronize()
        for n in want[0]:
            assert torch.equal(got[0][n], want[0][n]), n
        for n in want_boxes:
            assert torch.equal(got_boxes[n], want_boxes[n]), n
        preds = [[r] for r in want]
        want_idx = [d["topk_index"] for d in head.bbox_coder.decode(preds)]
        scores = torch.cat([p[0]["cls_logits"][-1] for p in preds], -1).sigmoid()
        for i in range(len(metas)):
            s = scores[i].flatten()
            assert torch.equal(s[want_boxes["topk_index"][i]], s[want_idx[i]])
