"""Kernel-level parity through the C ABI (ctypes -> libcmtcoop_b200.so) against the CPU oracle
(oracle/cmt_oracle.py) on the same seeded inputs.  Tolerances are written next to each check:
index / mask work is bit-exact, fp32 kernels are within a few ulps, bf16 kernels are compared
with an fp64 evaluation of the SAME bf16-rounded operands (so the tolerance covers accumulation
order and the bf16 rounding of the output only)."""
import math

import numpy as np
import pytest
import torch

from cmtcoop_b200 import ops, synth
from oracle import cmt_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NUSC = synth.NUSC_RANGE


def _rel(a, b):
    return O.rel_l2(a.detach().cpu(), b.detach().cpu())


def _mats(n, seed=0, pad_w=160.0, pad_h=96.0):
    rng = np.random.RandomState(seed)
    l2i = np.stack(synth.camera_matrices(n, rng, pad_w, pad_h))
    return l2i, np.linalg.inv(l2i).astype(np.float32)


# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(3, 6, 10, 96.0, 160.0), (6, 40, 100, 640.0, 1600.0)])
def test_ray_pe(shape):
    n_cam, H, W, pad_h, pad_w = shape
    _, i2l = _mats(n_cam, 1, pad_w, pad_h)
    want = O.ray_coords(i2l, H, W, 64, pad_h, pad_w, NUSC)
    got32 = ops.ray_pe(torch.from_numpy(i2l).to(DEV), H, W, 64, pad_h, pad_w, NUSC, out_dtype=torch.float32)
    assert got32.shape == want.shape
    # fp32: summation order of the 4-term dot product differs from the reference's einsum
    assert _rel(got32, want) < 2e-6
    assert (got32.cpu() - want).abs().max() < 1e-4 * max(1.0, float(want.abs().max()))
    got16 = ops.ray_pe(torch.from_numpy(i2l).to(DEV), H, W, 64, pad_h, pad_w, NUSC, out_dtype=torch.bfloat16)
    assert torch.equal(got16.cpu(), got32.cpu().to(torch.bfloat16))  # same math, one rounding


def test_ray_query_pe_and_view_sum():
    B, V, Nq = 2, 3, 77
    rng = np.random.RandomState(5)
    l2i = np.stack([np.stack(synth.camera_matrices(V, rng, 160.0, 96.0)) for _ in range(B)])
    i2l = np.linalg.inv(l2i)
    ref = torch.from_numpy(rng.uniform(0, 1, (B, Nq, 3)).astype(np.float32))
    l32, i32 = torch.from_numpy(l2i).float(), torch.from_numpy(i2l).float()
    want, wmask = O.rv_query_feats(ref, l32, i32, 64, 96.0, 160.0, NUSC)
    got, mask = ops.ray_query_pe(ref.to(DEV), l32.to(DEV), i32.to(DEV), 64, 96.0, 160.0, NUSC, out_dtype=torch.float32)
    # points within 1e-3 px of an image border / z=0 may legitimately flip; none do for this seed
    assert torch.equal(mask.cpu() > 0.5, wmask)
    assert 0 < int(wmask.sum()) < wmask.numel()
    sel = wmask.unsqueeze(-1).expand_as(want)
    assert _rel(got.cpu()[sel], want[sel]) < 1e-5
    emb = torch.randn(B, V, Nq, 64, device=DEV)
    s = ops.masked_view_sum(emb, mask)
    assert torch.allclose(s.cpu(), (emb.cpu() * wmask.unsqueeze(-1)).sum(1), atol=1e-6)
    sb = ops.masked_view_sum(emb.bfloat16(), mask)
    assert torch.allclose(sb.cpu(), (emb.bfloat16().float().cpu() * wmask.unsqueeze(-1)).sum(1), atol=1e-6)


def test_pos2embed_bit_exact_indexing():
    pos = O.coords_bev([192, 192, 40])  # 24 x 24 tokens
    want = O.pos2embed(pos, 256)
    got = ops.pos2embed(pos.to(DEV), 256, out_dtype=torch.float32).cpu()
    assert got.shape == want.shape == (576, 512)
    assert (got - want).abs().max() < 2e-6  # sinf/cosf of the GPU vs the CPU libm
    # token / feature indexing: the y block precedes the x block, sin on even, cos on odd features
    t = 5 * 24 + 7
    x, y = (7 + 0.5) / 24, (5 + 0.5) / 24
    assert abs(float(got[t, 0]) - math.sin(2 * math.pi * y)) < 1e-6
    assert abs(float(got[t, 256 + 1]) - math.cos(2 * math.pi * x)) < 1e-6
    r3 = torch.rand(4, 9, 3)
    assert (ops.pos2embed(r3.to(DEV), 256, out_dtype=torch.float32).cpu() - O.pos2embed(r3, 256)).abs().max() < 2e-6


@pytest.mark.parametrize("case", ["fusion", "lidar", "image"])
def test_gather_tokens(case):
    B, C, V = 2, 256, 3
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, C, 9, 11, generator=g) if case != "image" else None          # 99 tokens: ragged tile
    xi = torch.randn(B * V, C, 5, 7, generator=g) if case != "lidar" else None      # 35 tokens per camera
    bev_pos = torch.randn(99, C, generator=g) if x is not None else None
    rv_pos = torch.randn(B * V, 5, 7, C, generator=g) if xi is not None else None
    mem, pos = O.tokens(x, xi, bev_pos, rv_pos, B)
    d = lambda t: None if t is None else t.to(DEV)
    xk, xv = ops.gather_tokens(d(x), d(xi), d(bev_pos), d(rv_pos), B, V, out_dtype=torch.float32)
    assert torch.equal(xv.cpu(), mem.permute(1, 0, 2))                 # bit-exact token indexing / copy
    assert torch.equal(xk.cpu(), (mem + pos).permute(1, 0, 2))         # one fp32 add, same operands
    xk16, xv16 = ops.gather_tokens(d(x), d(xi), d(bev_pos), d(rv_pos), B, V, out_dtype=torch.bfloat16)
    assert torch.equal(xv16.cpu(), mem.permute(1, 0, 2).bfloat16())
    assert torch.equal(xk16.cpu(), (mem + pos).permute(1, 0, 2).bfloat16())


@pytest.mark.parametrize("fdt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("hw", [((9, 11), (5, 7)), ((10, 12), (6, 10))])   # odd / even token counts (scalar / paired loads)
def test_gather_tokens_16bit_features_and_token_range(fdt, hw):
    """Feature maps handed over in 16 bits (bf16 / fp16) and a token sub-range (KV-token split): bit-exact against the
    oracle's rearrange + cat on the same (already rounded) feature values."""
    (hb, wb), (hi_, wi) = hw
    B, C, V = 2, 256, 3
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, C, hb, wb, generator=g).to(fdt)
    xi = torch.randn(B * V, C, hi_, wi, generator=g).to(fdt)
    n_bev, n_img = hb * wb, hi_ * wi
    bev_pos = torch.randn(n_bev, C, generator=g)
    rv_pos = torch.randn(B * V, hi_, wi, C, generator=g)
    mem, pos = O.tokens(x.float(), xi.float(), bev_pos, rv_pos, B)
    d = lambda t: t.to(DEV)
    xk, xv = ops.gather_tokens(d(x), d(xi), d(bev_pos), d(rv_pos), B, V, out_dtype=torch.float32)
    assert torch.equal(xv.cpu(), mem.permute(1, 0, 2)) and torch.equal(xk.cpu(), (mem + pos).permute(1, 0, 2))
    n_kv = n_bev + V * n_img
    for lo, hi in ((0, 64), (64, n_bev + 17), (n_bev - 3, n_kv), (n_bev + n_img, n_bev + n_img)):
        xk16, xv16 = ops.gather_tokens(d(x), d(xi), d(bev_pos), d(rv_pos), B, V, out_dtype=torch.bfloat16, tok_range=(lo, hi))
        assert xk16.shape == (B, hi - lo, C)
        assert torch.equal(xv16.cpu(), mem.permute(1, 0, 2)[:, lo:hi].bfloat16())
        assert torch.equal(xk16.cpu(), (mem + pos).permute(1, 0, 2)[:, lo:hi].bfloat16())


@pytest.mark.parametrize("shape", [(2, 128, 64, 9, 11, torch.float32), (1, 64, 32, 5, 4, torch.bfloat16),
                                   (1, 512, 256, 180, 180, torch.bfloat16)])
def test_shared_conv_tokens(shape):
    """3x3 conv + folded BN + ReLU as a tcgen05 implicit GEMM writing token-major xv and xk = xv + pos
    (cmt_head.py:280-287,481): against conv2d on the same bf16-rounded operands (fp64 for the small cases), token
    indexing t = y*W + x, then the token sub-range form (KV-token split) and the image tokens appended by the gather."""
    import torch.nn.functional as F
    B, Cin, Cout, H, W, fdt = shape
    g = torch.Generator().manual_seed(H * W + Cin)
    x = torch.randn(B, Cin, H, W, generator=g).to(fdt)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) * (2.0 / (9 * Cin)) ** 0.5)
    bias = torch.randn(Cout, generator=g) * 0.1
    pos = torch.randn(H * W, Cout, generator=g)
    wt = w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).bfloat16()
    big = H * W > 1000
    ref_dt = torch.float32 if big else torch.float64
    xr = x.bfloat16().to(ref_dt)
    wr = wt.to(ref_dt).view(Cout, 3, 3, Cin).permute(0, 3, 1, 2)
    want = F.relu(F.conv2d(xr, wr, bias.to(ref_dt), padding=1)).flatten(2).transpose(1, 2)     # [B, H*W, Cout]
    d = lambda t: t.to(DEV)
    xp = ops.nchw_to_padded_nhwc(d(x))
    guard = ops.conv_guard_rows(W)
    # bit-exact layout of the padded operand: interior = bf16(x), everything else zero
    xpc = xp.cpu().float()
    inner = xpc[:, guard:guard + (H + 2) * (W + 2)].view(B, H + 2, W + 2, Cin)
    assert torch.equal(inner[:, 1:-1, 1:-1], x.bfloat16().float().permute(0, 2, 3, 1))
    assert int((xpc != 0).sum()) == int((inner[:, 1:-1, 1:-1] != 0).sum())     # borders and guard rows stay zero
    n_extra = 7
    xk = torch.full((B, H * W + n_extra, Cout), 7.0, dtype=torch.bfloat16, device=DEV)
    xv = torch.full((B, H * W + n_extra, Cout), 7.0, dtype=torch.bfloat16, device=DEV)
    ops.shared_conv_tokens(xp, d(wt), d(bias), d(pos), xk, xv, H, W)
    torch.cuda.synchronize()
    assert _rel(xv[:, :H * W].float(), want) < 4e-3
    assert _rel(xk[:, :H * W].float(), want + pos.to(ref_dt)) < 4e-3
    assert bool((xv[:, H * W:] == 7.0).all()) and bool((xk[:, H * W:] == 7.0).all())     # rows past the BEV tokens untouched
    # xk is one rounding of (fp32 value + pos): consistent with xv up to its own rounding
    assert ((xk[:, :H * W].float().cpu() - (xv[:, :H * W].float().cpu() + pos)).abs() <=
            0.01 * (xv[:, :H * W].float().cpu().abs() + pos.abs()) + 1e-6).all()
    # token sub-range: same values, row 0 = token lo
    lo, hi = (W + 3, H * W - 2 * W - 1)
    xk2 = torch.zeros((B, hi - lo, Cout), dtype=torch.bfloat16, device=DEV)
    xv2 = torch.zeros_like(xk2)
    ops.shared_conv_tokens(xp, d(wt), d(bias), d(pos), xk2, xv2, H, W, tok_range=(lo, hi))
    assert torch.equal(xv2, xv[:, lo:hi]) and torch.equal(xk2, xk[:, lo:hi])
    # the padded buffer is reusable: a second, different input through the same buffer
    x2 = (x.float() * 0.5 + 0.25).to(fdt)
    ops.nchw_to_padded_nhwc(d(x2), xp)
    ops.shared_conv_tokens(xp, d(wt), d(bias), d(pos), xk, xv, H, W)
    want2 = F.relu(F.conv2d(x2.bfloat16().to(ref_dt), wr, bias.to(ref_dt), padding=1)).flatten(2).transpose(1, 2)
    assert _rel(xv[:, :H * W].float(), want2) < 4e-3


def test_gemm_segmented_matches_shifted_products():
    """cmt_gemm_segmented: per-segment A column offset and row shift with zero fill outside the matrix, shared B per
    group of batches (the task-head first convolution over the query axis, cmt_head.py:116-150)."""
    g = torch.Generator().manual_seed(17)
    nb, M, N, seg_k, a_cols = 4, 300, 96, 64, 192
    guard = 2
    A = torch.zeros(nb, M + 2 * guard, a_cols)
    A[:, guard:guard + M] = torch.randn(nb, M, a_cols, generator=g)
    A = A.bfloat16()
    acol = [0, 64, 128, 0, 64]
    shift = [-1, 0, 1, 2, -2]
    Bm = (torch.randn(2, N, len(acol) * seg_k, generator=g) * 0.1).bfloat16()   # one weight set per 2 batches
    bias = torch.randn(N, generator=g)
    want = torch.zeros(nb, M, N, dtype=torch.float64)
    Af = A.double()
    for z in range(nb):
        for s, (c, sh) in enumerate(zip(acol, shift)):
            rows = Af[z, guard + sh:guard + sh + M, c:c + seg_k]
            want[z] += rows @ Bm[z // 2, :, s * seg_k:(s + 1) * seg_k].double().T
    want = want + bias.double()
    C = torch.empty(nb, M, N, dtype=torch.float32, device=DEV)
    ops.gemm_segmented(A.to(DEV), Bm.to(DEV), bias.to(DEV), C, M, N, seg_k, acol, shift, a_row_off=guard, a_rows=M + 2 * guard,
                       a_cols=a_cols, lda=a_cols, ldb=len(acol) * seg_k, ldc=N, batch=nb, strideA=(M + 2 * guard) * a_cols,
                       strideB=N * len(acol) * seg_k, b_batch_div=2, strideC=M * N)
    torch.cuda.synchronize()
    assert _rel(C, want) < 1e-5
    # rows shifted past either end of the matrix read zeros (no guard rows at all, shift beyond the matrix)
    A2 = torch.randn(1, M, a_cols, generator=g).bfloat16()
    C2 = torch.empty(1, M, N, dtype=torch.float32, device=DEV)
    ops.gemm_segmented(A2.to(DEV), Bm[:1].to(DEV), None, C2, M, N, seg_k, [0, 64], [-3, 5], a_row_off=0, a_rows=M,
                       a_cols=a_cols, lda=a_cols, ldb=len(acol) * seg_k, ldc=N)
    want2 = torch.zeros(M, N, dtype=torch.float64)
    A2f = torch.zeros(M + 16, a_cols, dtype=torch.float64)
    A2f[8:8 + M] = A2[0].double()
    want2 += A2f[8 - 3:8 - 3 + M, 0:64] @ Bm[0, :, 0:64].double().T
    want2 += A2f[8 + 5:8 + 5 + M, 64:128] @ Bm[0, :, 64:128].double().T
    torch.cuda.synchronize()
    assert _rel(C2[0], want2) < 1e-5


def test_coop_max_and_lse_merge():
    a = torch.randn(3, 2, 50, 256)
    b = torch.randn(3, 2, 50, 256)
    a[0, 0, 0, :4] = torch.tensor([float("nan"), float("inf"), -float("inf"), 1.0])
    want = torch.max(torch.stack([torch.nan_to_num(a), torch.nan_to_num(b)]), 0).values
    assert torch.equal(ops.coop_max(a.to(DEV), b.to(DEV)).cpu(), want)
    G, B, H, Nq = 3, 2, 8, 37
    o = torch.randn(G, B, Nq, H * 32)
    lse = torch.randn(G, B, H, Nq) * 3
    w = torch.softmax(lse, 0)                                            # exp(lse_g - LSE)
    want_o = (o.view(G, B, Nq, H, 32) * w.permute(0, 1, 3, 2).unsqueeze(-1)).sum(0).reshape(B, Nq, H * 32)
    got_o, got_l = ops.lse_merge(o.to(DEV), lse.to(DEV), o_dtype=torch.float32)
    assert _rel(got_o, want_o) < 1e-6
    assert torch.allclose(got_l.cpu(), torch.logsumexp(lse, 0), atol=1e-5)


def _peer_group_on_one_gpu(G, B, Nq, H, seed):
    """G emulated ranks in ordinary device memory of ONE GPU: per rank a packed (O | LSE) record, a context buffer and 64
    control words -- what parallel.PeerExchange lays out in symmetric memory."""
    g = torch.Generator().manual_seed(seed)
    n_o, n_l = B * Nq * H * 32, B * H * Nq
    o = torch.randn(G, B, Nq, H * 32, generator=g)
    lse = torch.randn(G, B, H, Nq, generator=g) * 3
    lse[0, 0, 0, :3] = float("-inf")                                   # a rank with no keys for these rows
    bufs = []
    for r in range(G):
        buf = torch.zeros(n_o + n_l + n_o + 64, dtype=torch.float32, device=DEV)
        buf[:n_o] = o[r].reshape(-1).to(DEV)
        buf[n_o:n_o + n_l] = lse[r].reshape(-1).to(DEV)
        bufs.append(buf)
    w = torch.nan_to_num(torch.softmax(lse, 0), nan=0.0)               # G = 1: no rank has keys for those rows -> zeros
    want = (o.view(G, B, Nq, H, 32) * w.permute(0, 1, 3, 2).unsqueeze(-1)).sum(0).reshape(B, Nq, H * 32)
    return bufs, n_o, n_l, want


@pytest.mark.parametrize("scatter", [0, 1])
def test_lse_merge_peer_single_rank(scatter):
    """The peer-memory exchange + merge kernel with a group of one (plain device memory): both handshakes with itself,
    the merge of one record is the identity, the exchange number advances across launches."""
    B, Nq, H = 2, 37, 8
    bufs, n_o, n_l, want = _peer_group_on_one_gpu(1, B, Nq, H, 3)
    base = bufs[0].data_ptr()
    for it in range(3):
        ops.lse_merge_peer([base], [base + (n_o + n_l) * 4], [base + (2 * n_o + n_l) * 4], base + (2 * n_o + n_l + 16) * 4,
                           0, B, Nq, H, torch.device(DEV), torch.float32, scatter)
        torch.cuda.synchronize()
        ctrl = bufs[0][2 * n_o + n_l:].view(torch.int32)
        assert int(ctrl[16]) == it + 1 and int(ctrl[17]) == 0 and int(ctrl[0]) == it + 1
        assert int(ctrl[8]) == (it + 1 if scatter else 0)
    got = bufs[0][n_o + n_l:2 * n_o + n_l].view(B, Nq, H * 32)
    assert _rel(got, want) < 1e-6


@pytest.mark.skipif(__import__("os").environ.get("CMT_TEST_PEER_EMULATION") != "1",
                    reason="opt-in: G kernels of one GPU wait for each other -- needs them co-resident (never under a "
                           "serialising profiler); the real multi-process check is tests/test_gpu_multi.py")
@pytest.mark.parametrize("G,scatter", [(2, 0), (3, 1), (8, 1)])
def test_lse_merge_peer_emulated_group(G, scatter):
    B, Nq, H = 2, 37, 8
    bufs, n_o, n_l, want = _peer_group_on_one_gpu(G, B, Nq, H, 5 + G)
    bases = [b.data_ptr() for b in bufs]
    streams = [torch.cuda.Stream() for _ in range(G)]
    torch.cuda.synchronize()
    for it in range(2):
        for r in range(G):
            with torch.cuda.stream(streams[r]):
                ops.lse_merge_peer(bases, [p + (n_o + n_l) * 4 for p in bases], [p + (2 * n_o + n_l) * 4 for p in bases],
                                   bases[r] + (2 * n_o + n_l + 16) * 4, r, B, Nq, H, torch.device(DEV), torch.bfloat16, scatter)
        torch.cuda.synchronize()
    for r in range(G):
        got = bufs[r][n_o + n_l:2 * n_o + n_l].view(torch.bfloat16)[:n_o].view(B, Nq, H * 32).float()
        assert _rel(got, want) < 4e-3, r                                  # bf16 output rounding
        assert torch.equal(got, bufs[0][n_o + n_l:2 * n_o + n_l].view(torch.bfloat16)[:n_o].view(B, Nq, H * 32).float())


# ------------------------------------------------------------------------------------------
GEMM_CASES = [
    # M, N, K, relu, bias, alpha
    (300, 256, 192, True, True, 1.0),      # rv-PE MLP layer 1 shape class (K=192: 3 k-blocks)
    (1000, 1024, 192, True, True, 1.0),
    (257, 256, 1024, False, True, 1.0),    # MLP layer 2 (K=1024), ragged M
    (900, 256, 256, False, True, 0.255),   # Q projection with the softmax pre-scale
    (129, 40, 64, False, False, 1.0),      # N not a multiple of 32 -> scalar tail path
]


@pytest.mark.parametrize("M,N,K,relu,bias,alpha", GEMM_CASES)
@pytest.mark.parametrize("mode", ["tcgen05", "simt_fp32"])
def test_gemm_plain(M, N, K, relu, bias, alpha, mode):
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / math.sqrt(K)
    b = torch.randn(N, generator=g) if bias else None
    dt = torch.bfloat16 if mode == "tcgen05" else torch.float32
    a_, w_ = a.to(dt), w.to(dt)
    want = (a_.double() @ w_.double().t() + (b.double() if bias else 0)) * alpha
    if relu:
        want = want.clamp_min(0)
    got = ops.linear(a_.to(DEV), w_.to(DEV), None if b is None else b.to(DEV), relu=relu, alpha=alpha,
                     out_dtype=torch.float32)
    # fp32 accumulation of K products: error ~ sqrt(K) * 2^-24 relative to the row norm
    assert _rel(got, want) < 5e-6
    if mode == "tcgen05":
        got16 = ops.linear(a_.to(DEV), w_.to(DEV), None if b is None else b.to(DEV), relu=relu, alpha=alpha)
        assert _rel(got16, want) < 4e-3  # one bf16 rounding of the output (2^-9 relative per element)


GEMM_LAYOUTS = [
    # M, N, K, batch, ldc, cb (None: N), cb_stride, strideC, bias ("col" / "row" / None), relu, alpha
    (200, 72, 128, 1, 72, None, 0, 0, "col", True, 0.5),             # N % 32 != 0 with a bias: ragged last chunk
    (200, 72, 128, 1, 80, None, 0, 0, "col", True, 0.5),             # ... 32-byte aligned rows: 256-bit chunks + ragged tail
    (150, 256, 64, 1, 260, None, 0, 0, "col", False, 1.0),           # row pitch not a multiple of 32 bytes
    (130, 96, 64, 3, 96, None, 0, 130 * 96 + 4, "row", False, 1.0),  # batch stride not a multiple of 32 bytes
    (140, 2304, 64, 1, 2304, None, 0, 0, "col", True, 1.0),          # column bias wider than the shared-memory cache
    (140, 2088, 64, 1, 2092, None, 0, 0, "col", False, 0.5),         # ... with ragged N and an unaligned row pitch
    (170, 128, 64, 2, 32, 32, 170 * 32 + 4, 4 * (170 * 32 + 4), "col", False, 1.0),  # column blocks, unaligned cb_stride
]


@pytest.mark.parametrize("M,N,K,batch,ldc,cb,cb_stride,strideC,bias,relu,alpha", GEMM_LAYOUTS)
@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float32])
def test_gemm_output_layouts(M, N, K, batch, ldc, cb, cb_stride, strideC, bias, relu, alpha, dt):
    """cmt_gemm_bias_act (tcgen05) into output layouts the 256-bit row stores cannot write: every element lands at
    z*strideC + (n // cb)*cb_stride + m*ldc + n % cb, and nothing else in the buffer is touched."""
    g = torch.Generator().manual_seed(M + N + K + batch)
    a = torch.randn(batch, M, K, generator=g).bfloat16()
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).bfloat16()
    b = torch.randn(M if bias == "row" else N, generator=g) if bias else None
    want = a.double() @ w.double().t()
    if bias == "row":
        want = want + b.double()[:, None]
    elif bias == "col":
        want = want + b.double()
    want = want * alpha
    if relu:
        want = want.clamp_min(0)
    cb = cb or N
    z, m, n = torch.meshgrid(torch.arange(batch), torch.arange(M), torch.arange(N), indexing="ij")
    idx = z * strideC + (n // cb) * cb_stride + m * ldc + n % cb
    size = int(idx.max()) + 1 + 8
    C = torch.full((size,), -7.0, dtype=dt, device=DEV)
    ops.gemm(a.to(DEV), w.to(DEV), None if b is None else b.to(DEV), C, M, N, K, lda=K, ldb=K, ldc=ldc, cb=cb,
             cb_stride=cb_stride, batch=batch, strideA=M * K if batch > 1 else 0, strideC=strideC, alpha=alpha, relu=relu,
             bias_per_row=bias == "row")
    torch.cuda.synchronize()
    out = C.cpu().float()
    # fp32: K products accumulated in fp32; bf16: one rounding of the output (2^-9 relative per element)
    assert _rel(out[idx], want) < (4e-3 if dt == torch.bfloat16 else 5e-6)
    untouched = torch.ones(size, dtype=torch.bool)
    untouched[idx.flatten()] = False
    assert bool((out[untouched] == -7.0).all())


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float32])
def test_gemm_head_layouts(dt):
    """All-layer K projection into [B,L,H,N_kv,32] and V^T projection into [B,L,H,32,ld]."""
    B, N_kv, C, L, H = 2, 333, 256, 2, 8
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, N_kv, C, generator=g).to(dt)
    w = (torch.randn(L * H * 32, C, generator=g) / 16).to(dt)
    b = torch.randn(L * H * 32, generator=g)
    want = (x.double() @ w.double().t() + b.double())                     # [B,N_kv,L*H*32]
    want_k = want.view(B, N_kv, L, H, 32).permute(0, 2, 3, 1, 4)
    k = ops.project_keys(x.to(DEV), w.to(DEV), b.to(DEV), L, H)
    tol = 4e-3 if dt == torch.bfloat16 else 5e-6
    assert k.shape == (B, L, H, N_kv, 32) and _rel(k.float(), want_k) < tol
    vt = ops.project_values_t(x.to(DEV), w.to(DEV), b.to(DEV), L, H)
    ld = vt.shape[-1]
    assert ld == 336 and ld % 8 == 0
    want_v = want.view(B, N_kv, L, H, 32).permute(0, 2, 3, 4, 1)
    assert _rel(vt[..., :N_kv].float(), want_v) < tol


# ------------------------------------------------------------------------------------------
def _attn_ref(q, k, vt, n_kv, lo, hi):
    """fp64 softmax(q k^T) v over tokens [lo,hi); q already carries log2(e)/sqrt(d) -> base-2 softmax."""
    B, Nq, HD = q.shape
    H = HD // 32
    qh = q.double().view(B, Nq, H, 32).permute(0, 2, 1, 3)
    s = qh @ k.double()[:, 0, :, lo:hi].transpose(-1, -2) * math.log(2.0)
    p = torch.softmax(s, -1)
    o = p @ vt.double()[:, 0, :, :, lo:hi].transpose(-1, -2)
    return o.permute(0, 2, 1, 3).reshape(B, Nq, HD), torch.logsumexp(s, -1)


ATTN_CASES = [
    # B, Nq, N_kv, lo, hi
    (1, 96, 300, 0, None),        # single ragged tile pair, one query block
    (2, 130, 1000, 0, None),      # two query tiles, second mostly padding
    (1, 900, 5000, 0, None),      # reference query count, 4 query blocks, many CTAs per item
    (3, 257, 2049, 0, None),      # three query tiles -> two blocks, ragged everything
    (2, 200, 4096, 1024, 3000),   # KV sub-range (multi-GPU token split)
    (1, 4, 64, 0, None),          # one tail tile, one step: fewer steps than warpgroup slots
    (1, 1, 130, 0, None),         # a single query
    (2, 388, 1500, 0, None),      # three full tiles + a 4-query tail tile (the 900 = 7*128+4 pattern)
]


@pytest.mark.parametrize("B,Nq,N_kv,lo,hi", ATTN_CASES)
@pytest.mark.parametrize("mode", ["simt_fp32", "tcgen05"])
def test_cross_attention(B, Nq, N_kv, lo, hi, mode):
    H = 8
    hi = N_kv if hi is None else hi
    g = torch.Generator().manual_seed(Nq + N_kv)
    dt = torch.float32 if mode == "simt_fp32" else torch.bfloat16
    q = (torch.randn(B, Nq, H * 32, generator=g) * (ops.LOG2E / math.sqrt(32)) * 2.0).to(dt)
    k = torch.randn(B, 1, H, N_kv, 32, generator=g).to(dt)
    ld = (N_kv + 7) // 8 * 8
    vt = torch.zeros(B, 1, H, 32, ld)
    vt[..., :N_kv] = torch.randn(B, 1, H, 32, N_kv, generator=g)
    vt = vt.to(dt)
    want_o, want_lse = _attn_ref(q, k, vt, N_kv, lo, hi)
    o, lse = ops.cross_attn(q.to(DEV), k.to(DEV), vt.to(DEV), 0, kv_begin=lo, kv_end=hi, o_dtype=torch.float32,
                            return_lse=True)
    # bf16 output: the same arithmetic rounded once at the end (the merge kernel's packed bf16 stores)
    o16 = ops.cross_attn(q.to(DEV), k.to(DEV), vt.to(DEV), 0, kv_begin=lo, kv_end=hi, o_dtype=torch.bfloat16)
    torch.cuda.synchronize()
    assert torch.equal(o16, o.bfloat16())
    if mode == "simt_fp32":
        assert _rel(o, want_o) < 2e-5 and (lse.cpu() - want_lse).abs().max() < 1e-4
    else:
        # P is rounded to bf16 before the PV product and exp2 is the MUFU approximation:
        # 2^-8 per element, averaged over many tokens
        assert _rel(o, want_o) < 4e-3, _rel(o, want_o)
        # the row sum l is accumulated in fp32 from the unrounded exponentials, so LSE carries only the exponential's
        # error (<= 7.5e-5 relative on the cubic lanes) and fp32 summation: ~1e-4 (tests/test_gpu_attention_edges.py)
        assert (lse.cpu() - want_lse).abs().max() < 1e-3


def test_cross_attention_matches_simt_on_same_bf16_inputs():
    """tcgen05 kernel vs the CUDA-core kernel fed the same bf16 operands (peaky scores: lazy rescale path)."""
    B, H, Nq, N_kv = 1, 8, 300, 3000
    g = torch.Generator().manual_seed(99)
    q = (torch.randn(B, Nq, H * 32, generator=g) * 1.5).bfloat16().to(DEV)
    k = (torch.randn(B, 1, H, N_kv, 32, generator=g) * 2).bfloat16().to(DEV)   # score std ~ 17 (log2 units)
    vt = torch.randn(B, 1, H, 32, N_kv, generator=g).bfloat16().to(DEV)
    a = ops.cross_attn(q, k, vt, 0, o_dtype=torch.float32)
    b = ops.cross_attn(q, k, vt, 0, o_dtype=torch.float32, simt=True)
    assert _rel(a, b) < 6e-3


@pytest.mark.parametrize("mode", ["simt_fp32", "tcgen05"])
def test_cross_attention_key_padding_mask(mode):
    """key_padding_mask branch (attention.py:76-90): padded keys carry no weight.  Frame 0: random padding; frame 1:
    the first 200 keys (three whole 64-key tiles) padded, so stream-K segments start on fully padded tiles; frame 2:
    valid prefix only (the usual var-len case)."""
    B, H, Nq, N_kv = 3, 8, 200, 1500
    g = torch.Generator().manual_seed(17)
    dt = torch.float32 if mode == "simt_fp32" else torch.bfloat16
    q = (torch.randn(B, Nq, H * 32, generator=g) * (ops.LOG2E / math.sqrt(32)) * 2.0).to(dt)
    k = torch.randn(B, 1, H, N_kv, 32, generator=g).to(dt)
    ld = (N_kv + 7) // 8 * 8
    vt = torch.zeros(B, 1, H, 32, ld)
    vt[..., :N_kv] = torch.randn(B, 1, H, 32, N_kv, generator=g)
    vt = vt.to(dt)
    keep = torch.rand(B, N_kv, generator=g) > 0.3
    keep[1, :200] = False
    keep[2] = torch.arange(N_kv) < 777
    qh = q.double().view(B, Nq, H, 32).permute(0, 2, 1, 3)
    s = qh @ k.double()[:, 0].transpose(-1, -2) * math.log(2.0)
    s = s.masked_fill(~keep[:, None, None, :], float("-inf"))
    want = (torch.softmax(s, -1) @ vt.double()[:, 0, :, :, :N_kv].transpose(-1, -2)).permute(0, 2, 1, 3).reshape(B, Nq, H * 32)
    want_lse = torch.logsumexp(s, -1)
    o, lse = ops.cross_attn(q.to(DEV), k.to(DEV), vt.to(DEV), 0, o_dtype=torch.float32, return_lse=True,
                            key_keep=keep.to(DEV))
    torch.cuda.synchronize()
    tol = 2e-5 if mode == "simt_fp32" else 4e-3
    assert _rel(o, want) < tol, _rel(o, want)
    ltol = 1e-4 if mode == "simt_fp32" else 1e-3
    assert (lse.cpu() - want_lse).abs().max() < ltol
    # a token range together with the mask (frame 1's padded prefix straddles lo), then also with the operand norms
    # (static-shift kernel: the score bound of these operands is below 60; the fp32 kernel ignores them)
    lo, hi = 128, 1472
    sr = s[..., lo:hi]
    want_r = (torch.softmax(sr, -1) @ vt.double()[:, 0, :, :, lo:hi].transpose(-1, -2)).permute(0, 2, 1, 3).reshape(B, Nq, H * 32)
    qn2 = q.float().view(B, Nq, H, 32).pow(2).sum(-1).amax(1).contiguous()
    kn2 = k.float().pow(2).sum(-1).amax(-1).contiguous()
    assert float((qn2 * kn2[:, 0]).sqrt().max()) * 1.0079 + 1e-3 < 60
    for norms in ({}, dict(q_norm2=qn2.to(DEV), k_norm2=kn2.to(DEV))):
        o_r, lse_r = ops.cross_attn(q.to(DEV), k.to(DEV), vt.to(DEV), 0, kv_begin=lo, kv_end=hi, o_dtype=torch.float32,
                                    return_lse=True, key_keep=keep.to(DEV), **norms)
        torch.cuda.synchronize()
        assert _rel(o_r, want_r) < tol, (bool(norms), _rel(o_r, want_r))
        assert (lse_r.cpu() - torch.logsumexp(sr, -1)).abs().max() < ltol, bool(norms)
    # and it is exactly the attention over the gathered keys (what unpad_input + cu_seqlens_k computes)
    idx = keep[2].nonzero().flatten()
    o2 = ops.cross_attn(q[2:3].to(DEV), k[2:3, :, :, idx].contiguous().to(DEV),
                        torch.nn.functional.pad(vt[2:3, ..., idx], (0, (-len(idx)) % 8)).contiguous().to(DEV), 0,
                        o_dtype=torch.float32)
    assert _rel(o[2:3], o2.cpu()) < tol


def test_gemm_norm2_max():
    """norm2_max of cmt_gemm_bias_act: running max over rows of the squared norm of each 32-column block."""
    g = torch.Generator().manual_seed(8)
    B, M, N, K = 3, 333, 256, 256
    x = torch.randn(B, M, K, generator=g).bfloat16()
    w = (torch.randn(N, K, generator=g) / 16).bfloat16()
    b = torch.randn(N, generator=g)
    n2 = torch.zeros(B, N // 32, device=DEV)
    q = ops.project_queries(x.to(DEV), w.to(DEV), b.to(DEV), N // 32, 0.5, norm2_max=n2)
    want = ((x.float() @ w.float().T + b) * 0.5)
    assert _rel(q.float(), want) < 4e-3
    want_n2 = want.view(B, M, N // 32, 32).pow(2).sum(-1).amax(1)
    assert torch.allclose(n2.cpu(), want_n2, rtol=2e-3)
    # per-head K layout
    kn2 = torch.zeros(B, 1, N // 32, device=DEV)
    k = ops.project_keys(x.to(DEV), w.to(DEV), b.to(DEV), 1, N // 32, norm2_max=kn2)
    want_k = (x.float() @ w.float().T + b).view(B, M, N // 32, 32)
    assert torch.allclose(kn2.cpu()[:, 0], want_k.pow(2).sum(-1).amax(1), rtol=2e-3)
    assert _rel(k[:, 0].float().permute(0, 2, 1, 3), want_k) < 4e-3


@pytest.mark.parametrize("masked", [False, True])
def test_cross_attention_static_shift(masked):
    """Static softmax shift: with the operand-norm maxima the kernel uses the Cauchy-Schwarz score bound as a fixed
    shift where it is <= 60 and the online softmax elsewhere.  Frame 0: small scores (static path); frame 1: large
    scores (bound > 60: online path); frame 2: mid-size norms.  Same result as the reference either way, and as the
    call without norms."""
    B, H, Nq, N_kv = 3, 8, 300, 3000
    g = torch.Generator().manual_seed(23)
    q = torch.randn(B, Nq, H * 32, generator=g) * 0.6
    k = torch.randn(B, 1, H, N_kv, 32, generator=g)
    q[1] *= 4.0
    k[1] *= 3.0          # score std ~ 7 * sqrt(32) / ... -> bound far above 60
    k[2] *= 2.0
    q, k = q.bfloat16(), k.bfloat16()
    vt = torch.randn(B, 1, H, 32, N_kv, generator=g).bfloat16()
    keep = None
    if masked:
        keep = torch.rand(B, N_kv, generator=g) > 0.25
        keep[0, :130] = False
    qn2 = q.float().view(B, Nq, H, 32).pow(2).sum(-1).amax(1).contiguous()
    kn2 = k.float().pow(2).sum(-1).amax(-1).contiguous()            # [B,1,H]
    bound = (qn2 * kn2[:, 0]).sqrt()
    assert bound[0].max() < 60 and bound[1].min() > 60             # both paths are exercised
    qh = q.double().view(B, Nq, H, 32).permute(0, 2, 1, 3)
    s = qh @ k.double()[:, 0].transpose(-1, -2) * math.log(2.0)
    if masked:
        s = s.masked_fill(~keep[:, None, None, :], float("-inf"))
    want = (torch.softmax(s, -1) @ vt.double()[:, 0].transpose(-1, -2)).permute(0, 2, 1, 3).reshape(B, Nq, H * 32)
    kw = dict(o_dtype=torch.float32, return_lse=True, key_keep=None if keep is None else keep.to(DEV))
    o, lse = ops.cross_attn(q.to(DEV), k.to(DEV), vt.to(DEV), 0, q_norm2=qn2.to(DEV), k_norm2=kn2.to(DEV), **kw)
    o0, lse0 = ops.cross_attn(q.to(DEV), k.to(DEV), vt.to(DEV), 0, **kw)
    torch.cuda.synchronize()
    assert _rel(o, want) < 6e-3, _rel(o, want)
    assert _rel(o, o0) < 6e-3
    assert (lse.cpu() - torch.logsumexp(s, -1)).abs().max() < 6e-3
    assert (lse - lse0).abs().max() < 6e-3


@pytest.mark.parametrize("ks", [1, 3])
def test_task_head_tail(ks):
    """cmt_task_head_tail against the eager GroupLayerNorm1d / ReLU / Conv1d(k) arithmetic (cmt_head.py:53-94, 116-150),
    k = 3 mixing neighbouring queries with zero padding at the ends of every frame, plus the reference-point decode
    (cmt_head.py:501-513) and the per-head contiguous output form."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(4)
    L, Bf, Nq, NH, HC, CMAX = 6, 2, 901, 6, 64, 10
    M = Bf * Nq
    h = torch.randn(L, M, NH, HC, generator=g) * 3 + 0.5
    gamma, beta = torch.randn(L, NH, HC, generator=g), torch.randn(L, NH, HC, generator=g)
    w2, b2 = torch.randn(L, NH, CMAX, ks, HC, generator=g) * 0.2, torch.randn(L, NH, CMAX, generator=g)
    eps = 1e-6
    hd = h.double()
    mu = hd.mean(-1, keepdim=True)
    var = (hd - mu).pow(2).mean(-1, keepdim=True)
    y = torch.relu((hd - mu) / (var + eps).sqrt() * gamma.double()[:, None] + beta.double()[:, None])   # [L,M,NH,HC]
    # Conv1d over the query axis of every frame: [L*NH groups] x [Bf] x [HC, Nq]
    yc = y.view(L, Bf, Nq, NH, HC).permute(1, 0, 3, 4, 2).reshape(Bf, L * NH * HC, Nq)
    wc = w2.double().permute(0, 1, 2, 4, 3).reshape(L * NH * CMAX, HC, ks)
    want = F.conv1d(yc, wc, b2.double().reshape(-1), padding=ks // 2, groups=L * NH)                   # [Bf, L*NH*CMAX, Nq]
    want = want.view(Bf, L, NH, CMAX, Nq).permute(1, 0, 4, 2, 3).reshape(L, M, NH, CMAX)
    d = lambda t: t.to(DEV)
    out = ops.task_head_tail(d(h), d(gamma), d(beta), d(w2), d(b2), eps, ksize=ks, Nq=Nq)
    assert out.shape == (L, M, NH, CMAX)
    assert torch.allclose(out.cpu().double(), want, atol=5e-5, rtol=1e-5)
    # decode of (head 0: outputs 0,1 -> ref x,y) and (head 1: output 0 -> ref z) + per-head contiguous outputs
    ref_logit = torch.randn(M, 3, generator=g)
    comp = torch.full((NH, CMAX), -1, dtype=torch.int32)
    scale, off = torch.ones(NH, CMAX), torch.zeros(NH, CMAX)
    comp[0, 0], comp[0, 1], comp[1, 0] = 0, 1, 2
    scale[0, 0], scale[0, 1], scale[1, 0] = 108.0, 108.0, 8.0
    off[0, 0], off[0, 1], off[1, 0] = -54.0, -54.0, -5.0
    couts = [2, 1, 3, 2, 2, 10]
    outs = ops.task_head_tail(d(h), d(gamma), d(beta), d(w2), d(b2), eps, ksize=ks, Nq=Nq, ref_logit=d(ref_logit), dec_comp=d(comp),
                              dec_scale=d(scale), dec_offset=d(off), head_couts=couts)
    assert [tuple(o.shape) for o in outs] == [(L, M, c) for c in couts] and all(o.is_contiguous() for o in outs)
    wantd = want.clone()
    wantd[:, :, 0, 0] = torch.sigmoid(want[:, :, 0, 0] + ref_logit[:, 0].double()) * 108.0 - 54.0
    wantd[:, :, 0, 1] = torch.sigmoid(want[:, :, 0, 1] + ref_logit[:, 1].double()) * 108.0 - 54.0
    wantd[:, :, 1, 0] = torch.sigmoid(want[:, :, 1, 0] + ref_logit[:, 2].double()) * 8.0 - 5.0
    for i, (o, c) in enumerate(zip(outs, couts)):
        assert torch.allclose(o.cpu().double(), wantd[:, :, i, :c], atol=1e-4, rtol=1e-5), i


def test_split3_and_fp32_grade_first_conv():
    """cmt_split3_bf16: the three bf16 terms sum back to the fp32 value (to 2^-24 relative), nan_to_num and the
    cooperative max are applied, guard rows are zero; and the six-product segmented GEMM built on it reproduces an fp32
    (fp64-checked) matrix product to ~1e-6 -- the task heads' first convolution (cmt_head.py:116-150)."""
    g = torch.Generator().manual_seed(8)
    L, Bf, Nq, C = 2, 2, 300, 256
    a = torch.randn(L, Bf, Nq, C, generator=g) * 2
    b = torch.randn(L, Bf, Nq, C, generator=g) * 2
    a[0, 0, 0, 0], a[0, 0, 0, 1], a[0, 0, 0, 2] = float("nan"), float("inf"), float("-inf")
    xs, merged = ops.split3(a.to(DEV), b.to(DEV), want_merged=True)
    want = torch.maximum(torch.nan_to_num(a), torch.nan_to_num(b))
    assert torch.equal(merged.cpu(), want)
    xs_c = xs.cpu().float().view(L * Bf, Nq + 2, 3, C)
    assert float(xs_c[:, 0].abs().max()) == 0.0 and float(xs_c[:, -1].abs().max()) == 0.0
    back = xs_c[:, 1:-1].double().sum(2).view(L, Bf, Nq, C)
    fin = want.abs() < 1e30
    assert ((back - want.double()).abs()[fin] <= want.double().abs()[fin] * 2.0 ** -23 + 1e-30).all()
    xs1 = ops.split3(a.to(DEV))
    inb = (torch.nan_to_num(a).abs() < 3e38).view(L * Bf, Nq, C)   # 3.4e38 is clamped to the largest bf16, not rounded to inf
    assert torch.equal(xs1.cpu().float().view(L * Bf, Nq + 2, 3, C)[:, 1:-1, 0][inb], torch.nan_to_num(a).bfloat16().float().view(L * Bf, Nq, C)[inb])
    # first conv, k = 1, through the plugin's own weight packing
    from cmtcoop_b200.plugin import SeparateTaskHead
    heads = dict(center=(2, 2), height=(1, 2), dim=(3, 2), rot=(2, 2), vel=(2, 2), cls_logits=(10, 2))
    for ks in (1, 3):
        th = SeparateTaskHead(256, heads, groups=L, head_conv=64, final_kernel=ks)
        torch.manual_seed(ks)
        th.init_weights()
        for n in heads:
            getattr(th, n)[1].weight.data.uniform_(0.5, 1.5)
            getattr(th, n)[1].bias.data.normal_(0, 0.1)
        sd = {"t." + k: v.detach().clone() for k, v in th.state_dict().items()}
        th = th.to(DEV).eval()
        x = torch.nan_to_num(a)
        x[0, 0, 0, 1:3] = 0.0   # +-3.4e38 entries overflow the fp32 GroupLayerNorm statistics of the reference itself (NaN row)
        with torch.no_grad():
            got = th(x.to(DEV))
        want_h = O.separate_task_head(x.double(), {k: v.double() for k, v in sd.items()}, "t", list(heads), ks)
        for n in heads:
            assert _rel(got[n], want_h[n]) < 3e-6, (ks, n, _rel(got[n], want_h[n]))


