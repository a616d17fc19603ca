"""The tcgen05 GEMM (csrc/gemm_tcgen05.cu) element by element, at the launch geometry the workload runs it under.

Every output element is held to an fp64 evaluation of the SAME rounded operands, with bias, alpha and ReLU in the
kernel's order (act((A B^T + bias) * alpha)):

    |got - want| <= C_ACC * ceil(K/16) * 2^-23 * S  +  u_out * |want|  +  tiny,    S = |alpha| * (|A| @ |B|^T + |bias|)

The first term is the fp32 accumulation (one K=16 MMA step at a time, each within a few fp32 ulps of the magnitudes
it adds), the second the rounding of the output (2^-8 bf16, 2^-11 fp16, 0 fp32), the third the subnormal spacing of
the output type.  A global relative L2 cannot see one wrong tile out of thousands; this bound sees one wrong element.
A failure names the first bad (batch, row, column), its tile (z, mt, nt) and the CTA that owned it under the host's
tile walk (launch_tc_gemm), together with the tile's place in that CTA's sequence.

  * host test (no GPU): the check accepts a simulated correct kernel and rejects five simulated kernel bugs;
  * synthetic cases: B-resident and streaming walks with 1..5 tiles per CTA, K edges, M / N edges, a broadcast A,
    in bf16 / fp16 operands with fp32 / 16-bit outputs and through the fp32 CUDA-core kernel;
  * replay: every GEMM launch of one eager forward of the benched workload (nusc, B = 8) and of coop_lidar.
"""
import math

import numpy as np
import pytest
import torch

from cmtcoop_b200 import ops, synth

DEV = "cuda:0"

# launch_tc_gemm's tile geometry (namespace gemm in gemm_tcgen05.cu)
BM, BN, BK = 128, 256, 64
RES_KB = 4                  # B-resident mode holds at most 4 K blocks of B (K <= 256)
BIAS_CAP = 2048             # the column bias is cached in shared memory for N <= BIAS_CAP - 64
B200_SMS = 148

# Accumulation constant of the bound, calibrated on a B200 (1000 W limit).  Every test prints the largest accumulation
# ratio (|got - want| - u_out |want| - tiny) / (ceil(K/16) 2^-23 S) it has seen.  Largest observed over this file:
#   tcgen05 bf16 -> fp32 1.32, bf16 -> bf16 0.25, fp16 -> fp32 1.45, fp16 -> fp16 0.17, fp32 CUDA-core 1.83
#   (all at K = 8, where the single MMA step shares its term with the bias add; K >= 64: <= 0.32),
#   workload replay: bf16 0.153, fp16 0.155, fp32 (CUDA-core) 0.317.
C_ACC = 3.0
U_OUT = {torch.float32: 0.0, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
TINY = {torch.float32: 2.0 ** -126, torch.bfloat16: 2.0 ** -126, torch.float16: 2.0 ** -24}
SENTINEL_BITS = {torch.float32: (torch.int32, 0x7FC0DEAD), torch.bfloat16: (torch.int16, 0x7FDE),
                 torch.float16: (torch.int16, 0x7E5A)}   # NaNs with a payload no kernel computes


# ------------------------------------------------------------------------------------------
# host replica of the launch geometry
class Walk:
    """The tile walk launch_tc_gemm sets up and TileWalk follows.  B-resident (K <= 256, B shared by the batch): CTA c
    keeps n-tile c % n_tiles and walks the (batch, m-tile) pairs c / n_tiles + i * gm; streaming: CTA c walks the tiles
    c + i * grid in (batch, m-tile, n-tile) order."""

    def __init__(self, M, N, K, batch, *, b_batched, sms, m_tiles=None, mt_off=0):
        self.m_tiles = -(-M // BM) if m_tiles is None else m_tiles
        self.mt_off = mt_off
        self.n_tiles = -(-N // BN)
        self.num_kb = -(-K // BK)
        self.batch = batch
        total = self.m_tiles * self.n_tiles * batch
        mz = self.m_tiles * batch
        self.resident = self.num_kb <= RES_KB and not b_batched and self.n_tiles <= sms
        if self.resident:
            self.gm = min(sms // self.n_tiles, mz)
            self.grid = self.gm * self.n_tiles
            self.tiles_per_cta = -(-mz // self.gm)
        else:
            self.grid = min(sms, total)
            self.tiles_per_cta = -(-total // self.grid)

    @property
    def mode(self):
        return "resident" if self.resident else "streaming"

    def owner(self, z, mt, nt):
        """(CTA, index of the tile in that CTA's sequence) of tile (z, mt, nt)."""
        mt -= self.mt_off
        if self.resident:
            cur = z * self.m_tiles + mt
            return (cur % self.gm) * self.n_tiles + nt, cur // self.gm
        t = (z * self.m_tiles + mt) * self.n_tiles + nt
        return t % self.grid, t // self.grid

    def tiles_of(self, cta):
        """The tiles CTA `cta` runs, in order: TileWalk of gemm_tcgen05.cu transliterated."""
        out = []
        if self.resident:
            cur, step, end, nt = cta // self.n_tiles, self.grid // self.n_tiles, self.m_tiles * self.batch, cta % self.n_tiles
            while cur < end:
                out.append((cur // self.m_tiles, cur % self.m_tiles + self.mt_off, nt))
                cur += step
        else:
            cur, step, end = cta, self.grid, self.m_tiles * self.n_tiles * self.batch
            tpb = self.m_tiles * self.n_tiles
            while cur < end:
                r = cur % tpb
                out.append((cur // tpb, r // self.n_tiles + self.mt_off, r % self.n_tiles))
                cur += step
        return out

    def describe(self):
        return f"{self.mode}, grid {self.grid}, {self.tiles_per_cta} tiles per CTA"


def store_form(*, c_ptr, esz, N, ldc, cb, cb_stride, strideC, batch, bias, bias_per_row, transpose=False):
    """The epilogue instantiation launch_tc_gemm picks for cmt_gemm_bias_act / cmt_gemm_segmented (enum Store)."""
    if transpose:
        return "Transposed"
    plain = cb >= N
    aligned = (c_ptr % 32 == 0 and (ldc * esz) % 32 == 0 and (plain or ((cb_stride * esz) % 32 == 0 and cb % 32 == 0))
               and (batch == 1 or (strideC * esz) % 32 == 0))
    bias_ok = bias is None or bias_per_row or N <= BIAS_CAP - 64
    return "Vec" if aligned and N % 32 == 0 and bias_ok else "Masked"


def conv_tiles(H, W, lo, hi):
    """(mt_off, m_tiles) of the shared_conv implicit GEMM computing tokens [lo, hi) (launch_tc_gemm)."""
    Wp = W + 2
    y_lo, y_hi = lo // W, (hi - 1) // W
    p_lo, p_hi = (y_lo + 1) * Wp + 1, (y_hi + 1) * Wp + W + 1
    return p_lo // BM, -(-p_hi // BM) - p_lo // BM


# ------------------------------------------------------------------------------------------
# the element-wise check
def reference(A, B, bias=None, *, alpha=1.0, relu=False, bias_per_row=False):
    """want = act((A B^T + bias) * alpha) and S = |alpha| (|A| |B|^T + |bias|), fp64, for A [R, K], B [N, K]."""
    A, B = A.double(), B.double()
    want = A @ B.T
    S = A.abs() @ B.abs().T
    if bias is not None:
        b = bias.double()
        b = b[:, None] if bias_per_row else b[None, :]
        want += b
        S += b.abs()
    if alpha != 1.0:
        want *= alpha
        S *= abs(alpha)
    if relu:
        want.clamp_min_(0.0)
    return want, S


class Stats:
    """Largest accumulation ratio seen: (|got - want| - u_out |want| - tiny) / (ceil(K/16) 2^-23 S)."""

    def __init__(self):
        self.ratio = 0.0

    def add(self, r):
        self.ratio = max(self.ratio, r)


def check_elements(got, want, S, K, out_dtype, *, what, z=0, rows=None, walk=None, stats=None):
    """Asserts the element bound for one frame z: got, want, S [R, N] (rows[r] = GEMM row of r, default r)."""
    c_acc = C_ACC
    got = got.double()
    acc_unit = math.ceil(K / 16) * 2.0 ** -23
    slack = want.abs() * U_OUT[out_dtype] + TINY[out_dtype]
    excess = (got - want).abs() - slack
    bound = S * (c_acc * acc_unit)
    bad = ~(excess <= bound)                       # NaN is bad
    if bool(bad.any()):
        n_bad = int(bad.sum())
        i = int(torch.argmax(bad.flatten().to(torch.uint8)))
        r, n = divmod(i, want.shape[1])
        m = int(rows[r]) if rows is not None else r
        mt, nt = m // BM, n // BN
        if walk is None:
            where = "CUDA-core kernel"
        else:
            cta, seq = walk.owner(z, mt, nt)
            where = f"tile (z={z}, mt={mt}, nt={nt}) of CTA {cta} (its tile {seq} of {walk.tiles_per_cta}, {walk.mode})"
        g, w, s = float(got[r, n]), float(want[r, n]), float(S[r, n])
        raise AssertionError(
            f"{what}: {n_bad} of {bad.numel()} elements of frame {z} outside the bound; first at (batch {z}, row {m}, "
            f"col {n}): got {g!r} want {w!r} |err| {abs(g - w):.3e} > bound "
            f"{c_acc * acc_unit * s + U_OUT[out_dtype] * abs(w) + TINY[out_dtype]:.3e} (S {s:.3e}); {where}")
    ratio = float((excess.clamp_min(0.0) / (S * acc_unit).clamp_min(1e-300)).max()) if S.numel() else 0.0
    if stats is not None:
        stats.add(ratio)
    return ratio


def check_norm2(n2, want, what):
    """norm2_max against the max over rows of the reference's squared 32-column norms: [.., N/32] each."""
    ok = (n2.double() - want).abs() <= 1e-4 * want + 1e-30
    assert bool(ok.all()), f"{what}: norm2_max off at {ok.logical_not().nonzero()[:4].tolist()}"


def _blocks(C, z_off, M, N, ldc, cb, cb_stride, transpose):
    """[M, N / cb, cb] view of the frame output at z_off: element (m, n) at
    z_off + (n // cb) cb_stride + (m ldc | (n % cb) ldc + m)."""
    if cb >= N:
        assert not transpose
        return C.as_strided((M, 1, N), (ldc, 0, 1), z_off)
    assert N % cb == 0
    st = (1, cb_stride, ldc) if transpose else (ldc, cb_stride, 1)
    return C.as_strided((M, N // cb, cb), st, z_off)


# ------------------------------------------------------------------------------------------
# 2. the check itself, on a simulated kernel (no GPU)
def _simulated_acc(A, B, perm):
    """fp32 accumulation of the rounded operands, K=16 slices in the order `perm` (what the tensor-core MMAs do, in a
    different summation order)."""
    acc = torch.zeros(A.shape[0], A.shape[1], B.shape[0], dtype=torch.float32)
    for k0 in range(0, A.shape[-1], 16):
        idx = perm[k0:k0 + 16]
        acc += A[..., idx].float() @ B[:, idx].float().T
    return acc


@pytest.mark.parametrize("in_dt,out_dt", [(torch.bfloat16, torch.float32), (torch.bfloat16, torch.bfloat16),
                                          (torch.float16, torch.float32), (torch.float16, torch.float16)])
def test_element_check_accepts_a_correct_kernel_and_rejects_mutants(in_dt, out_dt):
    """The bound passes an fp32 matmul of the rounded operands accumulated in shuffled K order and rounded to the output
    type, and rejects each of five kernel bugs built by editing that result -- and points at the tile that has it."""
    g = torch.Generator().manual_seed(5)
    batch, M, N, K, alpha = 2, 384, 768, 200, 0.75
    A = torch.randn(batch, M, K, generator=g).to(in_dt)
    B = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(in_dt)
    bias = torch.randn(N, generator=g)
    perm = torch.randperm(K, generator=g)
    walk = Walk(M, N, K, batch, b_batched=False, sms=8)
    assert walk.resident and walk.tiles_per_cta == 3
    acc = _simulated_acc(A, B, perm)

    def out(a, b=bias):
        return ((a + b) * alpha).to(out_dt)

    def check(got):
        for z in range(batch):
            want, S = reference(A[z], B, bias, alpha=alpha)
            check_elements(got[z], want, S, K, out_dt, what="simulated", z=z, walk=walk)

    check(out(acc))

    def tile(z, mt, nt):
        return (z, slice(mt * BM, (mt + 1) * BM), slice(nt * BN, (nt + 1) * BN))

    # one K=16 slice dropped in tile (1, 1, 1)
    bad = acc.clone()
    z, rs, cs = tile(1, 1, 1)
    idx = perm[32:48]
    bad[z, rs, cs] -= A[z, rs][:, idx].float() @ B[cs][:, idx].float().T
    with pytest.raises(AssertionError, match=r"tile \(z=1, mt=1, nt=1\) of CTA 1 "):
        check(out(bad))
    # a 32-column chunk of tile (0, 2, 1) copied from the neighbouring n-tile
    bad = acc.clone()
    bad[0, 2 * BM:3 * BM, BN + 64:BN + 96] = acc[0, 2 * BM:3 * BM, 2 * BN + 64:2 * BN + 96]
    with pytest.raises(AssertionError, match=r"row 256, col 320\b.*tile \(z=0, mt=2, nt=1\)"):
        check(out(bad))
    # the bias shifted by one column
    with pytest.raises(AssertionError, match=r"\(batch 0, row 0, col 0\)"):
        check(out(acc, torch.cat([bias[1:], bias[-1:]])))
    # one row read from m + 1, one from m - 1
    for src in (201, 199):
        bad = acc.clone()
        bad[1, 200] = acc[1, src]
        with pytest.raises(AssertionError, match=r"\(batch 1, row 200, col \d+\).*tile \(z=1, mt=1, nt=\d\)"):
            check(out(bad))
    # the accumulator of the last tile of CTA 4 still holds the CTA's previous tile
    seq = walk.tiles_of(4)
    assert len(seq) == 3
    (zp, mp, np_), (zc, mc, nc) = seq[-2], seq[-1]
    bad = acc.clone()
    bad[tile(zc, mc, nc)] += acc[tile(zp, mp, np_)]
    with pytest.raises(AssertionError, match=rf"tile \(z={zc}, mt={mc}, nt={nc}\) of CTA 4 \(its tile 2 of 3"):
        check(out(bad))


@pytest.mark.parametrize("M,N,K,batch,b_batched,sms", [(1000, 1536, 256, 3, False, 148), (300, 1792, 256, 2, False, 148),
                                                        (5000, 256, 1024, 2, False, 148), (900, 520, 192, 4, True, 148),
                                                        (129, 40, 72, 1, False, 148), (56400, 1536, 256, 8, False, 148)])
def test_walk_replica_covers_every_tile_once(M, N, K, batch, b_batched, sms):
    """owner() inverts the transliterated TileWalk: every tile belongs to exactly one CTA, at the stated place in its
    sequence, and no CTA runs more than tiles_per_cta tiles.  The benched K projection is the last shape."""
    w = Walk(M, N, K, batch, b_batched=b_batched, sms=sms)
    seen = {}
    for c in range(w.grid):
        for i, t in enumerate(w.tiles_of(c)):
            assert t not in seen
            seen[t] = (c, i)
    assert len(seen) == w.m_tiles * w.n_tiles * batch
    assert max(i for _, i in seen.values()) + 1 == w.tiles_per_cta
    for t, ci in seen.items():
        assert w.owner(*t) == ci
    if (M, N, K, batch) == (56400, 1536, 256, 8):
        assert w.resident and w.grid == 24 * 6 and w.tiles_per_cta == 147


# ------------------------------------------------------------------------------------------
# 3. synthetic geometry cases
VARIANTS = {
    # name: (operand dtype, output dtype, CUDA-core kernel)
    "bf16-f32": (torch.bfloat16, torch.float32, False),
    "bf16-bf16": (torch.bfloat16, torch.bfloat16, False),
    "f16-f32": (torch.float16, torch.float32, False),
    "f16-f16": (torch.float16, torch.float16, False),
    "f32-simt": (torch.float32, torch.float32, True),
}


def _case(name, **kw):
    c = dict(name=name, M=None, tiles=None, N=256, K=256, batch=1, lda=None, ldb=None, a_bcast=False, b_batched=False,
             bias="col", alpha=1.0, relu=False, layout="plain", ldc_pad=0, norm2=False, form=None)
    c.update(kw)
    return c


CASES = [
    # B-resident walk, K = 256: 1..5 tiles per CTA over 1, 6 and 7 n-tiles (6 and 7 do not divide 148)
    _case("res-t1-nt6-fewer-mtiles-than-ctas", tiles=1, N=1536, relu=True),
    _case("res-t2-nt7", tiles=2, N=1792, batch=2, alpha=0.37),
    _case("res-t3-nt1-norm2", tiles=3, N=256, relu=True, norm2=True),
    _case("res-t4-nt6-head-blocks-norm2", tiles=4, N=1536, batch=3, layout="blocks", norm2=True),
    _case("res-t5-nt7-row-bias", tiles=5, N=1760, batch=2, bias="row"),
    _case("res-t3-nt6-transposed", tiles=3, N=1536, batch=2, layout="vt"),
    # streaming walk: K > 256 ...
    _case("str-k320-t1-nt6", tiles=1, N=1536, K=320),
    _case("str-k320-t2-nt7-ragged-n", tiles=2, N=1700, K=320, batch=2, relu=True),
    _case("str-k1024-t3-nt1", tiles=3, N=256, K=1024, alpha=0.5),
    _case("str-k1024-t4-nt6", tiles=4, N=1536, K=1024, batch=2),
    _case("str-k320-t5-nt7", tiles=5, N=1792, K=320, relu=True),
    # ... and a batched B with K <= 256
    _case("str-bbatch-k192-t3-nt6", tiles=3, N=1536, K=192, batch=4, b_batched=True),
    _case("str-bbatch-k256-t5-nt1", tiles=5, N=256, K=256, batch=3, b_batched=True, relu=True),
    # K edges: TMA zero fill past K (NaN in the padding columns of lda / ldb > K)
    _case("k8", tiles=2, N=512, K=8),
    _case("k72-padded-lda", tiles=2, N=512, K=72, lda=136, ldb=80),
    _case("k136", tiles=2, N=512, K=136, relu=True),
    _case("k200", tiles=2, N=512, K=200, batch=2),
    _case("k256-last-resident", tiles=2, N=512, K=256),
    _case("k264-first-streaming", tiles=3, N=512, K=264, lda=328, batch=2),
    # M and N edges: 1984 is the widest N whose bias the shared-memory cache holds, 1992 takes the Masked form
    _case("m1-n1992", M=1, N=1992, K=128, form="Masked"),
    _case("m127-n1984", M=127, N=1984, K=64, form="Vec"),
    _case("m129-n8", M=129, N=8, K=136),
    _case("m129-n40", M=129, N=40, K=72, relu=True),
    _case("n1984-t3", tiles=3, N=1984, K=192, batch=2, form="Vec"),
    _case("n1992-t2", tiles=2, N=1992, K=192, batch=3, alpha=0.8, form="Masked"),
    _case("n1536-unaligned-ldc", tiles=2, N=1536, K=128, ldc_pad=4, form="Masked"),
    # one A broadcast to every batch (strideA == 0)
    _case("bcast-a-resident", tiles=3, N=768, K=128, batch=4, a_bcast=True),
    _case("bcast-a-bbatch", tiles=2, N=512, K=192, batch=5, a_bcast=True, b_batched=True, relu=True),
]


def _rows_for(tiles, n_tiles, batch, streaming, sms):
    """M (ragged last m-tile) that gives `tiles` tiles to the busiest CTA; 1 tile: fewer tiles than CTAs."""
    if streaming:
        total = sms // 2 if tiles == 1 else (tiles - 1) * sms + sms // 2 + 1
        mz = -(-total // n_tiles)
    else:
        per = sms // n_tiles
        mz = max(per // 2, 1) if tiles == 1 else (tiles - 1) * per + per // 2 + 1
    return -(-mz // batch) * BM - 37


def _shaped(case, sms):
    c = dict(case)
    streaming = c["b_batched"] or -(-c["K"] // BK) > RES_KB
    if c["M"] is None:
        c["M"] = _rows_for(c["tiles"], -(-c["N"] // BN), c["batch"], streaming, sms)
    c["lda"] = c["lda"] or c["K"]
    c["ldb"] = c["ldb"] or c["K"]
    return c


def _operand(nz, rows, cols, ld, stride, dt, g, scale):
    """nz frames of [rows, cols] at z*stride + r*ld + c of a flat buffer whose every other element is NaN."""
    size = (nz - 1) * stride + rows * ld
    flat = torch.full((size,), float("nan"), dtype=dt, device=DEV)
    vals = torch.randn(nz, rows, cols, generator=g, device=DEV) * scale
    flat.as_strided((nz, rows, cols), (stride, ld, 1)).copy_(vals)
    return flat


def _sentinel(size, dt):
    it, bits = SENTINEL_BITS[dt]
    C = torch.empty(size, dtype=dt, device=DEV)
    C.view(it).fill_(bits)
    return C


def _untouched(C, mask):
    it, bits = SENTINEL_BITS[C.dtype]
    return bool((C.view(it)[~mask] == bits).all())


PARAMS = [pytest.param(c, v, id=f"{c['name']}-{v}") for c in CASES for v in VARIANTS
          if not (c["layout"] == "vt" and (VARIANTS[v][2] or VARIANTS[v][1] == torch.float32))]
_stats = {}


@pytest.mark.gpu
@pytest.mark.parametrize("case,variant", PARAMS)
def test_gemm_geometry(case, variant):
    in_dt, out_dt, simt = VARIANTS[variant]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    c = _shaped(case, sms)
    M, N, K, batch, lda, ldb = c["M"], c["N"], c["K"], c["batch"], c["lda"], c["ldb"]
    g = torch.Generator(device=DEV).manual_seed(M * 7 + N * 3 + K + batch)
    nza = 1 if c["a_bcast"] or batch == 1 else batch
    nzb = batch if c["b_batched"] else 1
    strideA = 0 if nza == 1 else (M + 5) * lda           # NaN rows between the frames: zero fill past M
    strideB = 0 if nzb == 1 else (N + 3) * ldb
    A = _operand(nza, M, K, lda, strideA, in_dt, g, 1.0)
    B = _operand(nzb, N, K, ldb, strideB, in_dt, g, 1.0 / math.sqrt(K))
    bias = None
    if c["bias"]:
        bias = torch.randn(M if c["bias"] == "row" else N, generator=g, device=DEV)
    # output layout
    transpose = c["layout"] == "vt"
    if c["layout"] == "plain":
        ldc, cb, cb_stride = N + c["ldc_pad"], N, 0
        strideC = M * ldc
    elif c["layout"] == "blocks":                      # K projection: [B, N/32, M, 32]
        ldc, cb, cb_stride = 32, 32, M * 32
        strideC = N * M
    else:                                              # V^T: [B, N/32, 32, ld], ld = M rounded up to 8
        ldc = (M + 7) // 8 * 8
        cb, cb_stride = 32, 32 * ldc
        strideC = N * ldc
    size = (batch - 1) * strideC + (N // cb - 1) * cb_stride + (cb * ldc if transpose else M * ldc) + 8
    C = _sentinel(size, out_dt)
    n2 = torch.zeros(batch, N // 32, device=DEV) if c["norm2"] and not simt else None
    ops.gemm(A, B, bias, C, M, N, K, lda=lda, ldb=ldb, ldc=ldc, cb=cb, cb_stride=cb_stride, batch=batch, strideA=strideA,
             strideB=strideB, strideC=strideC, alpha=c["alpha"], relu=c["relu"], bias_per_row=c["bias"] == "row",
             force_simt=simt, transpose_out=transpose, norm2_max=n2)
    walk = None
    if not simt:
        walk = Walk(M, N, K, batch, b_batched=strideB != 0 and batch > 1, sms=sms)
        streaming = c["b_batched"] or -(-K // BK) > RES_KB
        assert walk.resident != streaming, walk.describe()
        if c["tiles"] is not None:
            assert walk.tiles_per_cta == c["tiles"], walk.describe()
        if c["form"] is not None:
            esz = 4 if out_dt == torch.float32 else 2
            assert store_form(c_ptr=C.data_ptr(), esz=esz, N=N, ldc=ldc, cb=cb, cb_stride=cb_stride, strideC=strideC,
                              batch=batch, bias=bias, bias_per_row=c["bias"] == "row") == c["form"]
    stats = _stats.setdefault(variant, Stats())
    mask = torch.zeros(size, dtype=torch.bool, device=DEV)
    for z in range(batch):
        a = A.as_strided((M, K), (lda, 1), z * strideA if nza > 1 else 0)
        b = B.as_strided((N, K), (ldb, 1), z * strideB if nzb > 1 else 0)
        want, S = reference(a, b, bias, alpha=c["alpha"], relu=c["relu"], bias_per_row=c["bias"] == "row")
        got = _blocks(C, z * strideC, M, N, ldc, cb, cb_stride, transpose).reshape(M, N)
        check_elements(got, want, S, K, out_dt, what=f"{c['name']} {variant}", z=z, walk=walk, stats=stats)
        _blocks(mask, z * strideC, M, N, ldc, cb, cb_stride, transpose).fill_(True)
        if n2 is not None:
            check_norm2(n2[z], want.view(M, N // 32, 32).pow(2).sum(-1).amax(0), c["name"])
    assert int(mask.sum()) == batch * M * N        # the layout addresses every element once
    assert _untouched(C, mask), f"{c['name']} {variant}: an element outside the output layout was written"
    print(f"{c['name']} {variant}: M={M} N={N} K={K} batch={batch} "
          f"{walk.describe() if walk else 'CUDA-core'}; max accumulation ratio {stats.ratio:.3f}")


# ------------------------------------------------------------------------------------------
# 4. replay of every GEMM launch of one eager forward
WORKLOADS = {"nusc": ("CmtHead", 6), "coop_lidar": ("CmtLidarHeadCoop", 0)}


class _Recorder:
    """Stands in for ops.gemm / ops.gemm_segmented / ops.shared_conv_tokens: calls the real function, then clones the
    operands and outputs on the same stream."""

    def __init__(self, monkeypatch):
        self.launches = []
        real = dict(gemm=ops.gemm, seg=ops.gemm_segmented, conv=ops.shared_conv_tokens)

        def gemm(A, Bm, bias, C, M, N, K, **kw):
            n2 = kw.get("norm2_max")
            n2_before = None if n2 is None else n2.clone()
            r = real["gemm"](A, Bm, bias, C, M, N, K, **kw)
            self._keep("gemm", dict(A=A, B=Bm, bias=bias, C=C, n2=n2), c_ptr=C.data_ptr(), M=M, N=N, K=K, n2_before=n2_before,
                       kw=kw)
            return r

        def seg(A, Bm, bias, C, M, N, seg_k, seg_acol, seg_shift, **kw):
            r = real["seg"](A, Bm, bias, C, M, N, seg_k, seg_acol, seg_shift, **kw)
            self._keep("seg", dict(A=A, B=Bm, bias=bias, C=C), c_ptr=C.data_ptr(), M=M, N=N, K=len(seg_acol) * seg_k, seg_k=seg_k,
                       acol=list(seg_acol), shift=list(seg_shift), kw=kw)
            return r

        def conv(xp, w, bias, bev_pos, xk, xv, H, W, tok_range=None):
            r = real["conv"](xp, w, bias, bev_pos, xk, xv, H, W, tok_range=tok_range)
            self._keep("conv", dict(A=xp, B=w, bias=bias, pos=bev_pos, xk=xk, xv=xv), H=H, W=W,
                       tok=(0, H * W) if tok_range is None else tuple(tok_range), K=w.shape[1], N=w.shape[0])
            return r

        monkeypatch.setattr(ops, "gemm", gemm)
        monkeypatch.setattr(ops, "gemm_segmented", seg)
        monkeypatch.setattr(ops, "shared_conv_tokens", conv)

    def _keep(self, op, tensors, **meta):
        self.launches.append(dict(op=op, t={k: None if v is None else v.clone() for k, v in tensors.items()}, **meta))


def _kind(L):
    if L["op"] == "conv":
        return "shared_conv"
    if L["op"] == "seg":
        return f"task_head_conv_{len(L['acol'])}seg"
    kw = L["kw"]
    if kw.get("transpose_out") or (kw.get("bias_per_row") and kw.get("strideA", 0) == 0 and kw.get("batch", 1) > 1):
        return "v_proj"
    if (kw.get("cb") or L["N"]) < L["N"]:
        return "k_proj"
    if (kw.get("tag") or "").startswith("rv_pe_mlp") or L["K"] == 192:
        return "rv_pe_mlp"
    if kw.get("alpha", 1.0) != 1.0:
        return "q_proj"
    return "linear"


def _frames(L, sms):
    """Normalises one recorded launch: (frames, out dtype, walk, form, per-frame callable giving
    (A_z [R, K], B_z [N, K], rows, [(got [R, N], added [R, N] or None)]), epilogue kwargs)."""
    t = L["t"]
    A, Bm, bias = t["A"].reshape(-1), t["B"].reshape(-1), t["bias"]
    if L["op"] == "gemm":
        kw = L["kw"]
        M, N, K = L["M"], L["N"], L["K"]
        C = t["C"].reshape(-1)
        batch, lda, ldb, ldc = kw.get("batch", 1), kw["lda"], kw["ldb"], kw["ldc"]
        sA, sB, sC = kw.get("strideA", 0), kw.get("strideB", 0), kw.get("strideC", 0)
        cb, cbs, tr = kw.get("cb") or max(N, 1), kw.get("cb_stride", 0), bool(kw.get("transpose_out"))
        simt = kw.get("force_simt") or t["A"].dtype == torch.float32
        walk = None if simt else Walk(M, N, K, batch, b_batched=sB != 0 and batch > 1, sms=sms)
        form = "SIMT" if simt else store_form(c_ptr=L["c_ptr"], esz=C.element_size(), N=N, ldc=ldc, cb=cb, cb_stride=cbs,
                                              strideC=sC, batch=batch, bias=bias, bias_per_row=kw.get("bias_per_row", False),
                                              transpose=tr)

        def frame(z):
            a = A.as_strided((M, K), (lda, 1), z * sA if batch > 1 else 0)
            b = Bm.as_strided((N, K), (ldb, 1), z * sB if batch > 1 else 0)
            return a, b, None, [(_blocks(C, z * sC, M, N, ldc, cb, cbs, tr).reshape(M, N), None)]
        epi = dict(alpha=kw.get("alpha", 1.0), relu=kw.get("relu", False), bias_per_row=kw.get("bias_per_row", False))
        return batch, C.dtype, walk, form, frame, epi, (M, N, K)
    if L["op"] == "seg":
        kw = L["kw"]
        M, N, K, seg_k = L["M"], L["N"], L["K"], L["seg_k"]
        C = t["C"].reshape(-1)
        batch, lda, ldb, ldc = kw.get("batch", 1), kw["lda"], kw["ldb"], kw["ldc"]
        sA, sB, sC, bdiv = kw.get("strideA", 0), kw.get("strideB", 0), kw.get("strideC", 0), max(kw.get("b_batch_div", 1), 1)
        a_rows, a_cols, a_off = kw["a_rows"], kw["a_cols"], kw["a_row_off"]
        walk = Walk(M, N, K, batch, b_batched=sB != 0 and batch > 1, sms=sms)
        form = store_form(c_ptr=L["c_ptr"], esz=C.element_size(), N=N, ldc=ldc, cb=N, cb_stride=0, strideC=sC, batch=batch,
                          bias=bias, bias_per_row=False)
        m = torch.arange(M, device=DEV)

        def frame(z):
            full = A.as_strided((a_rows, a_cols), (lda, 1), z * sA if batch > 1 else 0)
            a = torch.cat([_shifted(full, m + a_off + sh, col, seg_k) for col, sh in zip(L["acol"], L["shift"])], 1)
            b = Bm.as_strided((N, K), (ldb, 1), (z // bdiv) * sB if (sB != 0 and batch > 1) else 0)
            return a, b, None, [(C.as_strided((M, N), (ldc, 1), z * sC), None)]
        epi = dict(alpha=kw.get("alpha", 1.0), relu=kw.get("relu", False), bias_per_row=False)
        return batch, C.dtype, walk, form, frame, epi, (M, N, K)
    # shared_conv implicit GEMM: 9 taps over the zero-padded channel-last map, rows = padded positions of the tokens
    H, W, (lo, hi), N, K = L["H"], L["W"], L["tok"], L["N"], L["K"]
    xp, xk, xv, pos = t["A"], t["xk"], t["xv"], t["pos"].view(H * W, N)
    Bf, rows, Cin = xp.shape
    Wp = W + 2
    guard = ops.conv_guard_rows(W)
    mt_off, m_tiles = conv_tiles(H, W, lo, hi)
    walk = Walk(None, N, K, Bf, b_batched=False, sms=sms, m_tiles=m_tiles, mt_off=mt_off)
    tok = torch.arange(lo, hi, device=DEV)
    m = (tok // W + 1) * Wp + tok % W + 1
    shifts = [(ky - 1) * Wp + (kx - 1) for ky in range(3) for kx in range(3)]

    def frame(z):
        a = torch.cat([_shifted(xp[z], m + guard + sh, 0, Cin) for sh in shifts], 1)
        return a, Bm.view(N, K), m, [(xv[z, :hi - lo], None), (xk[z, :hi - lo], pos[lo:hi])]
    return Bf, xv.dtype, walk, "Conv", frame, dict(relu=True), ((H + 2) * Wp, N, K)


def _shifted(full, r, col, width):
    """full[r, col:col + width] with zeros where r falls outside the matrix (TMA zero fill)."""
    ok = (r >= 0) & (r < full.shape[0])
    v = full[r.clamp(0, full.shape[0] - 1), col:col + width]
    return torch.where(ok[:, None], v, torch.zeros((), dtype=v.dtype, device=v.device))


def _replay_check(L, sms, stats):
    frames, out_dt, walk, form, frame, epi, (M, N, K) = _frames(L, sms)
    kind = _kind(L)
    bias = L["t"]["bias"]
    for z in range(frames):
        a, b, rows, outs = frame(z)
        want, S = reference(a, b, bias, **epi)
        for got, added in outs:
            w, s = (want, S) if added is None else (want + added.double(), S + added.double().abs())
            check_elements(got, w, s, K, out_dt, what=f"{kind} M={M} N={N} K={K}", z=z, rows=rows, walk=walk, stats=stats)
        if L["op"] == "gemm" and L["t"].get("n2") is not None:
            nb = N // 32
            want_n2 = want.view(want.shape[0], nb, 32).pow(2).sum(-1).amax(0)
            before = L["n2_before"].reshape(frames, nb)[z].double()
            check_norm2(L["t"]["n2"].reshape(frames, nb)[z], torch.maximum(want_n2, before), f"{kind} norm2_max")
        del a, b, want, S
    return dict(kind=kind, M=M, N=N, K=K, batch=frames, form=form, mode=walk.mode if walk else "CUDA-core",
                tiles=walk.tiles_per_cta if walk else None, norm2=L["op"] == "gemm" and L["t"].get("n2") is not None)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("workload", ["nusc", "coop_lidar"])
def test_workload_gemm_launches(workload, precision, monkeypatch):
    """Every GEMM launch of one eager forward_single of the benched workload (B = 8, shared_conv included), checked
    element by element against fp64 on the launch's own operands."""
    from cmtcoop_b200.plugin import build_head
    kind, n_views = WORKLOADS[workload]
    cfg = synth.head_cfg(kind, num_query=900, num_layers=6, grid=8 * 180)
    inputs = synth.make_inputs(kind, B=8, bev_hw=180, n_views=max(n_views, 1), img_hw=(40, 100), in_channels=512, seed=0)
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision(precision)
    head.apply_shared_conv = True
    d = {k: (torch.from_numpy(v).to(DEV) if isinstance(v, np.ndarray) else v) for k, v in inputs.items()}
    rec = _Recorder(monkeypatch)
    with torch.no_grad():
        if kind.endswith("Coop"):
            head.forward_single(d["vehicle_pts_feats"], d["infrastructure_pts_feats"], d["vehicle_img_feats"],
                                d["infrastructure_img_feats"], d["img_metas"])
        else:
            head.forward_single(d["pts_feats"], d["img_feats"], d["img_metas"])
    monkeypatch.undo()
    del head, d
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    stats = _stats.setdefault(f"replay-{precision}", Stats())
    seen = []
    while rec.launches:
        L = rec.launches.pop(0)
        seen.append(_replay_check(L, sms, stats))
        del L
    print(f"\n{workload} {precision}: {len(seen)} GEMM launches, max accumulation ratio {stats.ratio:.3f}")
    for s in seen:
        print(f"  {s['kind']:<22} M={s['M']:<6} N={s['N']:<5} K={s['K']:<5} batch={s['batch']:<3} {s['form']:<10} "
              f"{s['mode']:<9} tiles/CTA={s['tiles']}{' norm2_max' if s['norm2'] else ''}")
    kinds = {s["kind"] for s in seen}
    tc = precision != "fp32"
    want_kinds = {"k_proj", "v_proj", "q_proj", "task_head_conv_6seg" if workload == "nusc" else "task_head_conv_18seg"}
    if tc:
        want_kinds.add("shared_conv")
    if workload == "nusc":
        want_kinds.add("rv_pe_mlp")
    assert want_kinds <= kinds, want_kinds - kinds
    assert any(s["K"] == 1024 and s["mode"] == ("streaming" if tc else "CUDA-core") for s in seen)   # second FFN layer
    if tc:
        kp = [s for s in seen if s["kind"] == "k_proj" and s["norm2"]]     # the all-layer projection of the memory
        assert kp and all(s["mode"] == "resident" and s["N"] == 1536 and s["tiles"] >= 3 for s in kp)
        assert all(s["form"] == "Transposed" for s in seen if s["kind"] == "v_proj")
        if workload == "nusc":
            # the benched launch: 6 n-tiles, grid 24 x 6 on 148 SMs, 147 tiles per CTA
            assert any(s["M"] == 56400 and s["batch"] == 8 and (s["tiles"] == 147 or sms != B200_SMS) for s in kp)
    conv_segs = [s for s in seen if s["kind"].startswith("task_head_conv")]
    assert conv_segs and all(s["batch"] > 1 for s in conv_segs)
