"""The tcgen05 cross-attention kernel (csrc/attn_tcgen05.cu) row by row at the edges where it can go wrong quietly:
the polynomial exponential lanes of every tile variant, stream-K segment boundaries and their merge, the lazy O rescale,
the static-shift decision per (frame, head), queries with no attended key, and the log-sum-exp merges.

Every output element is checked against an fp64 evaluation of the same bf16 operands, with a bound scaled by
A = sum_j p_j |v_j| of that element, so that one wrong row, lane or segment cannot hide in a global norm.

Tolerance of o (tau, per element, relative to A).  The kernel computes o = sum_j bf16(e_j) v_j / l with e_j = 2^(s_j - m)
and l = sum_j e_j in fp32 from the UNROUNDED e_j.  Against the exact p_j = e_j / sum e:
  - bf16(e_j) has relative error <= 2^-8 (8 significant bits, round to nearest);
  - e_j and l each carry the exponential's error: <= 7.5e-5 for the cubic lanes (ex2_poly), ~2^-22 for MUFU.EX2;
  - the scores of these tests are built from one or two exact bf16 x bf16 products plus small terms, so their fp32
    accumulation is one or two roundings: < 1e-4 relative to a weight even at |s| ~ 4000 (the ramps).
So |o - o_ref| <= (2^-8 + 1.5e-4 + 1e-4) A = 4.2e-3 A; tau = 2^-7 leaves a x1.9 margin.  A bf16 output adds one more
rounding of o (2^-8 |o_ref|).  The stream-K merge does not change this: every segment is normalised by its own l and
re-weighted by 2^(lse_s - max), which cancels the normalisation up to fp32 rounding.

Tolerance of LSE (natural log, per row): the exponentials (7.5e-5 relative on l) and the fp32 sums (64 products per
step, then one add per step: (64 + T) 2^-24 relative) give <= 1.1e-4 for T <= 200 steps (12 800 tokens); x2 margin and
rounding to a multiple of 1e-4: 3e-4, plus 2^-20 |lse| for the fp32 spacing of large scores and the ln 2 conversion.
"""
import math

import pytest
import torch

from cmtcoop_b200 import _lib, ops

DEV = "cuda:0"
H = 8
TAU = 2.0 ** -7
LSE_TOL = 3e-4

# attndb constants of csrc/attn_tcgen05.cu
QBLK, KT, NWG = 384, 64, 3
STATIC_LIMIT = 60.0


def _sms():
    """SM count the library plans with: the device's, or its fallback of 148 without a device."""
    if torch.cuda.is_available():
        return torch.cuda.get_device_properties(0).multi_processor_count
    return 148


# ------------------------------------------------------------------------------------------
# Python copy of attn_plan / range_start / cta_of (csrc/attn_tcgen05.cu)
class Plan:
    def __init__(self, B, Nq, n_tok, sms, static):
        self.qblocks = (Nq + QBLK - 1) // QBLK
        self.T = (n_tok + KT - 1) // KT
        self.BH = B * H
        rows_last = Nq - (self.qblocks - 1) * QBLK
        w_full = 10 if static else 4
        w_last = (7 if static else 3) if (rows_last + 127) // 128 < NWG else w_full
        S = self.BH * self.T
        nbf = self.qblocks - 1
        n_full, n_last = 0, sms
        if nbf > 0:
            n_full = (sms * w_full + (w_full * nbf + w_last) // 2) // (w_full * nbf + w_last)
            if n_full * nbf > sms - 1:
                n_full = (sms - 1) // nbf
            n_full = max(n_full, 1)
            n_last = max(sms - n_full * nbf, 1)
        self.n_full, self.n_last = min(n_full, S), min(n_last, S)
        self.S = S
        self.G = self.n_full * nbf + self.n_last
        len_min = S // self.n_last
        if nbf > 0 and S // self.n_full < len_min:
            len_min = S // self.n_full
        len_min = max(len_min, 1)
        self.S_max = (self.T - 1) // len_min + 2

    def range_start(self, c):
        full_ctas = (self.qblocks - 1) * self.n_full
        if c >= self.G:
            return self.qblocks * self.S
        if c < full_ctas:
            band, local = divmod(c, self.n_full)
            return band * self.S + (local * self.S) // self.n_full
        return (self.qblocks - 1) * self.S + ((c - full_ctas) * self.S) // self.n_last

    def cta_of(self, x):
        band, off = divmod(x, self.S)
        n = self.n_full if band < self.qblocks - 1 else self.n_last
        return band * self.n_full + ((off + 1) * n - 1) // self.S

    def segments(self, item):
        """[(j_begin, j_end)) tile-step ranges of `item` (= qb * BH + b * H + h), one per CTA range overlapping it."""
        x0, x1 = item * self.T, (item + 1) * self.T
        segs = []
        for c in range(self.cta_of(x0), self.cta_of(x1 - 1) + 1):
            lo, hi = max(self.range_start(c), x0), min(self.range_start(c + 1), x1)
            segs.append((lo - x0, hi - x0))
        return segs


def workspace_bytes(B, Nq, n_tok, sms):
    """tc_attn_workspace_bytes from the replica: partial slots of either plan, the packed mask, per-CTA flags."""
    on, st = Plan(B, Nq, n_tok, sms, False), Plan(B, Nq, n_tok, sms, True)
    slots = B * H * on.qblocks * max(on.S_max, st.S_max)
    return slots * QBLK * 33 * 4 + 256 + B * on.T * 8 + 8 + st.G * 4 + 16


def boundary_tiles(plan, item):
    """First and last tile-step of every segment of `item`."""
    tiles = set()
    for a, b in plan.segments(item):
        tiles.update((a, b - 1))
    return sorted(tiles)


# ------------------------------------------------------------------------------------------
def attn_ref(q, k, vt, keep=None, lo=0, hi=None):
    """fp64 attention of the same operands, one (frame, head) at a time.  q [B,Nq,H*32] in log2 units (pre-scaled by
    log2(e)/sqrt(32)), k [B,H,N,32], vt [B,H,32,ld], keep [B,N] bool or None; tokens [lo, hi).
    -> o [B,Nq,H*32], natural-log lse [B,H,Nq] (-inf and o = 0 where no key is attended), A [B,Nq,H*32]."""
    B, Nq, HD = q.shape
    hi = k.shape[2] if hi is None else hi
    o = torch.zeros(B, Nq, H, 32, dtype=torch.float64)
    A = torch.zeros_like(o)
    lse = torch.full((B, H, Nq), float("-inf"), dtype=torch.float64)
    for b in range(B):
        sel = torch.arange(lo, hi)
        if keep is not None:
            sel = sel[keep[b, lo:hi].bool()]
        if len(sel) == 0:
            continue
        for h in range(H):
            s = (q[b, :, h * 32:(h + 1) * 32].double() @ k[b, h, sel].double().T) * math.log(2.0)
            l = torch.logsumexp(s, -1)
            p = torch.exp(s - l[:, None])
            v = vt[b, h, :, sel].double().T
            o[b, :, h] = p @ v
            A[b, :, h] = p @ v.abs()
            lse[b, h] = l
    return o.reshape(B, Nq, HD), lse, A.reshape(B, Nq, HD)


def check(o, lse, ref, what=""):
    """Per element |o - o_ref| <= tau A (+ one bf16 rounding), per row |lse - lse_ref| <= LSE_TOL + 2^-20 |lse_ref|;
    rows without an attended key: o == 0 and lse == -inf exactly."""
    o_ref, lse_ref, A = ref
    tol = TAU * A + (2.0 ** -8 * o_ref.abs() if o.dtype == torch.bfloat16 else 0.0)
    o = o.detach().cpu().double()
    err = (o - o_ref).abs()
    bad = ~(err <= tol)
    assert not bad.any(), (f"{what}: {int(bad.sum())} elements out of bound, worst excess "
                           f"{float((err - tol)[bad].max()):.3e} at {bad.nonzero()[0].tolist()}")
    if lse is None:
        return
    lse = lse.detach().cpu().double()
    dead = torch.isinf(lse_ref)
    assert torch.equal(torch.isinf(lse) & (lse < 0), dead), f"{what}: -inf LSE rows differ"
    lerr = (lse - lse_ref).abs()[~dead]
    ltol = (LSE_TOL + 2.0 ** -20 * lse_ref.abs())[~dead]
    assert (lerr <= ltol).all(), f"{what}: LSE error {float((lerr - ltol).max()):.3e} over its bound"


def run(q, k, vt, *, keep=None, lo=0, hi=None, norms=None, o_dtype=torch.float32, simt=False):
    """cross_attn on the device; k [B,H,N,32] / vt [B,H,32,ld] get the layer axis here."""
    kw = dict(kv_begin=lo, kv_end=hi, o_dtype=o_dtype, return_lse=True, simt=simt,
              key_keep=None if keep is None else keep.to(DEV))
    if norms is not None:
        kw.update(q_norm2=norms[0].to(DEV), k_norm2=norms[1].to(DEV))
    o, lse = ops.cross_attn(q.to(DEV), k.unsqueeze(1).to(DEV), vt.unsqueeze(1).to(DEV), 0, **kw)
    torch.cuda.synchronize()
    return o, lse


def py_norms(q, k):
    """fp32 max |q|^2 [B,H] and max |k|^2 [B,1,H] of the bf16 operands."""
    B, Nq, _ = q.shape
    qn = q.float().view(B, Nq, H, 32).pow(2).sum(-1).amax(1).contiguous()
    kn = k.float().pow(2).sum(-1).amax(-1).unsqueeze(1).contiguous()
    return qn, kn


def _vt(B, N, g):
    ld = (N + 7) // 8 * 8
    vt = torch.zeros(B, H, 32, ld)
    vt[..., :N] = torch.randn(B, H, 32, N, generator=g)
    return vt.bfloat16()


# ------------------------------------------------------------------------------------------
# CPU checks of the helpers themselves (no GPU needed)
PLAN_SHAPES = [(1, 416, 1000), (1, 417, 1000), (2, 900, 1000), (1, 900, 8000), (8, 384, 640), (2, 300, 3000),
               (4, 417, 1500), (2, 300, 700), (8, 900, 56400)]


@pytest.mark.parametrize("B,Nq,N", PLAN_SHAPES)
def test_plan_replica_matches_library(B, Nq, N):
    """The replica's workspace size equals the library's, and its segments tile every item exactly."""
    sms = _sms()
    assert int(_lib.load().cmt_cross_attn_workspace_bytes(B, H, Nq, N)) == workspace_bytes(B, Nq, N, sms)
    for static in (False, True):
        p = Plan(B, Nq, N, sms, static)
        assert [p.cta_of(p.range_start(c)) for c in range(p.G)] == list(range(p.G))
        for item in range(p.qblocks * p.BH):
            segs = p.segments(item)
            assert segs[0][0] == 0 and segs[-1][1] == p.T and len(segs) <= p.S_max
            assert all(a < b for a, b in segs) and all(s[1] == t[0] for s, t in zip(segs, segs[1:]))


def test_plan_replica_shapes_reach_the_cases():
    """Shape (a) splits the items of its full query blocks into >= 6 segments (the last block's, with fewer CTAs per
    band, into 5); shape (b) has CTAs whose range covers parts of several items."""
    pa = Plan(1, 900, 8000, _sms(), False)
    full = (pa.qblocks - 1) * pa.BH
    assert min(len(pa.segments(i)) for i in range(full)) >= 6
    assert min(len(pa.segments(i)) for i in range(full, pa.qblocks * pa.BH)) >= 5
    pb = Plan(8, 384, 640, _sms(), False)
    multi = [c for c in range(pb.G) if pb.range_start(c) // pb.T != (pb.range_start(c + 1) - 1) // pb.T]
    assert len(multi) > pb.G // 4


def test_reference_on_cpu():
    """The fp64 reference: softmax weights, A, LSE, masks and the token range on a tiny case, against a direct sum."""
    g = torch.Generator().manual_seed(1)
    B, Nq, N = 2, 5, 70
    q = torch.randn(B, Nq, H * 32, generator=g).bfloat16()
    k = torch.randn(B, H, N, 32, generator=g).bfloat16()
    vt = _vt(B, N, g)
    keep = torch.rand(B, N, generator=g) > 0.5
    keep[1] = False
    o, lse, A = attn_ref(q, k, vt, keep, lo=3, hi=66)
    b, n, h = 0, 4, 6
    js = [j for j in range(3, 66) if keep[b, j]]
    s = torch.tensor([float(q[b, n, h * 32:(h + 1) * 32].double() @ k[b, h, j].double()) for j in js], dtype=torch.float64)
    w = torch.pow(2.0, s - s.max())
    w = w / w.sum()
    v = vt[b, h, :, js].double()
    assert torch.allclose(o[b, n, h * 32:(h + 1) * 32], v @ w, atol=1e-12)
    assert torch.allclose(A[b, n, h * 32:(h + 1) * 32], v.abs() @ w, atol=1e-12)
    assert abs(float(lse[b, h, n]) - float(torch.logsumexp(s * math.log(2.0), 0))) < 1e-12
    assert torch.equal(o[1], torch.zeros_like(o[1])) and bool(torch.isneginf(lse[1]).all())


# ------------------------------------------------------------------------------------------
def _dominant_case(B, Nq, N, masked, seed):
    """Every (frame, head) has 64 dominant keys, one per signed basis direction u (dimension u % 32, sign by u < 32);
    query row r points along direction (r + 32 h + 7 b) % 64 and scores 24 (log2 units) on its key, 0 or -24 on the
    other 63 and ~N(0, 0.3) on the noise keys.  Key u sits at tile position (u + 5 h + 11 b) % 64, so every (frame,
    head) puts a dominant key on each of the 64 lanes of a tile; its tile cycles through the first / last steps of the
    stream-K segments (online and static plans) and the ragged last tile."""
    g = torch.Generator().manual_seed(seed)
    a, c = 6.0, 4.0
    k = (torch.randn(B, H, N, 32, generator=g) * 0.05)
    q = torch.zeros(B, Nq, H, 32)
    T = (N + KT - 1) // KT
    valid_last = N - (T - 1) * KT
    keep = (torch.rand(B, N, generator=g) > 0.2) if masked else None
    plans = [Plan(B, Nq, N, _sms(), st) for st in (False, True)]
    where = []
    for b in range(B):
        for h in range(H):
            tiles = set()
            for pl in plans:
                for qb in range(pl.qblocks):
                    tiles.update(boundary_tiles(pl, qb * pl.BH + b * H + h))
            tiles = sorted(tiles) + [T - 1]
            for u in range(64):
                pos = (u + 5 * h + 11 * b) % 64
                j = tiles[(u + h) % len(tiles)]
                if j == T - 1 and pos >= valid_last:
                    j = T - 2 if T > 1 else j
                    pos = pos if j < T - 1 else pos % valid_last
                tok = j * KT + pos
                k[b, h, tok] = 0.0
                k[b, h, tok, u % 32] = c if u < 32 else -c
                where.append((b, h, u, j, pos))
                if masked:
                    keep[b, tok] = True
            for r in range(Nq):
                u = (r + 32 * h + 7 * b) % 64
                q[b, r, h, u % 32] = a if u < 32 else -a
    q = q.reshape(B, Nq, H * 32).bfloat16()
    k = k.bfloat16()
    return q, k, _vt(B, N, g), keep, where


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("Nq", [416, 417, 900])
def test_dominant_key_on_every_lane_and_boundary(Nq, masked):
    """416 queries leave 32 rows in the tail tile (the lone warp: LONE_MASK lanes), 417 leave 33 (two warps, the
    full-tile masks), 900 a 4-row lone warp next to a full tile.  Online and static kernels, each against fp64."""
    B, N = 2, 1000
    q, k, vt, keep, where = _dominant_case(B, Nq, N, masked, seed=Nq + masked)
    # every lane, and both ends of segments and the ragged last tile, carry a dominant key in every (frame, head)
    assert {w[4] for w in where} == set(range(64))
    ref = attn_ref(q, k, vt, keep)
    qn, kn = py_norms(q, k)
    assert float(((qn * kn[:, 0]).sqrt() * 1.0079 + 1e-3).max()) < STATIC_LIMIT   # the static kernel takes every item
    for name, norms in (("online", None), ("static", (qn, kn))):
        o, lse = run(q, k, vt, keep=keep, norms=norms)
        check(o, lse, ref, f"{name} Nq={Nq} masked={masked}")
        ob, _ = run(q, k, vt, keep=keep, norms=norms, o_dtype=torch.bfloat16)
        assert torch.equal(ob, o.bfloat16()), name


# ------------------------------------------------------------------------------------------
RAMP_SLOPES = [0.0, 2.0, 7.9, 8.1, 30.0, -5.0, -300.0]


def _ramp_case(B, Nq, N, masked, seed):
    """Row r of head h ramps its scores along the key axis by RAMP_SLOPES[(r + h) % 7] per 64-key tile (plus N(0, 1)
    noise on the key coordinate): no rescale (0), rare (2), every second step (7.9), every step (8.1, 30), a maximum
    in the first tile (-5) and scores falling below m - 125 within a tile (-300: the cubic's clamp).  The score is
    q0 k0 + q1 k1 exactly (other coordinates zero): k0 = t / 64 + noise, k1 = 1, q1 an offset per row."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(N, dtype=torch.float32)
    k = torch.zeros(B, H, N, 32)
    k[..., 0] = t / KT + torch.randn(B, H, N, generator=g)
    k[..., 1] = 1.0
    q = torch.zeros(B, Nq, H, 32)
    for h in range(H):
        idx = (torch.arange(Nq) + h) % len(RAMP_SLOPES)
        q[:, :, h, 0] = torch.tensor(RAMP_SLOPES)[idx]
        q[:, :, h, 1] = torch.randn(B, Nq, generator=g) * 4
    keep = None
    if masked:
        keep = torch.rand(B, N, generator=g) > 0.2
        # the first tile of every segment of head 0's items entirely padded: segments that open with m = -1e30
        pl = Plan(B, Nq, N, _sms(), False)
        for b in range(B):
            for qb in range(pl.qblocks):
                for j0, _ in pl.segments(qb * pl.BH + b * H)[1::2]:
                    keep[b, j0 * KT:(j0 + 1) * KT] = False
    return q.reshape(B, Nq, H * 32).bfloat16(), k.bfloat16(), _vt(B, N, g), keep


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("B,Nq,N", [(1, 900, 8000), (8, 384, 640)])
def test_running_max_ramps(B, Nq, N, masked):
    """Online kernel.  (1, 900, 8000): >= 6 segments per item; (8, 384, 640): CTAs carry parts of several items."""
    q, k, vt, keep = _ramp_case(B, Nq, N, masked, seed=B + N + masked)
    ref = attn_ref(q, k, vt, keep)
    o, lse = run(q, k, vt, keep=keep)
    check(o, lse, ref, f"ramps B={B} masked={masked}")


# ------------------------------------------------------------------------------------------
# target score bound |q||k| per head: even heads stay within STATIC_LIMIT (static kernel), odd heads exceed it
HEAD_BOUNDS = [20.0, 150.0, 59.0, 61.0, 40.0, 75.0, 57.0, 63.0]


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True])
def test_static_online_split_per_head(masked):
    """Norm maxima from the projection GEMMs' epilogues (project_queries / project_keys with norm2_max) choose the
    kernel per (frame, head): within one frame the even heads take the static kernel and the odd heads the online one,
    including heads just below and just above the bound 60.  Rows 0..63 have an aligned and an anti-aligned key, so the
    scores reach about +-0.95 of the bound."""
    B, Nq, N = 2, 300, 3000
    g = torch.Generator().manual_seed(41 + masked)
    alpha = ops.LOG2E / math.sqrt(32)
    dirs = torch.nn.functional.normalize(torch.randn(B, Nq, H, 32, generator=g), dim=-1)
    kdirs = torch.nn.functional.normalize(torch.randn(B, N, H, 32, generator=g), dim=-1)
    kmag = 0.3 + 0.7 * torch.rand(B, N, H, 1, generator=g)
    bnd = torch.tensor(HEAD_BOUNDS)
    qa = torch.sqrt(bnd) * (1.0 + 0.2 * (torch.arange(H) % 3))      # |q| per head, |k| = bound / |q|
    kc = bnd / qa
    kdirs = kdirs * kmag
    for r in range(64):
        kdirs[:, 10 * r + 5] = dirs[:, r]          # aligned
        kdirs[:, 10 * r + 9] = -dirs[:, r]         # anti-aligned
    xq = (dirs * qa[:, None] / alpha).reshape(B, Nq, H * 32).bfloat16()
    xk = (kdirs * kc[:, None]).reshape(B, N, H * 32).bfloat16()
    eye = torch.eye(H * 32).bfloat16().to(DEV)
    zero = torch.zeros(H * 32).to(DEV)
    qn = torch.zeros(B, H, device=DEV)
    kn = torch.zeros(B, H, device=DEV)
    qd = ops.project_queries(xq.to(DEV), eye, zero, H, alpha, norm2_max=qn)
    kd = ops.project_keys(xk.to(DEV), eye, zero, 1, H, norm2_max=kn)
    torch.cuda.synchronize()
    q, k = qd.cpu(), kd[:, 0].cpu()
    vt = _vt(B, N, g)
    keep = None
    if masked:
        keep = torch.rand(B, N, generator=g) > 0.25
        keep[:, 5:640:10] = True
        keep[:, 9:640:10] = True
    # the invariant the unclamped cubic of the static kernel relies on: no score exceeds the epilogue's bound
    s = (q.double().view(B, Nq, H, 32).permute(0, 2, 1, 3) @ k.double().transpose(-1, -2))   # [B,H,Nq,N]
    smax = s.abs().amax((-1, -2))
    bound = (qn.cpu().double() * kn.cpu().double()).sqrt()
    assert (smax <= bound * 1.0079 + 1e-3).all(), (smax, bound)
    assert (s.amax((-1, -2)) > 0.95 * bound).all() and (s.amin((-1, -2)) < -0.95 * bound).all()
    static = (bound.float() * 1.0079 + 1e-3) <= STATIC_LIMIT
    assert torch.equal(static, (torch.arange(H) % 2 == 0).expand(B, H))
    ref = attn_ref(q, k, vt, keep)
    o, lse = run(q, k, vt, keep=keep, norms=(qn.cpu(), kn.cpu().unsqueeze(1)))
    check(o, lse, ref, f"split masked={masked}")
    o0, lse0 = run(q, k, vt, keep=keep)
    check(o0, lse0, ref, f"no norms masked={masked}")
    assert ((o - o0).abs().cpu().double() <= 2 * TAU * ref[2]).all()


# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["simt_fp32", "online", "static"])
def test_no_attended_key(mode):
    """A query with no attended key gets o = 0 and lse = -inf (include/cmtcoop_b200.h, cmt_cross_attn_fwd).
    Frame 0: key_keep all False.  Frame 1: random padding (ordinary rows).  Token range [lo, hi) = [600, 1337):
    frame 2 has keys only outside it.  Frame 3: exactly one attended key, in the ragged last tile of the range.
    Frame 4: exactly one, on the first tile of a stream-K segment of its head-0 items."""
    B, Nq, N, lo, hi = 5, 417, 1500, 600, 1337
    g = torch.Generator().manual_seed(7)
    q = (torch.randn(B, Nq, H * 32, generator=g) * 0.3).bfloat16()
    k = torch.randn(B, H, N, 32, generator=g).bfloat16()
    vt = _vt(B, N, g)
    keep = torch.rand(B, N, generator=g) > 0.3
    keep[0] = False
    keep[2, lo:hi] = False
    keep[3] = False
    keep[3, hi - 3] = True
    pl = Plan(B, Nq, hi - lo, _sms(), mode == "static")
    j0 = pl.segments(0 * pl.BH + 4 * H)[-1][0]
    keep[4] = False
    keep[4, lo + j0 * KT + 17] = True
    ref = attn_ref(q, k, vt, keep, lo, hi)
    assert torch.isneginf(ref[1][[0, 2]]).all() and not torch.isinf(ref[1][[1, 3, 4]]).any()
    norms = py_norms(q, k) if mode == "static" else None
    if norms is not None:
        assert float(((norms[0] * norms[1][:, 0]).sqrt() * 1.0079 + 1e-3).max()) < STATIC_LIMIT
    if mode == "simt_fp32":
        o, lse = run(q.float(), k.float(), vt.float(), keep=keep, lo=lo, hi=hi)
    else:
        o, lse = run(q, k, vt, keep=keep, lo=lo, hi=hi, norms=norms)
    o, lse = o.cpu(), lse.cpu()
    assert torch.equal(o[[0, 2]], torch.zeros_like(o[[0, 2]])), f"{mode}: o of rows without keys {o[[0, 2]].abs().max()}"
    assert bool(torch.isneginf(lse[[0, 2]]).all()), f"{mode}: lse of rows without keys {lse[[0, 2]].max()}"
    if mode == "simt_fp32":   # fp32 CUDA-core kernel: exp2f and fp32 sums over <= 737 keys
        assert ((o.double() - ref[0]).abs() <= 1e-4 * ref[2] + 1e-6).all()
        fin = ~torch.isinf(ref[1])
        assert ((lse.double() - ref[1]).abs()[fin] <= 1e-4).all()
    else:
        check(o, lse, ref, mode)
    # the single-key frames: o is that key's value
    for b, t in ((3, hi - 3), (4, int(keep[4].nonzero()))):
        v = vt[b, :, :, t].double().reshape(H * 32)
        assert ((o[b].double() - v).abs() <= TAU * v.abs() + 1e-6).all(), (mode, b)


# ------------------------------------------------------------------------------------------
def _merge_ref(o, lse):
    """fp64 merge of G partials: o [G,B,Nq,H*32], natural-log lse [G,B,H,Nq]; rows whose every rank is -inf -> 0, -inf.
    Returns o, lse and A = sum_g w_g |o_g|."""
    G, B, Nq, HD = o.shape
    l = lse.double()
    tot = torch.logsumexp(l, 0)
    w = torch.exp(l - tot).nan_to_num(0.0)                            # all -inf: nan -> 0
    wt = w.permute(0, 1, 3, 2).unsqueeze(-1)                          # [G,B,Nq,H,1]
    ov = o.double().view(G, B, Nq, H, 32)
    return ((ov * wt).sum(0).reshape(B, Nq, HD), tot, (ov.abs() * wt).sum(0).reshape(B, Nq, HD))


def _merge_inputs(G, seed):
    """Rows in groups of four: rank LSEs 0, 30 and 100 apart (each rank g offset by g * gap, order shuffled), one rank at
    -inf, every rank at -inf."""
    g = torch.Generator().manual_seed(seed)
    B, Nq = 2, 37
    o = torch.randn(G, B, Nq, H * 32, generator=g)
    base = torch.randn(1, B, H, Nq, generator=g) * 5
    gap = torch.tensor([0.0, 30.0, 100.0])[torch.arange(Nq) % 3]
    order = torch.stack([torch.randperm(G, generator=g) for _ in range(Nq)], 1).float()   # [G, Nq]
    lse = (base + order[:, None, None, :] * gap).contiguous()
    if G > 1:
        lse[1, :, :, 1::4] = float("-inf")
    lse[:, :, :, 3::4] = float("-inf")
    lse[:, 0, 2, 5] = float("-inf")
    return o, lse


@pytest.mark.gpu
@pytest.mark.parametrize("o_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_lse_merge_edges(G, o_dtype):
    """cmt_lse_merge through both front ends: the stacked arrays (lse_merge) and the packed (O | LSE) records of one
    all-gather (lse_merge_packed).  The weights use __expf = 2^(x log2 e): for the |x| <= 90 that carry weight the
    rounding of x log2 e costs <= 130 * 2^-24 = 7.7e-6 relative, in numerator and denominator, so |o - o_ref| <= 2e-5 A,
    plus one bf16 rounding of o."""
    o, lse = _merge_inputs(G, 100 + G)
    want_o, want_l, A = _merge_ref(o, lse)
    tol = 2e-5 * A + (2.0 ** -8 * want_o.abs() if o_dtype == torch.bfloat16 else 0.0)
    got_o, got_l = ops.lse_merge(o.to(DEV), lse.to(DEV), o_dtype=o_dtype)
    B, Nq = o.shape[1], o.shape[2]
    rec = B * Nq * H * 32 + B * H * Nq
    parts = torch.empty(G * rec, device=DEV)                          # G packed records back to back
    for r in range(G):
        parts[r * rec:r * rec + B * Nq * H * 32] = o[r].reshape(-1).to(DEV)
        parts[r * rec + B * Nq * H * 32:(r + 1) * rec] = lse[r].reshape(-1).to(DEV)
    got_p = ops.lse_merge_packed(parts, G, B, Nq, H, o_dtype=o_dtype)
    torch.cuda.synchronize()
    for name, got in (("stacked", got_o), ("packed", got_p)):
        err = (got.cpu().double() - want_o).abs()
        assert (err <= tol).all(), (name, float((err - tol).max()))
    assert torch.equal(got_o.cpu(), got_p.cpu())
    dead = torch.isneginf(want_l)
    assert int(dead.sum()) > 0 and torch.equal(torch.isneginf(got_l.cpu()), dead)
    o_rows = got_o.cpu().view(B, Nq, H, 32).permute(0, 2, 1, 3)[dead]
    assert torch.equal(o_rows, torch.zeros_like(o_rows))
    lerr = (got_l.cpu().double() - want_l).abs()[~dead]
    assert (lerr <= 1e-5 + 2.0 ** -20 * want_l.abs()[~dead]).all(), float(lerr.max())
