"""Every non-GEMM launch of one eager forward of the benched workloads, replayed element by element against fp64 on the
launch's own recorded operands (the GEMM family is replayed by test_gpu_gemm_geometry.py).

A recorder stands in for every public function of ops that launches a kernel (each one that calls ops._count), clones
the launch's operands and outputs on the same stream and, for a launch that writes into part of a larger buffer
(cross_attn(out=ctx[f0:f0 + nb]), add_layernorm(y2=out[li]), gather_tokens(out=(xk, xv), n_bev_reserved=...)), the
whole buffer before and after: only the addressed elements may change.  The per-launch launch_count() deltas must add
up to the forward's, and every recorded op must be checked here, by the GEMM replay, or be listed in EXCLUDED with its
reason, so a kernel added to the forward later fails until it has a check.

Bounds (u = 2^-24, fp32 unit roundoff; u_out = 2^-8 bf16, 2^-11 fp16, 0 fp32 output rounding):

Attention (cross_attn, cross and self).  Per element |o - o_ref| <= (tau + eps_score) A + u_out |o_ref| (+ sub), with
A = sum_j p_j |v_j| and tau from test_gpu_attention_edges.py, which derives it for scores that are one or two exact
products.  Here the scores are general 32-term dot products accumulated in fp32: each carries at most
32 u sum_i |q_i k_ji| (log2 units; x ln2 in natural units).  A weight p_j = e^(s_j) / sum e^(s_k) whose scores are
each off by at most d moves by a factor within e^(+-2d), so o moves by <= 2 d A and the LSE by <= d:
    eps_score = GAMMA * 32 u ln2 max_j sum_i |q_i k_ji|,     GAMMA = 2.
tau per operand type: bf16 2^-7 (edges file: 2^-8 rounding of P, 1.5e-4 exponential, x1.9 margin); fp16: P rounded
to fp16 (2^-11) + the same 1.5e-4 = 6.4e-4, tau = 2^-10 (x1.5 margin); the fp16 online kernel's lazy rescale can
leave weights below 2^-14, where P is subnormal with absolute error <= 2^-25 while l >= 1 / p_max:
sub = 2^-25 p_max sum_j |v_j|.  fp32 (CUDA-core kernel, keys summed one at a time into o and l):
tau = 2^-22 + 2 (N + 32) u.
LSE (natural log, per row): the edges file's 3e-4 covers (64 + T) u of fp32 sums plus 7.5e-5 of the exponential with
a x2 margin up to T ~ 1100 tile-steps (the benched 56 400 keys are T = 882); plus eps_score and 2^-20 |lse| (fp32
spacing and the ln 2 conversion).  fp32 kernel: 2 (N + 32) u + 2^-21.  The forward does not ask for the LSE, so each
recorded call is launched again with return_lse=True and an fp32 output, and the recorded output must be that output
rounded to the compute type, bit for bit.  A dropped or repeated 64-key tile of near-uniform attention over 56 400 keys
moves o by ~1e-3 A (inside tau) but the LSE by ~1.1e-3 (outside): the LSE check is what sees it.

LayerNorm (add_layernorm).  y against the fp64 LayerNorm of the fp32-rounded x + r (what the kernel normalises), y2
against the fp64 LayerNorm of the kernel's own y:
    |y - y_ref| <= C_LN 2^-23 (|gamma| rstd (|v - mu| + mean|v|) + |beta|)
(the mean is off by a few u of mean|v|, the variance and rsqrtf by a few u relative, each step of the affine map by one
rounding).  ylp == y.to(lp) and yadd == (y + add).to(lp) bit for bit.

Task-head tail.  fp64 GroupLayerNorm -> ReLU -> Conv1d(k) (zero padding at both ends of each frame) -> decode
(sigmoid with scale and offset) from the recorded h:  |out - ref| <= C_TH 2^-23 S before the decode, S =
sum_t sum_c (|y| + E_LN) |w2| + |b2| with E_LN = |gamma| (|h - mu| + mean|h|) / sd + |beta| the LayerNorm's error scale;
through the decode: scale (sigma (1 - sigma) C_TH 2^-23 S + 4 u sigma) + 2 u |ref|.

Position encodings.  ray_pe / ray_query_pe: C_PE u (sum of the magnitudes of the projection's terms) / |range|, plus
the propagated error of px, py, pz (query PE) and u_out |ref|.  pos2embed: C_POS u (|a| + 1) + u_out |ref|, a the
angle.  The query PE's view mask is exact except for points whose fp64 px / py lie within their error bound of an image
border or whose depth is within 1e-3 of the camera plane; there either mask value is accepted, and a point that comes
out outside the view must have zero features.  masked_view_sum: fp64 with (V + 1) u (sum |e m| + |base|), and bit for
bit against the same fp32 sum in the kernel's fixed view order with the base added last.

Bit exact against a torch emulation: gather_tokens, nchw_to_padded_nhwc (guard and border rows exactly zero),
sensor_key_keep, split3 (nan_to_num, the node max and the clamp of the largest bf16 included).

Constants calibrated on a B200 (148 SMs, 1000 W power limit).  Largest observed ratio over the whole replay (all
workloads, precisions and mask cases) of the error, output rounding taken out, to the unit each constant multiplies:
    C_LN = 4     y 1.71, y2 1.79                    C_TH = 16    6.28 (k = 1 and k = 3 with the decode)
    C_PE = 16    ray_pe 2.11, ray_query_pe 2.12    C_POS = 8    1.71
and of the error to the whole attention bound:  o   bf16 0.34, fp16 0.46, fp32 0.029;
                                                LSE bf16 0.12, fp16 0.11, fp32 0.019.
"""
import inspect
import math
import re
import time

import numpy as np
import pytest
import torch

from cmtcoop_b200 import ops, synth
from test_gpu_attention_edges import H, KT, LSE_TOL, QBLK, TAU, Plan

DEV = "cuda:0"
B200_SMS = 148
U = 2.0 ** -24
LN2 = math.log(2.0)
U_OUT = {torch.float32: 0.0, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
GAMMA = 2.0
TAU_F16 = 2.0 ** -10
STATIC_LIMIT = {torch.bfloat16: 60.0, torch.float16: 14.0}
C_LN = 4.0
C_TH = 16.0
C_PE = 16.0
C_POS = 8.0

# ops that launch kernels, by who checks them
CHECKED = {"add_layernorm", "cross_attn", "ray_pe", "ray_query_pe", "masked_view_sum", "pos2embed", "gather_tokens",
           "nchw_to_padded_nhwc", "sensor_key_keep", "split3", "task_head_tail"}
GEMM_REPLAYED = {"gemm", "gemm_segmented", "shared_conv_tokens"}     # test_gpu_gemm_geometry.py
EXCLUDED = {
    "bbox_topk_decode": "not in forward_single; test_gpu_bbox_decode.py checks it bit for bit against torch",
    "lse_merge": "KV-split merge, not in the single-GPU forward; test_gpu_attention_edges.py covers it",
    "lse_merge_packed": "KV-split merge, not in the single-GPU forward; test_gpu_attention_edges.py covers it",
    "lse_merge_peer": "KV-split merge over peer memory, not in the single-GPU forward; test_gpu_fp16.py covers it",
    "coop_max": "not on the fused path (the cooperative max rides in split3); test_gpu_kernels.py checks it exactly",
}


def launching_ops():
    """Public functions of ops that launch a kernel: the ones that call _count."""
    return sorted(n for n, f in vars(ops).items() if inspect.isfunction(f) and f.__module__ == ops.__name__
                  and not n.startswith("_") and re.search(r"(?<!\w)_count\(", inspect.getsource(f)))


def _ulp_ratio(err, unit):
    """max err / unit over the elements with unit > 0 (0 for empty)."""
    if err.numel() == 0:
        return 0.0
    return float((err / unit.clamp_min(1e-300)).max())


def _first(bad):
    """Index tuple of the first True of a bool tensor."""
    i = int(torch.argmax(bad.flatten().to(torch.uint8)))
    return tuple(int(v) for v in np.unravel_index(i, tuple(bad.shape)))


def _bits(t):
    return t.view({1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


def same_bits(got, want, what):
    assert got.shape == want.shape and got.dtype == want.dtype, f"{what}: {got.shape} {got.dtype} vs {want.shape} {want.dtype}"
    ne = _bits(got.contiguous()) != _bits(want.contiguous())
    if bool(ne.any()):
        idx = _first(ne)
        raise AssertionError(f"{what}: {int(ne.sum())} of {ne.numel()} elements differ; first at {list(idx)}: "
                             f"got {float(got[idx])!r} want {float(want[idx])!r}")


# ------------------------------------------------------------------------------------------
# 1. grid replicas of the launchers (grid-stride loops whose grid is capped at a multiple of the SM count)
def grid_replica(op, a, sms):
    """(work items, items one pass of the capped grid covers) of a recorded launch, or None for the kernels that launch
    one block per tile / row (ray_pe, gather_tokens, nchw_to_padded_nhwc, task_head_tail, cross_attn): no grid-stride
    loop, nothing to wrap."""
    cap16 = sms * 16
    if op == "add_layernorm":
        C = a["x"].shape[-1]
        M = math.prod(a["rows"]) if a["rows"] is not None else a["x"].numel() // C
        return M, min(-(-M // 8), sms * 8) * 8                                       # 8 rows (warps) per block
    if op == "split3":
        L, B, Nq, _ = a["a"].shape
        if a["stacked_nodes"]:
            B //= 2
        rows = L * B * (Nq + 2)
        return rows, min(-(-rows // 8), cap16) * 8
    if op == "ray_query_pe":
        B, Nq, _ = a["ref"].shape
        total = B * a["lidar2img"].shape[1] * Nq * (a["depth_num"] * 3 // 8)
    elif op == "masked_view_sum":
        B, V, Nq, C = a["emb"].shape
        total = B * Nq * C
    elif op == "pos2embed":
        total = a["pos"].numel() // a["pos"].shape[-1] * 2 * a["num_pos_feats"]
    elif op == "sensor_key_keep":
        total = a["B"] * (a["n_bev"] + a["V"] * a["n_img"])
    else:
        return None
    return total, min(-(-total // 256), cap16) * 256


def wraps(op, a, sms):
    r = grid_replica(op, a, sms)
    return None if r is None else r[0] > r[1]


def test_every_launching_op_is_classified():
    """A new kernel entry point of ops must get a check (here or in the GEMM replay) or an exclusion with a reason."""
    ops_ = set(launching_ops())
    assert ops_ == CHECKED | GEMM_REPLAYED | set(EXCLUDED), (ops_ - (CHECKED | GEMM_REPLAYED | set(EXCLUDED)),
                                                             (CHECKED | GEMM_REPLAYED | set(EXCLUDED)) - ops_)
    assert not (CHECKED & GEMM_REPLAYED) and not (CHECKED & set(EXCLUDED)) and not (GEMM_REPLAYED & set(EXCLUDED))


def test_grid_replicas_at_the_benched_sizes():
    """Which launches of the benched forward (B = 8, Nq = 900, 6 layers, 180 x 180 BEV, 6 cameras of 40 x 100) run a
    second pass of their grid-stride loop on 148 SMs.  add_layernorm wraps only in the cooperative pass (both nodes'
    frames: 14 400 rows against 9 472 per pass); gather_tokens has no grid-stride loop (one block per 32-token tile and
    frame), so it cannot wrap -- the replay checks that its tiles address every gathered row once instead."""
    sms = B200_SMS
    t = torch.empty(0)

    def ln(M):
        return dict(x=t.new_empty(M, 256), rows=None)
    assert grid_replica("add_layernorm", ln(7200), sms) == (7200, 7200)
    assert grid_replica("add_layernorm", ln(14400), sms) == (14400, 9472)
    assert grid_replica("add_layernorm", dict(x=t.new_empty(256), rows=(8, 900)), sms) == (7200, 7200)
    assert grid_replica("split3", dict(a=t.new_empty(6, 8, 900, 256), stacked_nodes=False), sms) == (43296, 18944)
    assert grid_replica("split3", dict(a=t.new_empty(6, 16, 900, 256), stacked_nodes=True), sms) == (43296, 18944)
    assert grid_replica("ray_query_pe", dict(ref=t.new_empty(8, 900, 3), lidar2img=t.new_empty(8, 6, 4, 4), depth_num=64),
                        sms) == (1036800, 606208)
    assert grid_replica("masked_view_sum", dict(emb=t.new_empty(8, 6, 900, 256)), sms) == (1843200, 606208)
    assert grid_replica("pos2embed", dict(pos=t.new_empty(32400, 2), num_pos_feats=256), sms) == (16588800, 606208)
    assert not wraps("pos2embed", dict(pos=t.new_empty(1, 900, 3), num_pos_feats=256), sms)      # the query grid
    assert not wraps("sensor_key_keep", dict(B=8, n_bev=32400, V=6, n_img=4000), sms)
    for op in ("gather_tokens", "nchw_to_padded_nhwc", "ray_pe", "task_head_tail", "cross_attn"):
        assert grid_replica(op, {}, sms) is None


# ------------------------------------------------------------------------------------------
# 2. references and element checks (device-agnostic: the host tests run them on the CPU)
def tau(dtype, n_keys):
    if dtype == torch.float32:
        return 2.0 ** -22 + 2 * (n_keys + 32) * U
    return TAU if dtype == torch.bfloat16 else TAU_F16


def lse_tol(dtype, n_keys):
    if dtype == torch.float32:
        return 2 * (n_keys + 32) * U + 2.0 ** -21
    assert -(-n_keys // KT) <= 1100, "LSE_TOL is derived for at most ~1100 tile-steps"
    return LSE_TOL


def attn_reference(q, k, v, keep=None):
    """fp64 attention of one frame: q [h, Nq, 32] (log2 units), k, v [h, N, 32], keep [N] bool or None.
    -> dict(o, lse (natural log, -inf without a key), A, smax = max_j sum_i |q_i k_ji|, pmax, V1 = sum_j |v_j|)."""
    qd, kd, vd = q.double(), k.double(), v.double()
    if keep is not None:
        kd, vd = kd[:, keep], vd[:, keep]
    h, Nq, _ = qd.shape
    if kd.shape[1] == 0:
        z = torch.zeros(h, Nq, dtype=torch.float64, device=qd.device)
        return dict(o=torch.zeros_like(qd), A=torch.zeros_like(qd), lse=z - math.inf, smax=z, pmax=z,
                    V1=torch.zeros(h, 32, dtype=torch.float64, device=qd.device))
    s = torch.matmul(qd, kd.transpose(1, 2)).mul_(LN2)
    smax = torch.matmul(qd.abs(), kd.abs().transpose(1, 2)).amax(-1)
    lse = torch.logsumexp(s, -1)
    p = s.sub_(lse[..., None]).exp_()
    return dict(o=torch.matmul(p, vd), A=torch.matmul(p, vd.abs()), lse=lse, smax=smax, pmax=p.amax(-1),
                V1=vd.abs().sum(1))


def check_attention(o, lse, ref, dtype, n_keys, *, what, frame, head0=0, where=lambda h, r: "", stats=None):
    """o [h, Nq, 32] as stored (dtype: the operand type; o in that type or fp32), lse [h, Nq] or None; the h heads are
    heads head0, head0 + 1, ... of the frame."""
    u_out = U_OUT[o.dtype]
    eps = GAMMA * 32 * U * LN2 * ref["smax"]
    dead = torch.isneginf(ref["lse"])
    od = o.double()
    if bool(dead.any()):
        hd, r = _first(dead)
        assert bool((od[dead] == 0).all()), f"{what}: frame {frame}, head {hd + head0}: rows without a key must be 0"
        if lse is not None:
            assert bool(torch.isneginf(lse[dead]).all()), f"{what}: frame {frame}: LSE of rows without a key must be -inf"
    live = ~dead
    if lse is not None:
        lerr = (lse.double() - ref["lse"]).abs()
        ltol = lse_tol(dtype, n_keys) + eps + 2.0 ** -20 * ref["lse"].abs()
        bad = live & ~(lerr <= ltol)
        if bool(bad.any()):
            hd, r = _first(bad)
            raise AssertionError(
                f"{what}: LSE of {int(bad.sum())} rows outside the bound; first at frame {frame}, head {hd + head0}, query {r} "
                f"(query block {r // QBLK}): got {float(lse[hd, r])!r} want {float(ref['lse'][hd, r])!r} |err| "
                f"{float(lerr[hd, r]):.3e} > {float(ltol[hd, r]):.3e}{where(hd + head0, r)}")
        if stats is not None:
            stats["lse"] = max(stats.get("lse", 0.0), _ulp_ratio(lerr[live], ltol[live]))
    tol = (tau(dtype, n_keys) + eps[..., None]) * ref["A"] + u_out * ref["o"].abs()
    if dtype == torch.float16:
        tol = tol + 2.0 ** -25 * ref["pmax"][..., None] * ref["V1"][:, None, :]
    err = (od - ref["o"]).abs()
    bad = live[..., None] & ~(err <= tol)
    if bool(bad.any()):
        hd, r, d = _first(bad)
        raise AssertionError(
            f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; first at frame {frame}, head {hd + head0}, "
            f"query {r} (query block {r // QBLK}), dim {d}: got {float(od[hd, r, d])!r} want "
            f"{float(ref['o'][hd, r, d])!r} |err| {float(err[hd, r, d]):.3e} > {float(tol[hd, r, d]):.3e} "
            f"(A {float(ref['A'][hd, r, d]):.3e}){where(hd + head0, r)}")
    if stats is not None:
        stats["o"] = max(stats.get("o", 0.0), _ulp_ratio(err[live], tol[live]))


def plan_where(plan, b, static):
    """Names the stream-K segments of the failing row's item: its 64-key tiles and the CTAs that own them."""
    if plan is None:
        return lambda hd, r: f"; CUDA-core kernel block ({r // 128}, head {hd}, frame {b})"

    def where(hd, r):
        item = (r // QBLK) * plan.BH + b * H + hd
        segs = ", ".join(f"tiles [{j0}, {j1}) -> CTA {plan.cta_of(item * plan.T + j0)}" for j0, j1 in plan.segments(item))
        return f"; item {item} ({'static' if static else 'online'} plan, {plan.T} tiles): {segs}"
    return where


def ln_reference(v, gamma, beta, eps):
    """fp64 LayerNorm of rows v [..., C] and the unit of its bound: S = |gamma| rstd (|v - mu| + mean|v|) + |beta|."""
    v = v.double()
    mu = v.mean(-1, keepdim=True)
    d = v - mu
    rstd = (d.pow(2).mean(-1, keepdim=True) + eps).rsqrt()
    g, b = gamma.double(), beta.double()
    return d * rstd * g + b, g.abs() * rstd * (d.abs() + v.abs().mean(-1, keepdim=True)) + b.abs()


def check_ln(got, want, S, *, what, Nq, grid_rows=None, stats=None, key="y"):
    """got, want, S [M, C]; grid_rows: rows one pass of the launch covers (names the pass of a failing row)."""
    err = (got.double() - want).abs()
    bound = C_LN * 2.0 ** -23 * S
    bad = ~(err <= bound)
    if bool(bad.any()):
        r, c = _first(bad)
        gi = c // 4
        pas = f", grid pass {r // grid_rows}" if grid_rows else ""
        raise AssertionError(
            f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; first at row {r} (frame {r // Nq}, "
            f"query {r % Nq}{pas}), column {c} (4-column group {gi}: lane {gi % 32}, step {gi // 32}): got "
            f"{float(got[r, c])!r} want {float(want[r, c])!r} |err| {float(err[r, c]):.3e} > {float(bound[r, c]):.3e}")
    if stats is not None:
        stats[key] = max(stats.get(key, 0.0), _ulp_ratio(err, 2.0 ** -23 * S))


def task_tail_reference(h, gamma, beta, w2, b2, eps, ksize, Nq, ref_logit=None, comp=None, scale=None, offset=None):
    """fp64 GroupLayerNorm -> ReLU -> Conv1d(ksize) over each frame's query axis (zero padded) -> decode.
    h [L, M, NH, 64]; w2 [L, NH, CMAX, ksize, 64].  -> (out [L, M, NH, CMAX], bound [L, M, NH, CMAX])."""
    L, M, NH, HC = h.shape
    hd = h.double()
    mu = hd.mean(-1, keepdim=True)
    d = hd - mu
    sd = (d.pow(2).mean(-1, keepdim=True) + eps).sqrt()
    g, b = gamma.double()[:, None], beta.double()[:, None]
    y = (d / sd * g + b).clamp_min(0.0)
    E = g.abs() * (d.abs() + hd.abs().mean(-1, keepdim=True)) / sd + b.abs()
    w = w2.double()
    out = b2.double()[:, None].expand(L, M, NH, w.shape[2]).clone()
    S = out.abs()
    q = torch.arange(M, device=h.device) % Nq
    for t in range(ksize):
        dq = t - ksize // 2
        ok = ((q + dq >= 0) & (q + dq < Nq)).double()[None, :, None, None]
        yt = torch.roll(y, -dq, 1) * ok
        et = torch.roll(E, -dq, 1) * ok
        out += torch.einsum("lmnc,lnoc->lmno", yt, w[:, :, :, t])
        S += torch.einsum("lmnc,lnoc->lmno", yt.abs() + et, w[:, :, :, t].abs())
    bound = C_TH * 2.0 ** -23 * S
    if ref_logit is not None:
        NHC = comp.reshape(NH, -1)
        for hh in range(NH):
            for o in range(NHC.shape[1]):
                c = int(NHC[hh, o])
                if c < 0:
                    continue
                z = out[:, :, hh, o] + ref_logit.double()[None, :, c]
                sig = torch.sigmoid(z)
                sc, of = float(scale.reshape(NH, -1)[hh, o]), float(offset.reshape(NH, -1)[hh, o])
                val = sig * sc + of
                bound[:, :, hh, o] = abs(sc) * (sig * (1 - sig) * bound[:, :, hh, o] + 4 * U * sig) + 2 * U * val.abs()
                out[:, :, hh, o] = val
    return out, bound


def check_task_tail(outs, want, bound, couts, *, what, Nq, stats=None):
    """outs: the kernel's per-head tensors [L, M, c_i]; want, bound [L, M, NH, CMAX]."""
    for hh, (o, co) in enumerate(zip(outs, couts)):
        err = (o.double() - want[:, :, hh, :co]).abs()
        bnd = bound[:, :, hh, :co]
        bad = ~(err <= bnd)
        if bool(bad.any()):
            l, m, c = _first(bad)
            raise AssertionError(
                f"{what}: {int(bad.sum())} elements of head {hh} outside the bound; first at layer {l}, row {m} "
                f"(frame {m // Nq}, query {m % Nq}), output {c}: got {float(o[l, m, c])!r} want "
                f"{float(want[l, m, hh, c])!r} |err| {float(err[l, m, c]):.3e} > {float(bnd[l, m, c]):.3e}")
        if stats is not None:
            stats["th"] = max(stats.get("th", 0.0), _ulp_ratio(err, bnd / C_TH))


def view_sum_emulation(emb, mask, base, view_valid):
    """The kernel's fp32 sum in its order: views 0..V-1 (absent views skipped), then base + sum."""
    B, V, Nq, C = emb.shape
    acc = torch.zeros(B, Nq, C, dtype=torch.float32, device=emb.device)
    for v in range(V):
        term = emb[:, v].float() * mask[:, v, :, None]
        if view_valid is None:
            acc = acc + term
        else:
            acc = torch.where(view_valid[v][:, None, None], acc + term, acc)
    return acc if base is None else base + acc


def view_sum_reference(emb, mask, base, view_valid):
    """fp64 base + sum_v e m and its bound (V + 1) u (sum |e m| + |base|)."""
    B, V, Nq, C = emb.shape
    e = emb.double() * mask.double()[..., None]
    if view_valid is not None:
        e = torch.where(view_valid.t()[:, :, None, None], e, torch.zeros((), dtype=e.dtype, device=e.device))
    want, S = e.sum(1), e.abs().sum(1)
    if base is not None:
        want, S = want + base.double(), S + base.double().abs()
    return want, (V + 1) * U * S


def check_view_sum(got, want, bound, *, what, stats=None):
    err = (got.double() - want).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        b, n, c = _first(bad)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; first at frame {b}, "
                             f"query {n}, channel {c}: got {float(got[b, n, c])!r} want {float(want[b, n, c])!r}")
    if stats is not None:
        stats["sum"] = max(stats.get("sum", 0.0), _ulp_ratio(err, bound))


def query_pe_reference(ref, l2i, i2l, D, pad_h, pad_w, pc):
    """fp64 reference-point re-projection (cmt_head.py:439-464) of the fp32 operands.
    -> dict(feat [B,V,Nq,3D], mask [B,V,Nq] bool, amb [B,V,Nq] bool (mask decision within rounding), bound [B,V,Nq,3D])."""
    f32 = lambda x: float(np.float32(x))   # noqa: E731
    pmin = torch.tensor([f32(pc[c]) for c in range(3)], dtype=torch.float64, device=ref.device)
    rng = torch.tensor([f32(f32(pc[c + 3]) - f32(pc[c])) for c in range(3)], dtype=torch.float64, device=ref.device)
    P = ref.double() * rng + pmin                                            # [B, Nq, 3]
    Ph = torch.cat([P, torch.ones_like(P[..., :1])], -1)                     # [B, Nq, 4]
    L = l2i.double()[:, :, :3]                                               # [B, V, 3, 4]
    s = torch.einsum("bvci,bni->bvnc", L, Ph)
    Ts = torch.einsum("bvci,bni->bvnc", L.abs(), Ph.abs())
    zpos = s[..., 2] > 0
    den = torch.where(zpos, s[..., 2] + 1e-6, s[..., 2] - 1e-6)
    p = s / den[..., None]                                                   # px, py, pz
    ep = 8 * U * (Ts + p.abs() * Ts[..., 2:3]) / den.abs()[..., None]        # absolute error of px, py, pz
    inside = (p[..., 0] < pad_w) & (p[..., 0] >= 0) & (p[..., 1] < pad_h) & (p[..., 1] >= 0) & zpos
    amb = ((p[..., 0].abs() <= ep[..., 0]) | ((p[..., 0] - pad_w).abs() <= ep[..., 0]) |
           (p[..., 1].abs() <= ep[..., 1]) | ((p[..., 1] - pad_h).abs() <= ep[..., 1]) | (s[..., 2].abs() <= 1e-3))
    k = torch.arange(3 * D, device=ref.device) // 3
    c = torch.arange(3 * D, device=ref.device) % 3
    d = 1.0 + k.double() * f32(f32(pc[3]) - 1.0) / D                         # [3D]
    R = i2l.double()[:, :, :3]                                               # [B, V, 3, 4]
    Rc = R[:, :, c]                                                          # [B, V, 3D, 4]
    terms = p[:, :, :, None, :] * d[:, None] * Rc[:, :, None, :, :3]         # [B, V, Nq, 3D, 3]
    acc = terms.sum(-1) + Rc[:, :, None, :, 3]
    feat = (acc - pmin[c]) / rng[c]
    T = terms.abs().sum(-1) + Rc[:, :, None, :, 3].abs() + pmin[c].abs()
    prop = (ep[:, :, :, None, :] * d[:, None] * Rc[:, :, None, :, :3].abs()).sum(-1)
    bound = (C_PE * U * T + prop) / rng[c]
    return dict(feat=feat, mask=inside, amb=amb, bound=bound)


def check_query_pe(feat, mask, ref, *, what, stats=None):
    """feat [B,V,Nq,3D] (stored type), mask [B,V,Nq] fp32 from the kernel against query_pe_reference."""
    got_in = mask != 0
    assert bool(((mask == 0) | (mask == 1)).all()), f"{what}: mask values other than 0 / 1"
    diff = (got_in != ref["mask"]) & ~ref["amb"]
    if bool(diff.any()):
        b, v, n = _first(diff)
        raise AssertionError(f"{what}: view mask of {int(diff.sum())} points differs; first at frame {b}, view {v}, "
                             f"query {n}: got {bool(got_in[b, v, n])} want {bool(ref['mask'][b, v, n])}")
    out = ~got_in
    zero = feat[out] == 0
    assert bool(zero.all()), f"{what}: a point outside the view has non-zero features"
    if feat.dtype == torch.float16:
        assert bool(torch.isfinite(feat).all()), f"{what}: non-finite fp16 features"
    err = (feat.double() - ref["feat"]).abs()
    bound = ref["bound"] + U_OUT[feat.dtype] * ref["feat"].abs()
    bad = got_in[..., None] & ~(err <= bound)
    if bool(bad.any()):
        b, v, n, f = _first(bad)
        raise AssertionError(
            f"{what}: {int(bad.sum())} features outside the bound; first at frame {b}, view {v}, query {n}, feature {f} "
            f"(depth bin {f // 3}, coordinate {f % 3}): got {float(feat[b, v, n, f])!r} want "
            f"{float(ref['feat'][b, v, n, f])!r} |err| {float(err[b, v, n, f]):.3e} > {float(bound[b, v, n, f]):.3e}")
    if stats is not None:
        sel = got_in[..., None].expand_as(err)           # in units of the C_PE term, the output rounding taken out
        stats["qpe"] = max(stats.get("qpe", 0.0), _ulp_ratio((err - U_OUT[feat.dtype] * ref["feat"].abs())[sel],
                                                             ref["bound"][sel] / C_PE))
    return int((ref["amb"] & (got_in != ref["mask"])).sum()), int(ref["amb"].sum())


# ------------------------------------------------------------------------------------------
# 3. host tests of the bounds: a simulated correct fp32 kernel passes, simulated bugs fail and are located
def _sim_attention(q, k, v, keep=None, drop=None):
    """What the tcgen05 kernel computes, in fp32 on the host: q [h, Nq, 32], k, v [h, N, 32] bf16; scores in fp32,
    weights 2^(s - m) rounded to bf16 for P V, the normaliser from the unrounded weights.  drop: keys left out."""
    s = torch.matmul(q.float(), k.float().transpose(1, 2))
    if keep is not None:
        s[:, :, ~keep] = -math.inf
    if drop is not None:
        s[:, :, drop] = -math.inf
    m = s.amax(-1, keepdim=True)
    e = torch.exp2(s - m)
    l = e.sum(-1, keepdim=True)
    o = torch.matmul(e.bfloat16().float(), v.float()) / l
    return o.bfloat16(), ((m + torch.log2(l)) * LN2)[..., 0]


def test_attention_check_accepts_a_correct_kernel_and_rejects_mutants():
    """(a) Near-uniform attention of 16 queries over the benched 56 400 keys (32 400 BEV + 6 cameras x 4 000), two
    frames, the second with camera 2 masked out: a dropped tile and an unmasked camera.  (b) Peaked attention over 3 000
    keys: swapped heads, the wrong frame in a coop slice, a query row read from its neighbour."""
    g = torch.Generator().manual_seed(3)

    def case(B, Nq, N, qscale, keep):
        q = (torch.randn(B, H, Nq, 32, generator=g) * qscale).bfloat16()
        k = torch.randn(B, H, N, 32, generator=g).bfloat16()
        v = torch.randn(B, H, N, 32, generator=g).bfloat16()
        refs = [attn_reference(q[b], k[b], v[b], None if keep is None else keep[b]) for b in range(B)]
        sims = [_sim_attention(q[b], k[b], v[b], None if keep is None else keep[b]) for b in range(B)]
        plan = Plan(B, Nq, N, B200_SMS, False)

        def check(outs, label="sim"):
            for b in range(B):
                check_attention(outs[b][0], outs[b][1], refs[b], torch.bfloat16, N, what=label, frame=b,
                                where=plan_where(plan, b, False))
        check(sims)
        return q, k, v, refs, sims, check

    # (a)
    B, Nq, N, n_bev, n_img = 2, 16, 56400, 32400, 4000
    keep = torch.ones(B, N, dtype=torch.bool)
    cam2 = slice(n_bev + 2 * n_img, n_bev + 3 * n_img)
    keep[1, cam2] = False
    q, k, v, refs, sims, check = case(B, Nq, N, 0.05, keep)
    # a dropped 64-key tile (tile 300 of frame 0, head 3): o stays inside tau, the LSE does not
    o3, l3 = _sim_attention(q[0, 3:4], k[0, 3:4], v[0, 3:4], keep[0], drop=slice(300 * KT, 301 * KT))
    o, l = sims[0][0].clone(), sims[0][1].clone()
    o[3], l[3] = o3[0], l3[0]
    check_attention(o, None, refs[0], torch.bfloat16, N, what="o alone", frame=0)
    with pytest.raises(AssertionError, match=r"LSE of 16 rows .* frame 0, head 3, query 0 .*item 3 .*tiles \[0, "):
        check([(o, l), sims[1]])
    # one camera's key span left unmasked in frame 1
    keep_bad = keep[1].clone()
    keep_bad[cam2] = True
    with pytest.raises(AssertionError, match=r"LSE of 128 rows .* frame 1, head 0, query 0 "):
        check([sims[0], _sim_attention(q[1], k[1], v[1], keep_bad)])
    # (b)
    q, k, v, refs, sims, check = case(2, 40, 3000, 0.5, None)
    perm = [0, 1, 5, 3, 4, 2, 6, 7]
    with pytest.raises(AssertionError, match=r"frame 1, head 2, query \d+ "):
        check([sims[0], (sims[1][0][perm], sims[1][1][perm])])
    with pytest.raises(AssertionError, match=r"frame 1, head 0, query \d+ "):     # frame 1's slice holds frame 0's rows
        check([sims[0], sims[0]])
    o, l = sims[0][0].clone(), sims[0][1].clone()
    o[6, 10], l[6, 10] = o[6, 11], l[6, 11]
    with pytest.raises(AssertionError, match=r"frame 0, head 6, query 10 \(query block 0\)"):
        check([(o, l), sims[1]])


def _sim_ln(v, g, b, eps, *, unbiased=False, eps_outside=False):
    mean = v.sum(-1, keepdim=True) / v.shape[-1]
    d = v - mean
    var = (d * d).sum(-1, keepdim=True) / (v.shape[-1] - (1 if unbiased else 0))
    rstd = 1.0 / (var.sqrt() + eps) if eps_outside else torch.rsqrt(var + eps)
    return d * rstd * g + b


def test_layernorm_check_accepts_a_correct_kernel_and_rejects_mutants():
    gen = torch.Generator().manual_seed(4)
    M, C, Nq, eps = 1800, 256, 900, 1e-5
    x = torch.randn(M, C, generator=gen) * 3 + 0.5
    r = torch.randn(M, C, generator=gen)
    g = 1 + 0.05 * torch.randn(C, generator=gen)
    b = 0.02 * torch.randn(C, generator=gen)
    g2 = 1 + 0.05 * torch.randn(C, generator=gen)
    b2 = 0.02 * torch.randn(C, generator=gen)
    v = x + r
    y = _sim_ln(v, g, b, eps)
    y2 = _sim_ln(y, g2, b2, eps)
    want, S = ln_reference(v, g, b, eps)
    want2, S2 = ln_reference(y, g2, b2, eps)
    check_ln(y, want, S, what="y", Nq=Nq)
    check_ln(y2, want2, S2, what="y2", Nq=Nq)
    with pytest.raises(AssertionError, match=r"^y: .*first at row 0 \(frame 0, query 0\)"):
        check_ln(_sim_ln(v, g, b, eps, unbiased=True), want, S, what="y", Nq=Nq)
    with pytest.raises(AssertionError, match=r"^y: .*outside the bound"):
        check_ln(_sim_ln(v, g, b, eps, eps_outside=True), want, S, what="y", Nq=Nq)
    gbad = g.clone()
    gbad[148:152] = g[152:156]                         # group 37 (lane 5, step 1) reads group 38's gamma
    with pytest.raises(AssertionError, match=r"row 0 .*column 1(4[89]|5[01]) \(4-column group 37: lane 5, step 1\)"):
        check_ln(_sim_ln(v, gbad, b, eps), want, S, what="y", Nq=Nq)
    with pytest.raises(AssertionError, match=r"^y2: .*first at row 0"):
        check_ln(_sim_ln(v, g2, b2, eps), want2, S2, what="y2", Nq=Nq)


def _sim_task_tail(h, g, b, w2, b2, eps, ks, Nq, cross_frames=None):
    """fp32 task-head tail; cross_frames: row whose k = 3 left neighbour is read across the frame boundary."""
    L, M, NH, HC = h.shape
    mu = h.mean(-1, keepdim=True)
    d = h - mu
    sd = torch.sqrt((d * d).mean(-1, keepdim=True) + eps)
    y = torch.relu(d / sd * g[:, None] + b[:, None])
    out = b2[:, None].expand(L, M, NH, w2.shape[2]).clone()
    q = torch.arange(M) % Nq
    for t in range(ks):
        dq = t - ks // 2
        ok = ((q + dq >= 0) & (q + dq < Nq))
        if cross_frames is not None and dq == -1:
            ok = ok.clone()
            ok[cross_frames] = True
        yt = torch.roll(y, -dq, 1) * ok.float()[None, :, None, None]
        out += torch.einsum("lmnc,lnoc->lmno", yt, w2[:, :, :, t])
    return out


def test_task_tail_check_accepts_a_correct_kernel_and_rejects_mutants():
    gen = torch.Generator().manual_seed(6)
    L, B, Nq, NH, CMAX, ks, eps = 2, 3, 40, 3, 5, 3, 1e-6
    M = B * Nq
    h = torch.randn(L, M, NH, 64, generator=gen) * 2
    g = 1 + 0.05 * torch.randn(L, NH, 64, generator=gen)
    bb = 0.02 * torch.randn(L, NH, 64, generator=gen)
    w2 = torch.randn(L, NH, CMAX, ks, 64, generator=gen) * 0.1
    b2 = torch.randn(L, NH, CMAX, generator=gen) * 0.1
    couts = [5, 2, 3]
    want, bound = task_tail_reference(h, g, bb, w2, b2, eps, ks, Nq)

    def split(o):
        return [o[:, :, i, :c] for i, c in enumerate(couts)]
    check_task_tail(split(_sim_task_tail(h, g, bb, w2, b2, eps, ks, Nq)), want, bound, couts, what="tail", Nq=Nq)
    with pytest.raises(AssertionError, match=r"layer 0, row 80 \(frame 2, query 0\)"):
        check_task_tail(split(_sim_task_tail(h, g, bb, w2, b2, eps, ks, Nq, cross_frames=2 * Nq)), want, bound, couts,
                        what="tail", Nq=Nq)


def test_view_sum_and_query_pe_checks_accept_a_correct_kernel_and_reject_mutants():
    gen = torch.Generator().manual_seed(8)
    B, V, Nq, C = 2, 6, 50, 64
    emb = torch.randn(B, V, Nq, C, generator=gen).bfloat16()
    mask = (torch.rand(B, V, Nq, generator=gen) > 0.5).float()
    base = torch.randn(Nq, C, generator=gen)
    valid = torch.ones(V, B, dtype=torch.bool)
    valid[2, 1] = False
    want, bound = view_sum_reference(emb, mask, base, valid)
    got = view_sum_emulation(emb, mask, base, valid)
    check_view_sum(got, want, bound, what="sum")
    with pytest.raises(AssertionError, match=r"frame 1, query \d+"):       # camera 2 of frame 1 left in the sum
        check_view_sum(view_sum_emulation(emb, mask, base, None), want, bound, what="sum")
    bad = got.clone()
    bad[0, 7] = got[0, 8]
    with pytest.raises(AssertionError, match=r"frame 0, query 7, channel 0"):
        check_view_sum(bad, want, bound, what="sum")
    # query PE: a simulated fp32 kernel (the same formulas in fp32) and a query row read from its neighbour
    pc = synth.NUSC_RANGE
    rng = np.random.RandomState(2)
    l2i = torch.tensor(np.stack([synth.camera_matrices(V, rng, 1600.0, 640.0) for _ in range(B)]), dtype=torch.float32)
    i2l = torch.linalg.inv(l2i.double()).float()
    ref = torch.rand(B, Nq, 3, generator=gen)
    D = 64
    want = query_pe_reference(ref, l2i, i2l, D, 640.0, 1600.0, pc)

    def sim(refp):
        r32 = query_pe_reference(refp.double(), l2i.double(), i2l.double(), D, 640.0, 1600.0, pc)
        feat = torch.where(r32["mask"][..., None], r32["feat"], torch.zeros((), dtype=torch.float64)).bfloat16()
        return feat, r32["mask"].float()
    feat, m = sim(ref)
    check_query_pe(feat, m, want, what="qpe")
    n = int(torch.nonzero(want["mask"][1].any(0))[0])        # a query inside some view of frame 1
    bad_ref = ref.clone()
    bad_ref[1, n] = ref[1, n + 1]
    with pytest.raises(AssertionError, match=rf"frame 1, view \d, query {n}\b"):
        check_query_pe(*sim(bad_ref), want, what="qpe")


def test_untouched_check_names_the_frame():
    """A write outside a launch's slice of a shared buffer (here: into the neighbouring node's frame) is reported."""
    before = torch.zeros(4, 3, 8)
    geom = _geom(before[2:4])
    after = before.clone()
    after[3, 0, 1] = 1.0                               # inside the slice
    check_untouched(before, after, [geom], what="ctx")
    after[1, 2, 5] = 1.0                               # frame 1: the other node's
    with pytest.raises(AssertionError, match=r"ctx: 1 elements outside the launch's slice changed; first at \[1, 2, 5\]"):
        check_untouched(before, after, [geom], what="ctx")


def check_untouched(before, after, geoms, *, what):
    """Only the elements of the views `geoms` [(storage offset, shape, stride)] of the contiguous buffer may differ."""
    mask = torch.zeros(before.numel(), dtype=torch.bool, device=before.device)
    for off, shape, stride in geoms:
        mask.as_strided(shape, stride, off).fill_(True)
    ne = (_bits(before).reshape(-1) != _bits(after).reshape(-1)) & ~mask
    if bool(ne.any()):
        i = int(torch.argmax(ne.to(torch.uint8)))
        idx = [int(v) for v in np.unravel_index(i, tuple(before.shape))]
        raise AssertionError(f"{what}: {int(ne.sum())} elements outside the launch's slice changed; first at {idx}")


# ------------------------------------------------------------------------------------------
# 4. the recorder
def _clone(x):
    if isinstance(x, torch.Tensor):
        return x.clone()
    if isinstance(x, (tuple, list)):
        return type(x)(_clone(v) for v in x)
    return x


def _base(t):
    return t._base if t._base is not None else t


def _geom(t):
    return t.storage_offset() - _base(t).storage_offset(), tuple(t.shape), t.stride()


class Recorder:
    """Stands in for every kernel-launching function of ops: calls the real one and keeps clones of its operands and
    outputs (GEMM-family launches: only the launch count, test_gpu_gemm_geometry.py replays them)."""

    def __init__(self, monkeypatch):
        self.calls = []
        self.kv = {}
        self.real = {n: getattr(ops, n) for n in launching_ops()}
        for n, f in self.real.items():
            monkeypatch.setattr(ops, n, self._wrap(n, f))

    def _arg(self, op, name, v):
        if op == "cross_attn" and name in ("k", "vt"):          # the K / V^T caches of all layers: once per buffer
            key = (v.data_ptr(), tuple(v.shape), v.dtype)
            if key not in self.kv:
                self.kv[key] = v.clone()
            return self.kv[key]
        return _clone(v)

    def _wrap(self, op, real):
        sig = inspect.signature(real)

        def wrapper(*args, **kw):
            n0 = ops.launch_count()
            if op in GEMM_REPLAYED:
                r = real(*args, **kw)
                self.calls.append(dict(op=op, n=ops.launch_count() - n0))
                return r
            ba = sig.bind(*args, **kw)
            ba.apply_defaults()
            a = {k: self._arg(op, k, v) for k, v in ba.arguments.items()}
            shared = {k: ba.arguments[k] for k in ("out", "y2") if ba.arguments.get(k) is not None}
            views = {k: [v] if isinstance(v, torch.Tensor) else list(v) for k, v in shared.items()}
            before = {k: [_base(t).clone() for t in vs] for k, vs in views.items()}
            r = real(*args, **kw)
            n = ops.launch_count() - n0
            after = {k: [_base(t).clone() for t in vs] for k, vs in views.items()}
            geoms = {k: [_geom(t) for t in vs] for k, vs in views.items()}
            rgeom = [_geom(t) for t in r] if isinstance(r, list) else None      # task_head_tail's per-head views
            self.calls.append(dict(op=op, n=n, a=a, r=_clone(r), rgeom=rgeom, before=before, after=after, geoms=geoms))
            return r
        return wrapper


# ------------------------------------------------------------------------------------------
# 5. per-op replay checks: each returns (shape / dtype description, worst ratio text)
def _desc(t):
    return f"{list(t.shape)} {str(t.dtype).replace('torch.', '')}"


def replay_add_layernorm(c, ctx):
    a = c["a"]
    y, y2, ylp, yadd = c["r"]
    C = y.shape[-1]
    M = y.numel() // C
    eps = float(np.float32(a["eps"]))
    x = a["x"].reshape(1, C).expand(M, C) if a["rows"] is not None else a["x"].reshape(M, C)
    v = x if a["r"] is None else x + a["r"].reshape(M, C)          # the kernel's fp32 add
    Nq = y.shape[-2]
    rep = grid_replica("add_layernorm", a, ctx["sms"])
    st = {}
    want, S = ln_reference(v, a["gamma"], a["beta"], eps)
    check_ln(y.reshape(M, C), want, S, what="add_layernorm y", Nq=Nq, grid_rows=rep[1], stats=st, key="y")
    if y2 is not None:
        w2, S2 = ln_reference(y.reshape(M, C), a["gamma2"], a["beta2"], eps)
        check_ln(y2.reshape(M, C), w2, S2, what="add_layernorm y2", Nq=Nq, grid_rows=rep[1], stats=st, key="y2")
        check_untouched(c["before"]["y2"][0], c["after"]["y2"][0], c["geoms"]["y2"], what="add_layernorm y2 buffer")
    lp = a["lp_dtype"] or torch.float32
    if ylp is not None:
        same_bits(ylp, y.to(lp), "add_layernorm ylp")
    if yadd is not None:
        same_bits(yadd, (y + a["add"]).to(lp), "add_layernorm yadd")
    form = "row-broadcast " if a["rows"] is not None else ""
    return f"{form}{_desc(y)}{' +y2' if y2 is not None else ''} lp={str(lp).replace('torch.', '')}", \
        " ".join(f"{k} {v:.3f}" for k, v in st.items())


def replay_cross_attn(c, ctx):
    a = c["a"]
    o = c["r"][0] if isinstance(c["r"], tuple) else c["r"]
    q, k, vt, layer = a["q"], a["k"], a["vt"], a["layer"]
    B, Nq, HD = q.shape
    N_kv = k.shape[3]
    lo, hi = a["kv_begin"], N_kv if a["kv_end"] is None else a["kv_end"]
    dt = q.dtype
    tc = dt != torch.float32
    qn, kn = a["q_norm2"], a["k_norm2"]
    use_norms = qn is not None and kn is not None and tc
    o32, lse = ctx["cross_attn"](q, k, vt, layer, kv_begin=lo, kv_end=hi, o_dtype=torch.float32, return_lse=True,
                                 simt=a["simt"], key_keep=a["key_keep"], q_norm2=qn if use_norms else None,
                                 k_norm2=kn if use_norms else None)
    same_bits(o, o32.to(o.dtype), f"cross_attn ({a['tag']}) recorded output vs the fp32 re-launch")
    if "out" in c["geoms"]:
        check_untouched(c["before"]["out"][0], c["after"]["out"][0], c["geoms"]["out"], what="cross_attn out= buffer")
    f0 = c["geoms"]["out"][0][0] // (Nq * HD) if "out" in c["geoms"] else 0
    n_keys = hi - lo
    st = {}
    for b in range(B):
        keep = None if a["key_keep"] is None else a["key_keep"][b, lo:hi].bool()
        static = False
        if use_norms:
            bound = (qn[b].double() * kn[b, layer].double()).sqrt() * 1.0079 + 1e-3
            static = bool((bound <= STATIC_LIMIT[dt]).all())
        plan = Plan(B, Nq, n_keys, ctx["sms"], static) if tc else None
        qb = q[b].view(Nq, H, 32).transpose(0, 1)
        for h0 in range(0, H, 4):
            hs = slice(h0, h0 + 4)
            ref = attn_reference(qb[hs], k[b, layer, hs, lo:hi], vt[b, layer, hs, :, lo:hi].transpose(1, 2), keep)
            got = o[b].view(Nq, H, 32).transpose(0, 1)[hs]
            where = plan_where(plan, b, static)
            check_attention(got, lse[b, hs], ref, dt, n_keys, what=f"cross_attn ({a['tag']}) layer {layer}",
                            frame=f0 + b, head0=h0, where=where, stats=st)
            del ref
    ctx["stats"].setdefault("attn", {})
    for key, v in st.items():
        ctx["stats"]["attn"][key] = max(ctx["stats"]["attn"].get(key, 0.0), v)
    mask = "masked " if a["key_keep"] is not None else ""
    slice_ = f" out=ctx[{f0}:{f0 + B}]" if "out" in c["geoms"] else ""
    return (f"{a['tag']} layer {layer} {mask}q {_desc(q)} keys {n_keys}{slice_}"
            f"{' static-shift' if use_norms else ''}", f"o {st.get('o', 0):.3f} lse {st.get('lse', 0):.3f}")


def replay_ray_pe(c, ctx):
    a = c["a"]
    out = c["r"]
    M = a["img2lidar"].double()
    n_cam, Hh, W, F = out.shape
    D = a["depth_num"]
    pc = a["pc_range"]
    f32 = lambda x: float(np.float32(x))   # noqa: E731
    dev = out.device
    u = torch.arange(W, device=dev, dtype=torch.float64) * float(a["pad_w"]) / W
    vv = torch.arange(Hh, device=dev, dtype=torch.float64) * float(a["pad_h"]) / Hh
    d = 1.0 + torch.arange(D, device=dev, dtype=torch.float64) * f32(f32(pc[3]) - 1.0) / D
    st = {}
    for c3 in range(3):
        pmin, rng = f32(pc[c3]), f32(f32(pc[c3 + 3]) - f32(pc[c3]))
        Mc = M[:, c3]                                                       # [n_cam, 4]
        t0 = u[None, None, :, None] * d * Mc[:, 0, None, None, None]        # [n_cam, 1, W, D]
        t1 = vv[None, :, None, None] * d * Mc[:, 1, None, None, None]       # [n_cam, H, 1, D]
        t2 = (d * Mc[:, 2, None])[:, None, None, :]
        t3 = Mc[:, 3, None, None, None]
        want = ((t0 + t1 + t2 + t3) - pmin) / rng
        T = (t0.abs() + t1.abs() + t2.abs() + t3.abs() + abs(pmin)) / abs(rng)
        got = out[..., c3::3].double()
        err = (got - want).abs()
        bound = C_PE * U * T + U_OUT[out.dtype] * want.abs()
        bad = ~(err <= bound)
        if bool(bad.any()):
            cam, i, j, kk = _first(bad)
            raise AssertionError(f"ray_pe: {int(bad.sum())} features of coordinate {c3} outside the bound; first at camera "
                                 f"{cam}, row {i}, column {j}, depth bin {kk}: got {float(got[cam, i, j, kk])!r} want "
                                 f"{float(want[cam, i, j, kk])!r} (block {cam * Hh + i})")
        st["pe"] = max(st.get("pe", 0.0), _ulp_ratio(err - U_OUT[out.dtype] * want.abs(), U * T))
    if out.dtype == torch.float16:
        assert bool(torch.isfinite(out).all())
    return _desc(out), f"pe {st['pe']:.3f}"


def replay_ray_query_pe(c, ctx):
    a = c["a"]
    feat, mask = c["r"]
    ref = query_pe_reference(a["ref"], a["lidar2img"], a["img2lidar"], a["depth_num"], float(a["pad_h"]),
                             float(a["pad_w"]), a["pc_range"])
    st = {}
    n_flip, n_amb = check_query_pe(feat, mask, ref, what="ray_query_pe", stats=st)
    assert n_amb <= max(16, mask.numel() // 1000), f"ray_query_pe: {n_amb} ambiguous points"
    return (f"{_desc(feat)} mask {list(mask.shape)}; {n_amb} ambiguous points, {n_flip} decided the other way",
            f"pe {st['qpe']:.3f}")


def replay_masked_view_sum(c, ctx):
    a = c["a"]
    out = c["r"]
    vv = a["view_valid"]
    same_bits(out, view_sum_emulation(a["emb"], a["mask"], a["base"], vv), "masked_view_sum vs its fp32 order")
    want, bound = view_sum_reference(a["emb"], a["mask"], a["base"], vv)
    st = {}
    check_view_sum(out, want, bound, what="masked_view_sum", stats=st)
    return f"emb {_desc(a['emb'])}{' +base' if a['base'] is not None else ''}{' view_valid' if vv is not None else ''}", \
        f"exact; fp64 {st['sum']:.3f}"


def replay_pos2embed(c, ctx):
    a = c["a"]
    out = c["r"]
    F = a["num_pos_feats"]
    pos = a["pos"].reshape(-1, a["pos"].shape[-1]).double()
    m = torch.arange(2 * F, device=out.device) % F
    is_x = torch.arange(2 * F, device=out.device) >= F
    pv = torch.where(is_x, pos[:, 0:1], pos[:, 1:2]) * (2 * math.pi)
    dim_t = 2.0 * (m // 2).double() / F + 1.0
    ang = pv / dim_t
    want = torch.where(m % 2 == 1, torch.cos(ang), torch.sin(ang))
    got = out.reshape(-1, 2 * F).double()
    err = (got - want).abs()
    bound = C_POS * U * (ang.abs() + 1) + U_OUT[out.dtype] * want.abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        n, f = _first(bad)
        raise AssertionError(f"pos2embed: {int(bad.sum())} of {bad.numel()} outside the bound; first at token {n}, "
                             f"feature {f}: got {float(got[n, f])!r} want {float(want[n, f])!r}")
    ratio = _ulp_ratio(err - U_OUT[out.dtype] * want.abs(), U * (ang.abs() + 1))
    return _desc(out), f"pe {ratio:.3f}"


def replay_gather_tokens(c, ctx):
    a = c["a"]
    xk, xv = c["r"]
    B, V, lp = a["B"], a["V"], a["out_dtype"]
    sv = a["sensor_valid"]
    n_bev = a["x_bev"].shape[2] * a["x_bev"].shape[3] if a["x_bev"] is not None else a["n_bev_reserved"]
    lo, hi = a["tok_range"] if a["tok_range"] is not None else (0, xk.shape[1])
    assert (lo, hi) == (0, xk.shape[1]) and a["rv_rows"] is None
    ks, vs = [], []
    zero = torch.zeros((), device=xk.device)

    def part(feat, pos, present):
        k_ = torch.where(present[:, None, None], feat + pos, zero)
        v_ = torch.where(present[:, None, None], feat, zero)
        ks.append(k_.to(lp))
        vs.append(v_.to(lp))
    ones = torch.ones(B, dtype=torch.bool, device=xk.device)
    row = 0
    if a["x_bev"] is not None:
        C = a["x_bev"].shape[1]
        part(a["x_bev"].float().reshape(B, C, n_bev).transpose(1, 2), a["bev_pos"].reshape(1, n_bev, C),
             ones if sv is None else sv[0])
        row = 1
    elif n_bev:
        row = 1
    if a["x_img"] is not None:
        C = a["x_img"].shape[1]
        n_img = a["x_img"].shape[2] * a["x_img"].shape[3]
        f = a["x_img"].float().reshape(B, V, C, n_img).transpose(2, 3)
        p = a["rv_pos"].reshape(B, V, n_img, C)
        for v in range(V):
            part(f[:, v], p[:, v], ones if sv is None else sv[row + v])
    k_want, v_want = torch.cat(ks, 1), torch.cat(vs, 1)
    first = 0 if a["x_bev"] is not None else n_bev          # rows this launch writes
    same_bits(xk[:, first:], k_want, "gather_tokens xk")
    same_bits(xv[:, first:], v_want, "gather_tokens xv")
    if a["out"] is not None:
        C = xk.shape[2]
        geom = [(first * C, (B, xk.shape[1] - first, C), (xk.shape[1] * C, C, 1))]
        for i, name in enumerate(("xk", "xv")):
            check_untouched(c["before"]["out"][i], c["after"]["out"][i], geom, what=f"gather_tokens {name} (reserved BEV rows)")
    tiles = -(-n_bev // 32) if a["x_bev"] is not None else 0
    if a["x_img"] is not None:
        tiles += V * -(-(a["x_img"].shape[2] * a["x_img"].shape[3]) // 32)
    return (f"xk {_desc(xk)} rows [{first}, {xk.shape[1]}){' sensor_valid' if sv is not None else ''}; "
            f"grid ({tiles}, {B}), one block per 32-token tile"), "exact"


def replay_nchw(c, ctx):
    a = c["a"]
    out = c["r"]
    x = a["x"]
    B, C, Hh, W = x.shape
    guard = ops.conv_guard_rows(W)
    want = torch.zeros_like(out)
    inner = want[:, guard:guard + (Hh + 2) * (W + 2)].view(B, Hh + 2, W + 2, C)
    vals = x.permute(0, 2, 3, 1).to(out.dtype)
    if a["frame_valid"] is not None:
        vals = torch.where(a["frame_valid"].reshape(B, 1, 1, 1), vals, torch.zeros((), dtype=vals.dtype, device=vals.device))
    inner[:, 1:Hh + 1, 1:W + 1] = vals
    same_bits(out, want, "nchw_to_padded_nhwc (guard and border rows zero)")
    return f"x {_desc(x)} -> {_desc(out)}", "exact"


def replay_sensor_key_keep(c, ctx):
    a = c["a"]
    keep = c["r"]
    sv = a["sensor_valid"]
    rows = ([torch.zeros(a["n_bev"], dtype=torch.long)] if a["n_bev"] else []) + \
        [torch.full((a["n_img"],), (1 if a["n_bev"] else 0) + v, dtype=torch.long) for v in range(a["V"])]
    want = sv[torch.cat(rows).to(sv.device)].t().contiguous()
    same_bits(keep, want, "sensor_key_keep")
    return _desc(keep), "exact"


def replay_split3(c, ctx):
    a = c["a"]
    r = c["r"]
    out, merged = r if isinstance(r, tuple) else (r, None)
    x = a["a"]
    L, B, Nq, C = x.shape
    if a["stacked_nodes"]:
        B //= 2
        A, Bn = x[:, :B], x[:, B:]
    else:
        A, Bn = x, a["b"]
    va = torch.nan_to_num(A)
    if Bn is None:
        v = va
    else:
        vb = torch.nan_to_num(Bn)
        nv = a["node_valid"]
        if nv is None:
            v = torch.maximum(va, vb)
        else:
            ha, hb = nv[0].view(1, B, 1, 1), nv[1].view(1, B, 1, 1)
            v = torch.where(ha & hb, torch.maximum(va, vb), torch.where(ha, va, torch.where(hb, vb, torch.zeros_like(va))))
    t1 = v.bfloat16()
    big = torch.tensor(torch.finfo(torch.bfloat16).max, dtype=torch.bfloat16, device=v.device)
    t1 = torch.where(torch.isinf(t1), torch.copysign(big, t1), t1)
    r1 = v - t1.float()
    t2 = r1.bfloat16()
    t3 = (r1 - t2.float()).bfloat16()
    want = torch.zeros(L * B, Nq + 2, 3 * C, dtype=torch.bfloat16, device=v.device)
    want[:, 1:Nq + 1] = torch.cat([t1, t2, t3], -1).reshape(L * B, Nq, 3 * C)
    same_bits(out, want, "split3")
    if merged is not None:
        same_bits(merged, v, "split3 merged")
    form = "stacked nodes" if a["stacked_nodes"] else ("two stacks" if a["b"] is not None else "one stack")
    return f"{_desc(x)} {form}{' node_valid' if a['node_valid'] is not None else ''} -> {_desc(out)}", "exact"


def replay_task_head_tail(c, ctx):
    a = c["a"]
    outs = c["r"]
    h = a["h"]
    w2 = a["w2"] if a["w2"].dim() == 5 else a["w2"].unsqueeze(3)
    L, M, NH, _ = h.shape
    Nq = M if a["Nq"] is None else a["Nq"]
    want, bound = task_tail_reference(h, a["gamma"], a["beta"], w2, a["b2"], float(np.float32(a["eps"])), a["ksize"], Nq,
                                      a["ref_logit"], a["dec_comp"], a["dec_scale"], a["dec_offset"])
    couts = a["head_couts"]
    assert couts is not None, "the forward uses the packed per-head output"
    # packed: one buffer, head i at the sum of the previous heads' sizes
    starts = np.cumsum([0] + [L * M * co for co in couts])[:-1]
    assert [g[0] for g in c["rgeom"]] == [int(s) for s in starts] and all(g[2] == (M * co, co, 1) for g, co in
                                                                           zip(c["rgeom"], couts))
    st = {}
    check_task_tail(outs, want, bound, couts, what=f"task_head_tail k={a['ksize']}", Nq=Nq, stats=st)
    return f"h {_desc(h)} k={a['ksize']} couts {list(couts)}{' +decode' if a['ref_logit'] is not None else ''}", \
        f"th {st['th']:.3f}"


REPLAY = {"add_layernorm": replay_add_layernorm, "cross_attn": replay_cross_attn, "ray_pe": replay_ray_pe,
          "ray_query_pe": replay_ray_query_pe, "masked_view_sum": replay_masked_view_sum, "pos2embed": replay_pos2embed,
          "gather_tokens": replay_gather_tokens, "nchw_to_padded_nhwc": replay_nchw,
          "sensor_key_keep": replay_sensor_key_keep, "split3": replay_split3, "task_head_tail": replay_task_head_tail}
assert set(REPLAY) == CHECKED


# ------------------------------------------------------------------------------------------
# 6. the replay
WORKLOADS = {"nusc": ("CmtHead", 6), "coop_lidar": ("CmtLidarHeadCoop", 0)}
_inputs = {}


def _workload_inputs(kind, n_views):
    if kind not in _inputs:
        _inputs.clear()
        _inputs[kind] = synth.make_inputs(kind, B=8, bev_hw=180, n_views=max(n_views, 1), img_hw=(40, 100),
                                          in_channels=512, seed=0)
    return _inputs[kind]


def _sensor_mask(d, B, V):
    """Frame 1 without its LiDAR, frame 3 without cameras 2 and 4, frame 5 without any sensor; the absent sensors'
    features are NaN (they must not reach any output)."""
    sv = torch.ones(1 + V, B, dtype=torch.bool)
    sv[0, 1] = False
    sv[[3, 5], 3] = False
    sv[:, 5] = False
    pts, img = d["pts_feats"].clone(), d["img_feats"].clone()
    pts[~sv[0].to(pts.device)] = float("nan")
    img.view(B, V, *img.shape[1:])[~sv[1:].t().to(img.device)] = float("nan")
    return sv.to(DEV), pts, img


CASES = [pytest.param(w, p, False, id=f"{w}-{p}") for w in WORKLOADS for p in ("bf16", "fp16", "fp32")] + \
    [pytest.param("nusc", p, True, id=f"nusc-{p}-sensor-mask") for p in ("bf16", "fp16")]
_stats = {}


@pytest.mark.gpu
@pytest.mark.parametrize("workload,precision,masked", CASES)
def test_forward_launches(workload, precision, masked, monkeypatch):
    """Every launch of one eager forward_single of a freshly built head (B = 8, shared_conv included), each checked
    against fp64 (or bit for bit) on its own recorded operands."""
    from cmtcoop_b200.plugin import build_head
    t0 = time.time()
    kind, n_views = WORKLOADS[workload]
    cfg = synth.head_cfg(kind, num_query=900, num_layers=6, grid=8 * 180)
    inputs = _workload_inputs(kind, n_views)
    head = build_head(cfg)
    synth.load_synth_weights(head, 0)
    head = head.to(DEV).eval().set_precision(precision)
    head.apply_shared_conv = True
    d = {k: (torch.from_numpy(v).to(DEV) if isinstance(v, np.ndarray) else v) for k, v in inputs.items()}
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ctx = dict(sms=sms, cross_attn=ops.cross_attn, stats=_stats.setdefault(precision, {}))
    rec = Recorder(monkeypatch)
    n0 = ops.launch_count()
    with torch.no_grad():
        if kind.endswith("Coop"):
            head.forward_single(d["vehicle_pts_feats"], d["infrastructure_pts_feats"], d["vehicle_img_feats"],
                                d["infrastructure_img_feats"], d["img_metas"])
        elif masked:
            sv, pts, img = _sensor_mask(d, 8, n_views)
            head.forward_single(pts, img, d["img_metas"], sensor_valid=sv)
        else:
            head.forward_single(d["pts_feats"], d["img_feats"], d["img_metas"])
    total = ops.launch_count() - n0
    monkeypatch.undo()
    del head, d
    t_fwd = time.time() - t0
    # accounting: the recorded calls add up to the forward, and every op is checked somewhere or excluded
    ops_seen = [c["op"] for c in rec.calls]
    n_here = sum(c["n"] for c in rec.calls if c["op"] in CHECKED)
    n_gemm = sum(c["n"] for c in rec.calls if c["op"] in GEMM_REPLAYED)
    n_excl = sum(c["n"] for c in rec.calls if c["op"] in EXCLUDED)
    unknown = set(ops_seen) - CHECKED - GEMM_REPLAYED - set(EXCLUDED)
    assert not unknown, f"ops launched by the forward without a check or an exclusion: {unknown}"
    label = f"{workload} {precision}{' sensor-mask' if masked else ''}"
    print(f"\n{label}: {len(rec.calls)} recorded calls")
    wrapped = {}
    rec.kv.clear()
    while rec.calls:
        c = rec.calls.pop(0)
        if c["op"] not in CHECKED:
            continue
        desc, ratio = REPLAY[c["op"]](c, ctx)
        w = wraps(c["op"], c["a"], sms)
        wrapped.setdefault(c["op"], []).append(w)
        print(f"  {c['op']:<20} {desc}; wraps {'-' if w is None else ('yes' if w else 'no')}; worst {ratio}")
        del c
    torch.cuda.empty_cache()
    print(f"  accounting: {n_here} checked here + {n_gemm} GEMM-replay + {n_excl} excluded = {total} launches "
          f"(launch_count delta); forward {t_fwd:.1f} s, replay {time.time() - t0 - t_fwd:.1f} s")
    assert n_here + n_gemm + n_excl == total
    # the grid-stride families reach a second pass of their loop in at least one launch
    must_wrap = {"split3", "pos2embed"} | ({"ray_query_pe", "masked_view_sum"} if workload == "nusc" else {"add_layernorm"})
    if sms == B200_SMS:
        for op in must_wrap:
            assert any(wrapped.get(op, [])), f"{op}: no recorded launch wraps its grid"
    assert all(w is None for w in wrapped.get("gather_tokens", [])) and all(w is None for w in wrapped["cross_attn"])
    want_ops = {"add_layernorm", "cross_attn", "pos2embed", "split3", "task_head_tail"}
    if workload == "nusc":
        want_ops |= {"ray_pe", "ray_query_pe", "masked_view_sum", "gather_tokens"}
    if precision != "fp32":
        want_ops |= {"nchw_to_padded_nhwc"}
    else:
        want_ops |= {"gather_tokens"}
    if masked:
        want_ops |= {"sensor_key_keep"}
    assert want_ops <= set(wrapped), want_ops - set(wrapped)
