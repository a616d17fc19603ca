"""Debug: clock64 event trace of CTA 0 of the attention kernel at the nuScenes shape.
Needs a trace build of the library: make -C cmt-cooperative-perception_b200/csrc clean all EXTRA=-DCMT_ATTN_TRACE
(or tools/build_variant.sh + tools/ab_trace.sh).  Slots per (warpgroup, step): 0 S ready, 1 S in registers, 2 row max done,
3/8/9/10 P stored by warps 0..3; issuer: 6 loop top, 7 K/V stages seen, 11 before the P wait, 4 P seen, 5 PV + next S issued."""
import ctypes, os, sys, statistics, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cmtcoop_b200 import ops, _lib
lib = _lib.load()
dev = "cuda:0"
B, N_kv, L, H, Nq = 8, 56400, 1, 8, (int(sys.argv[3]) if len(sys.argv) > 3 else 900)
STEPS, SL = 96, 16
q = (torch.randn(B, Nq, 256, device=dev) * 0.25).bfloat16()
k = torch.randn(B, L, H, N_kv, 32, device=dev).bfloat16()
vt = torch.randn(B, L, H, 32, N_kv, device=dev).bfloat16()
STATIC = len(sys.argv) > 4 and sys.argv[4] == "static"
kw = {}
if STATIC:   # operand norms -> static softmax shift kernel
    kw = dict(q_norm2=q.float().view(B, Nq, H, 32).pow(2).sum(-1).amax(1).contiguous(),
              k_norm2=k.float().pow(2).sum(-1).amax(-1).contiguous())
ops.cross_attn(q, k, vt, 0, **kw); torch.cuda.synchronize()
buf = torch.zeros(3 * STEPS * SL + 148, dtype=torch.int64, device=dev)
lib.cmt_debug_attn_timing.argtypes = [ctypes.c_void_p]
lib.cmt_debug_attn_timing(ctypes.c_void_p(buf.data_ptr()))
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(); ops.cross_attn(q, k, vt, 0, **kw); e1.record(); torch.cuda.synchronize()
lib.cmt_debug_attn_timing(ctypes.c_void_p(0))
cyc = buf[3 * STEPS * SL:].cpu().tolist()
us = e0.elapsed_time(e1) * 1e3
print(f"kernel+merge {us:.0f} us; per-CTA cycles min {min(cyc)} median {sorted(cyc)[74]} max {max(cyc)} -> SM clock >= {max(cyc) / us / 1e3:.2f} GHz")
t = buf[:3 * STEPS * SL].cpu().view(3, STEPS, SL)
t0 = int(t[0, 0, 0])
lo, hi = int(sys.argv[1]) if len(sys.argv) > 1 else 40, int(sys.argv[2]) if len(sys.argv) > 2 else 56
print("step wg |  S_ready | +ld +max +exp(w0) | P_stored w0..w3 (rel. S_ready) | issuer rel. last P: top kv pwait seen issued | next S_ready - issued | period")
def rel(x, base): return int(x) - int(base) if int(x) else -1
for st in range(lo, hi):
    for wg in range(3):
        e = t[wg, st]
        s0 = int(e[0])
        pl = max(int(e[3]), int(e[8]), int(e[9]), int(e[10]))
        nxt = int(t[wg, st + 2, 0]) if st + 2 < STEPS else 0
        print(f"{st:4d} {wg:2d} | {s0 - t0:8d} | {rel(e[1], s0):4d} {rel(e[2], e[1]):4d} {rel(e[3], e[2]):5d} | "
              f"{rel(e[3], s0):5d} {rel(e[8], s0):5d} {rel(e[9], s0):5d} {rel(e[10], s0):5d} | "
              f"{rel(e[6], pl):5d} {rel(e[7], pl):5d} {rel(e[11], pl):5d} {rel(e[4], pl):5d} {rel(e[5], pl):5d} | {rel(nxt, e[5]):5d} | "
              f"{s0 - int(t[wg, st - 1, 0]):5d}")
for wg in range(3):
    rng = range(20, STEPS - 2)
    med = lambda f: statistics.median(f(s) for s in rng)
    pl = lambda s: max(int(t[wg, s, 3]), int(t[wg, s, 8]), int(t[wg, s, 9]), int(t[wg, s, 10]))
    print(f"wg{wg}: period {med(lambda s: int(t[wg, s, 0] - t[wg, s - 1, 0]))}, max {med(lambda s: int(t[wg, s, 2] - t[wg, s, 1]))}, "
          f"exps(w0) {med(lambda s: int(t[wg, s, 3] - t[wg, s, 2]))}, "
          f"warp skew of P {med(lambda s: pl(s) - min(int(t[wg, s, 3]), int(t[wg, s, 8]), int(t[wg, s, 9]), int(t[wg, s, 10])))}, "
          f"last P -> issuer saw it {med(lambda s: int(t[wg, s, 4]) - pl(s))}, issue {med(lambda s: int(t[wg, s, 5] - t[wg, s, 4]))}, "
          f"issued -> S(g+2) ready {med(lambda s: int(t[wg, s + 2, 0] - t[wg, s, 5]))}, "
          f"w0: P stored -> next S ready {med(lambda s: int(t[wg, s + 1, 0] - t[wg, s, 3]))}")
