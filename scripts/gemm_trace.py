"""Role timelines of CTA 0 of the tcgen05 GEMM (debug): TM, TN, TK, TCFG (bn | cg2<<12 like gemm_sweep), TRESID env."""
import ctypes, os, sys, math
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import seqdiff_b200 as sd
lib = sd.lib(); dev = "cuda:0"
M, N, K = int(os.environ.get("TM", 8192)), int(os.environ.get("TN", 768)), int(os.environ.get("TK", 768))
cfg = int(os.environ.get("TCFG", 192)); cg2, bn = cfg // 1000, cfg % 1000
resid = int(os.environ.get("TRESID", 0))
p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
A = torch.randn(M, K, device=dev).bfloat16(); W = (torch.randn(N, K, device=dev) / math.sqrt(K)).bfloat16()
bias = torch.randn(N, device=dev); R = torch.randn(M, N, device=dev) if resid else None
C = torch.empty(M, N, device=dev, dtype=torch.float32 if resid else torch.bfloat16)
def call():
    rc = lib.seqdiff_op_gemm(1 | (bn << 8) | (cg2 << 20), M, N, K, p(A), p(W), p(bias), p(R), 0, p(C), stream)
    assert rc == 0, lib.seqdiff_last_error()
for _ in range(3): call()
buf = torch.zeros(4 * 1024, dtype=torch.int64, device=dev)
lib.seqdiff_debug_attn_trace(p(buf)); call(); torch.cuda.synchronize(); lib.seqdiff_debug_attn_trace(None)
t = buf.cpu().tolist()
names = {40: "kernel entry", 41: "prologue done", 42: "pdl_wait done", 43: "role done", 1: "tma slot free", 11: "mma stage full", 12: "mma tile committed",
         20: "epi wait acc", 21: "epi acc ready", 23: "epi tile stored"}
ev = []
for role in range(4):
    n = t[role * 1024]
    for x in t[role * 1024 + 1: role * 1024 + 1 + n]:
        ev.append((x >> 8, role, x & 255))
ev.sort(); t0 = ev[0][0]; last = {}
print(f"M={M} N={N} K={K} cfg={cfg} resid={resid}")
for c, role, e in ev[:int(os.environ.get("TLIM", 200))]:
    d = c - last.get(role, c); last[role] = c
    print(f"{c - t0:8d}  {'   ' * role * 5}r{role} {names.get(e, e)} (+{d})")
