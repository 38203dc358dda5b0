"""Per-shape timing of the 16-bit attention core (the pipelined tcgen05 kernel) through the C ABI."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import seqdiff_b200 as sd
lib = sd.lib(); dev = "cuda:0"
heads, H = 12, 768
# (name, launches per forward, B, Lq, Lk, P, rel)
SHAPES = [("cfg2 se_lig self (lig|rec stacked)", 1, 128, 128, 128, 128, True), ("cfg2 dec/se_dec self", 7, 64, 128, 128, 128, True),
          ("cfg2 dec cross", 6, 64, 128, 128, 128, False), ("cfg3/8gpu self", 7, 32, 512, 512, 512, True),
          ("cfg3/8gpu cross", 6, 32, 512, 512, 512, False)]
if os.environ.get("ATTN_SHAPES"):
    SHAPES = [SHAPES[int(i)] for i in os.environ["ATTN_SHAPES"].split(",")]
p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
tot = 0.0
for name, cnt, B, Lq, Lk, P, rel in SHAPES:
    qkv = torch.randn(B * Lq, 3 * H, device=dev).bfloat16()
    E = (torch.randn(2 * P - 1, 64, device=dev) * 0.5).bfloat16() if rel else None
    if os.environ.get("ATTN_RAGGED"):  # cfg-2-like ragged pockets: peptide 5..64 residues (self), pocket 16..128 (cross), scaled with L
        g = torch.Generator().manual_seed(3)
        lo, hi = ((5, 64) if "self" in name and "stacked" not in name else (16, 128))
        n = torch.randint(lo * Lk // 128, hi * Lk // 128 + 1, (B,), generator=g)
        mask = (torch.arange(Lk)[None, :] < n[:, None]).float().to(dev)
    else:
        mask = torch.ones(B, Lk, device=dev)
    out = torch.empty(B * Lq, H, device=dev, dtype=torch.bfloat16)
    def call():
        rc = lib.seqdiff_op_attention(1, B, heads, Lq, Lk, p(qkv), 3 * H, p(qkv[:, H:]), 3 * H, p(qkv[:, 2 * H:]), 3 * H, p(E), P, p(mask), p(out), stream)
        assert rc == 0, lib.seqdiff_last_error()
    for _ in range(3): call()
    torch.cuda.synchronize()
    ts = []
    for _ in range(10):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); call(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    gr = torch.cuda.CUDAGraph()  # device time per launch: 20 launches captured in a graph (eager launches are CPU-bound)
    with torch.cuda.graph(gr):
        st2 = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        for _ in range(20):
            rc = lib.seqdiff_op_attention(1, B, heads, Lq, Lk, p(qkv), 3 * H, p(qkv[:, H:]), 3 * H, p(qkv[:, 2 * H:]), 3 * H, p(E), P, p(mask), p(out), st2)
            assert rc == 0, lib.seqdiff_last_error()
    gr.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); gr.replay(); e1.record(); torch.cuda.synchronize()
    warm = e0.elapsed_time(e1) / 20 * 1e3
    fl = B * heads * (4.0 + (4.0 if rel else 0.0)) * Lq * Lk * 64
    cold = sorted(ts)[len(ts) // 2]
    tot += cnt * warm if Lq == 128 else 0
    print(f"{name:36s} x{cnt} B={B:4d} L={Lq:4d} rel={int(rel)}  cold {cold:7.1f} us  graph x20 {warm:7.1f} us  {fl / warm / 1e6:7.1f} TF/s")
print(f"cfg2 attention per forward (graph x20): {tot/1e3:.3f} ms")
