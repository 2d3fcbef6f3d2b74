import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from a2f_b200 import ops, lib as L
dev = torch.device("cuda:0")
lib = L.load()
g = torch.Generator().manual_seed(0)
def run(M, N, K, resid=False):
    a = torch.randn(M, K, generator=g).to(dev).bfloat16()
    w = (torch.randn(N, K, generator=g) * K ** -0.5).to(dev).bfloat16()
    b = torch.randn(N, generator=g).to(dev)
    r = torch.randn(M, N, generator=g).to(dev).bfloat16() if resid else None
    out = torch.empty((M, N), device=dev, dtype=torch.bfloat16)
    tl = torch.zeros(2 * 148 * 8, dtype=torch.int64, device=dev)
    for _ in range(3):
        ops.gemm(a, w, out, bias=b, resid=r, backend=L.TCGEN05)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(10):
        ops.gemm(a, w, out, bias=b, resid=r, backend=L.TCGEN05)
    e.record(); torch.cuda.synchronize()
    print(f"M{M} N{N} K{K} resid={resid}: {s.elapsed_time(e)*100:.1f} us/launch (10 back-to-back), {2*M*N*K/(s.elapsed_time(e)*1e-4)/1e12*1e-6*1e6:.0f} TFLOP/s")
    lib.a2f_debug_set_timeline(tl.data_ptr())
    ops.gemm(a, w, out, bias=b, resid=r, backend=L.TCGEN05)
    torch.cuda.synchronize()
    lib.a2f_debug_set_timeline(None)
    tall = tl.view(2 * 148, 8).cpu()
    ncta = int((tall[:, 0] > 0).sum()) // 2
    t = tall[:ncta]
    cyc = tall[ncta:2 * ncta]
    lead = t[:, 2] > 0
    dc = (cyc[lead][:, 3] - cyc[lead][:, 2]).float()
    dt = (t[lead][:, 3] - t[lead][:, 2]).float()
    kbs = K // 64
    print(f"   mainloop tile0: {float(dc.median()):.0f} cycles = {float(dc.median())/kbs:.0f} cyc/k-block; {float(dt.median())/1000:.2f} us -> SM clock {float(dc.median())/float(dt.median())*1000:.0f} MHz")
    used = t[:, 2] > 0
    t = t[used]
    t0 = t[:, 0].min()
    rel = (t - t0).float() / 1000.0
    names = ["entry", "setup", "1st-landed", "tile0-issued", "acc0-done", "epi0-issued", "all-epi", "drained"]
    print("   ctas", ncta, " | ".join(f"{n} {float(rel[:, i].median()):.2f}/{float(rel[:, i].max()):.2f}" for i, n in enumerate(names)), "(median/max us)")
for shp in [(4800, 768, 768, True), (4800, 768, 3072, True), (4800, 2304, 768, False), (4800, 3072, 768, False), (131072, 512, 1536, False)]:
    run(*shp)
