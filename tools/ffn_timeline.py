"""In-kernel timeline of a2f_encoder_block at the bench shape (M=4800, d=768, ff=3072, all four phases): stamps of the
leader CTAs, and launch-to-launch gaps of four back-to-back launches (globaltimer).
    python tools/ffn_timeline.py [ffn]        ("ffn": only the feed-forward phases, no att / wq)
Slots: 0 entry, 1 setup done (barriers, TMEM, cluster sync, griddepcontrol.wait), 2 first operands landed, 3 MMAs of phase 0
issued, 4 MMAs of the last phase-1 tile issued, 5 MMAs of phase 2 issued, 6 MMAs of the last phase-3 tile issued, 7 h1
published, 8..11 phase-1 tile t stored and published, 12 epilogue enters the second LayerNorm tile, 13 its stores issued,
14 all stores drained, 15 after the final cluster sync."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from a2f_b200 import ops, lib as L

only_ffn = len(sys.argv) > 1 and sys.argv[1] == "ffn"
dev = torch.device("cuda:0")
M, N, F, NQ = 4800, 768, 3072, 2304
g = torch.Generator().manual_seed(1)
rnd = lambda *sh, s=1.0: (torch.randn(*sh, generator=g) * s)
att, h_in = rnd(M, N).bfloat16().to(dev), rnd(M, N).bfloat16().to(dev)
wo, w1 = rnd(N, N, s=N ** -0.5).bfloat16().to(dev), rnd(F, N, s=N ** -0.5).bfloat16().to(dev)
w2, wq = rnd(N, F, s=F ** -0.5).bfloat16().to(dev), rnd(NQ, N, s=N ** -0.5).bfloat16().to(dev)
bo, b1, b2, bq = rnd(N).to(dev), rnd(F).to(dev), rnd(N).to(dev), rnd(NQ).to(dev)
g1, be1, g2, be2 = torch.rand(N, generator=g).to(dev), rnd(N).to(dev), torch.rand(N, generator=g).to(dev), rnd(N).to(dev)
bf = lambda *sh: torch.empty(sh, dtype=torch.bfloat16, device=dev)
h1, f, ho, q = (h_in.clone() if only_ffn else bf(M, N)), bf(M, F), bf(M, N), bf(M, NQ)


def run():
    if only_ffn:
        ops.encoder_block(h1, w1, b1, w2, b2, g2, be2, f, ho)
    else:
        ops.encoder_block(h1, w1, b1, w2, b2, g2, be2, f, ho, att=att, wo=wo, bo=bo, h_in=h_in, ln1_g=g1, ln1_b=be1,
                          wq=wq, bq=bq, qkv=q)


lib = L.load()
n_cta = 6 * 19
tls = [torch.zeros(2 * n_cta * 16, dtype=torch.int64, device=dev) for _ in range(4)]
for _ in range(3):
    run()
for tl_i in tls:                        # four launches back to back, each with its own stamp buffer
    lib.a2f_debug_set_timeline(tl_i.data_ptr())
    run()
lib.a2f_debug_set_timeline(None)
torch.cuda.synchronize()
gt = [tl_i.view(2, n_cta, 16)[1].cpu().double() for tl_i in tls]     # globaltimer (ns)
t0 = gt[0][:, 0].min()
print("launch   first entry   median entry   last entry | median setup-done | first exit   median exit   last exit   (us, globaltimer)")
for i, g_ in enumerate(gt):
    en, sd, ex = (g_[:, 0] - t0) / 1e3, (g_[:, 1] - t0) / 1e3, (g_[:, 15] - t0) / 1e3
    print(f"{i:6d} {en.min():13.2f} {en.median():14.2f} {en.max():12.2f} | {sd.median():17.2f} | {ex.min():10.2f} {ex.median():13.2f} {ex.max():11.2f}")
t = tls[1].view(2, n_cta, 16)[0].cpu().double()
t = (t - t[:, :1])                      # cycles since this CTA's entry
lead = t[0::2]                          # leader CTAs (MMA stamps live there)
names = ["entry", "setup done", "first operands", "mma phase 0", "mma phase 1 (last)", "mma phase 2", "mma phase 3 (last)",
         "pub h1", "pub f0", "pub f1", "pub f2", "pub f3", "enter LN 2", "LN 2 stores issued", "stores drained",
         "after cluster sync"]
clk = 1965.0
print(f"cycles since CTA entry, leaders of {lead.shape[0]} pairs (median / min / max); us at {clk:.0f} MHz")
for i, nme in enumerate(names):
    col = lead[:, i]
    if float(col.max()) <= 0 and i > 0:
        continue
    print(f"{i:2d} {nme:20s} {col.median():9.0f} {col.min():9.0f} {col.max():9.0f}   {col.median() / clk:7.2f} us")
