"""Time of the FaceFormer training step with parts of the audio encoder frozen (requires_grad False).

One step = trainer.FaceformerTrainer.step at the bench training shape (bf16; B utterances of S seconds at F fps): re-pack of
the changed operands, forward, fused head + loss, backward down to the lowest trainable op, fused Adam.  Configurations:
"none" (everything trains: the bench step), "feature_encoder" (audio_encoder.freeze_feature_encoder()), "lower_layers"
(feature encoder, feature projection, positional conv, encoder.layer_norm and layers 0-5 frozen), "audio_encoder"
(audio_encoder.requires_grad_(False): the decoder side trains).  Each configuration has its own trainer and copy of
the weights; their steps alternate in one loop, so drift of the machine hits all alike.  Every step is timed by its
own pair of CUDA events with the L2 cache flushed (a 256 MB buffer overwritten) before it; the median is reported for
the eager step and for the replay of its CUDA graph (trainer.GraphedTrainStep), with the kernel launches per step and
the peak memory the eager step allocates on top of the resident state (parameters, gradients, Adam moments).

    python tools/frozen_encoder_step.py [--batch 8] [--seconds 5] [--fps 60] [--steps 20] [--warmup 3] [--out ...]
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = ("none", "feature_encoder", "lower_layers", "audio_encoder")


def freeze(model, config: str) -> None:
    ae = model.audio_encoder
    if config == "feature_encoder":
        ae.freeze_feature_encoder()
    elif config == "lower_layers":
        for mod in (ae.feature_extractor, ae.feature_projection, ae.encoder.pos_conv_embed, ae.encoder.layer_norm):
            mod.requires_grad_(False)
        for blk in ae.encoder.layers[:6]:
            blk.requires_grad_(False)
    elif config == "audio_encoder":
        ae.requires_grad_(False)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--seconds", type=float, default=5.0)
    ap.add_argument("--fps", type=int, default=60)
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS), choices=CONFIGS)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import a2f_b200
    from a2f_b200 import modules, trainer as tr
    from oracle import inputs as oin, weights as ow

    if not torch.cuda.is_available():
        raise SystemExit("frozen_encoder_step: needs a CUDA device")
    dev = torch.device("cuda:0")
    lib = a2f_b200.lib.load()
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)      # 256 MB > 126 MB of L2
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:  # noqa: BLE001
        gpu = torch.cuda.get_device_name(0) + " (power limit not read)"

    B, n = args.batch, int(16000 * args.seconds)
    T = n * args.fps // 16000
    sd = ow.make_state_dict("faceformer", 13)
    tp = oin.batch_templates(B, 100, scale=100.0)
    d_in = [oin.audio(B, n, 100).to(dev), oin.one_hot(B, 12, 100).to(dev), tp.to(dev),
            oin.gt_like((B, T, 5023, 3), tp[:, None], 200, scale=100.0).to(dev)]
    trainers, graphs, launches, peak, ntrain, loss0 = {}, {}, {}, {}, {}, {}
    for c in args.configs:
        m = modules.Faceformer(15069, 12)
        m.load_state_dict(sd, strict=True)
        m = m.to(dev).eval().set_precision("bf16")
        freeze(m, c)
        t = trainers[c] = tr.FaceformerTrainer(m, lr=1e-4, fps=args.fps)
        ntrain[c] = sum(p.numel() for _, p, *_ in t.flat.entries)
        loss0[c] = float(t.step(*d_in)["loss"])                   # first step at the initial weights: the same loss
        for _ in range(args.warmup):
            t.step(*d_in)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        n0 = lib.a2f_launch_count()
        t.step(*d_in)
        torch.cuda.synchronize()
        launches[c] = int(lib.a2f_launch_count() - n0)
        peak[c] = torch.cuda.max_memory_allocated() - base
        graphs[c] = t.graphed(*d_in)
        for _ in range(args.warmup):
            graphs[c](*d_in)
    torch.cuda.synchronize()
    events = {(c, mode): [] for c in args.configs for mode in ("eager", "graph")}
    for _ in range(args.steps):
        for mode in ("eager", "graph"):
            for c in args.configs:
                fn = trainers[c].step if mode == "eager" else graphs[c]
                flush.zero_()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                fn(*d_in)
                e.record()
                events[(c, mode)].append((s, e))
    torch.cuda.synchronize()
    ms = {k: [s.elapsed_time(e) for s, e in v] for k, v in events.items()}
    med = {k: statistics.median(v) for k, v in ms.items()}
    lines = [
        f"FaceFormer training step (trainer.FaceformerTrainer), bf16, B = {B} x {args.seconds:g} s at {args.fps} fps "
        f"(T = {T}), one GPU;",
        "configurations alternate in one loop, eager steps and graph replays interleaved; L2 flushed before every step;",
        f"median of {args.steps} steps after {args.warmup} warm-up steps each",
        f"GPU: {gpu}",
    ]
    for c in args.configs:
        e, g = ms[(c, "eager")], ms[(c, "graph")]
        lines.append(f"frozen {c:16s}: eager {med[(c, 'eager')]:7.3f} ms (min {min(e):.3f}, max {max(e):.3f}), "
                     f"graph {med[(c, 'graph')]:7.3f} ms (min {min(g):.3f}, max {max(g):.3f}); "
                     f"{launches[c]} launches; {ntrain[c] / 1e6:.1f} M trainable parameters; "
                     f"step peak {peak[c] / 2**20:.0f} MiB above the resident state; first loss {loss0[c]:.6f}")
    if "none" in args.configs:
        for c in args.configs:
            if c != "none":
                lines.append(f"frozen {c:16s} / none: eager {med[(c, 'eager')] / med[('none', 'eager')]:.3f}, "
                             f"graph {med[(c, 'graph')] / med[('none', 'graph')]:.3f}")
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
