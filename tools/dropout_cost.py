"""What the wav2vec2 encoder dropout costs in the graphed FaceFormer training step (trainer.GraphedTrainStep).

Same workload as bench.py's training leg (batch 8 x 5 s at 60 fps, bf16, weights seed 13), with the model in train()
mode and SpecAugment off, once with `encoder_dropout = False` and once with it on at p = 0.1 everywhere and LayerDrop 0
(a graph cannot take LayerDrop's host-side draw).  The two variants are timed alternately in rounds in one process;
each round times `--steps` replays with CUDA events; the median round is reported.

    python tools/dropout_cost.py [--rounds 5] [--steps 20] [--out profiles/r3_dropout_cost.txt]
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--seconds", type=float, default=5.0)
    ap.add_argument("--fps", type=int, default=60)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import a2f_b200  # noqa: F401
    from a2f_b200 import modules, trainer as tr
    from oracle import inputs as oin, weights as ow

    if not torch.cuda.is_available():
        raise SystemExit("dropout_cost: needs a CUDA device")
    dev = torch.device("cuda:0")
    B, n = args.batch, int(16000 * args.seconds)
    T = n * args.fps // 16000
    tp = oin.batch_templates(B, 100, scale=100.0)
    d_in = [oin.audio(B, n, 100).to(dev), oin.one_hot(B, 12, 100).to(dev), tp.to(dev),
            oin.gt_like((B, T, 5023, 3), tp[:, None], 200, scale=100.0).to(dev)]
    sd = ow.make_state_dict("faceformer", 13)

    def graphed(dropout: bool):
        m = modules.Faceformer(15069, 12)
        m.load_state_dict(sd, strict=True)
        m = m.to(dev).train().set_precision("bf16")
        m.spec_augment = False
        m.encoder_dropout = dropout
        m.dropout_p = {"hidden": 0.1, "attention": 0.1, "activation": 0.1, "feat_proj": 0.1, "layerdrop": 0.0}
        m.dropout_seed = 1
        t = tr.FaceformerTrainer(m, lr=1e-4, fps=args.fps)
        return t.graphed(*d_in)

    steps = {"off": graphed(False), "on": graphed(True)}
    for g in steps.values():
        for _ in range(3):
            g(*d_in)
    torch.cuda.synchronize()
    times = {k: [] for k in steps}
    for _ in range(args.rounds):
        for k, g in steps.items():
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(args.steps):
                g(*d_in)
            e.record()
            e.synchronize()
            times[k].append(s.elapsed_time(e) / args.steps)
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:  # noqa: BLE001
        gpu = torch.cuda.get_device_name(0) + " (power limit not read)"
    med = {k: statistics.median(v) for k, v in times.items()}
    lines = [
        f"graphed FaceFormer training step, bf16, batch {B} x {args.seconds:g} s @ {args.fps} fps (T = {T}), train() mode, "
        "SpecAugment off",
        f"GPU: {gpu}",
        f"{args.rounds} alternating rounds x {args.steps} replays, CUDA events; per-step ms per round:",
    ]
    for k in steps:
        lines.append(f"  encoder_dropout {k:3s}: " + " ".join(f"{x:.3f}" for x in times[k]) + f"   median {med[k]:.3f} ms")
    lines.append(f"  launches per replay: off {steps['off'].launches_per_replay}, on {steps['on'].launches_per_replay}")
    lines.append(f"cost of encoder dropout (p = 0.1 at feat_proj, enc_in, attn_prob, attn_out, ffn_act, ffn_out; LayerDrop 0): "
                 f"{med['on'] - med['off']:+.3f} ms = {100 * (med['on'] / med['off'] - 1):+.1f} %")
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
