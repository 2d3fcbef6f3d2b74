"""Time of the eager Audio2Mesh / Song2Face training step with every BatchNorm training against every BatchNorm frozen.

One step = trainer.ConvModelTrainer.step on precomputed features (a2m_features: [B, 52, 32] windows): forward, VocaLoss,
backward, fused Adam.  "training": ConvModelTrainer(freeze_bn=False), batch statistics + running-stat update in every
BatchNorm; "frozen": ConvModelTrainer(freeze_bn=True), every BatchNorm in eval() (running statistics, no moments pass; γ
and β still trained).  The two trainers hold separate copies of the same weights and their steps alternate in one loop,
so drift of the machine hits both alike.  Every step is timed by its own pair of CUDA events, with the L2 cache flushed
(a 256 MB buffer overwritten) before it; the median step is reported, with the kernel launches of the library per step.

    python tools/frozen_bn_step.py [--models audio2mesh song2face] [--batches 64 128] [--steps 20] [--warmup 3] [--out ...]
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED_W = {"audio2mesh": 11, "song2face": 14}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", nargs="+", default=["audio2mesh", "song2face"], choices=sorted(SEED_W))
    ap.add_argument("--batches", type=int, nargs="+", default=[64, 128])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import a2f_b200
    from a2f_b200 import modules, trainer as tr
    from oracle import inputs as oin, weights as ow

    if not torch.cuda.is_available():
        raise SystemExit("frozen_bn_step: needs a CUDA device")
    dev = torch.device("cuda:0")
    lib = a2f_b200.lib.load()
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)      # 256 MB > 126 MB of L2

    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:  # noqa: BLE001
        gpu = torch.cuda.get_device_name(0) + " (power limit not read)"
    lines = [
        "eager training step (trainer.ConvModelTrainer: forward, VocaLoss, backward, fused Adam), fp32, features [B, 52, 32]",
        "given; every BatchNorm training (batch statistics) vs every BatchNorm frozen (freeze_bn=True), steps alternating in",
        f"one loop; L2 flushed before every step; median of {args.steps} steps after {args.warmup} warm-up steps each",
        f"GPU: {gpu}",
    ]
    for kind in args.models:
        cls = modules.Audio2Mesh if kind == "audio2mesh" else modules.Song2Face
        sd = ow.make_state_dict(kind, seed=SEED_W[kind])
        for B in args.batches:
            tp = oin.batch_templates(B, 5)
            d_in = [oin.a2m_features(B, 5).to(dev), oin.one_hot(B, 12, 5).to(dev), tp.to(dev),
                    oin.gt_like((B, 5023, 3), tp, 6).to(dev)]
            trainers = {}
            for label, freeze in (("training", False), ("frozen", True)):
                m = cls(15069, 12)
                m.load_state_dict(sd, strict=True)
                trainers[label] = tr.ConvModelTrainer(m.to(dev), lr=1e-4, freeze_bn=freeze)
            launches = {}
            for label, t in trainers.items():
                for _ in range(args.warmup):
                    t.step(*d_in)
                torch.cuda.synchronize()
                n0 = lib.a2f_launch_count()
                t.step(*d_in)
                launches[label] = int(lib.a2f_launch_count() - n0)
            torch.cuda.synchronize()
            events = {label: [] for label in trainers}
            for _ in range(args.steps):
                for label, t in trainers.items():
                    flush.zero_()
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record()
                    t.step(*d_in)
                    e.record()
                    events[label].append((s, e))
            torch.cuda.synchronize()
            ms = {label: [s.elapsed_time(e) for s, e in ev] for label, ev in events.items()}
            for label in trainers:
                v = ms[label]
                lines.append(f"{kind} B = {B} windows, BatchNorm {label:8s}: {statistics.median(v):.3f} ms per step "
                             f"(median; min {min(v):.3f}, max {max(v):.3f}) = {1000.0 * B / statistics.median(v):.0f} "
                             f"windows/s; {launches[label]} library kernel launches per step")
            ratio = statistics.median(ms["frozen"]) / statistics.median(ms["training"])
            lines.append(f"{kind} B = {B} windows: frozen / training = {ratio:.3f}")
            del trainers
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
