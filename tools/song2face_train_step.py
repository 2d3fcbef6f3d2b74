"""Time of the eager Song2Face training step and its split: forward recurrences, LSTM backpropagation through time, the rest.

One step = trainer.ConvModelTrainer.step on precomputed features (a2m_features: [B, 52, 32] windows): train-mode forward,
VocaLoss, backward, fused Adam.  Weights seed 14.  Every step is timed by its own pair of CUDA events, with the L2 cache
flushed (a 256 MB buffer overwritten) before it; the median step is reported.  A second set of steps runs with CUDA events
around every a2f_lstm_recurrence_train and a2f_lstm_bptt call (two each per step) for the split; "everything else" is
that set's step time minus the four calls.

    python tools/song2face_train_step.py [--batches 64 128] [--steps 20] [--warmup 3] [--out profiles/...txt]
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
    ap.add_argument("--batches", type=int, nargs="+", default=[64, 128])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import a2f_b200  # noqa: F401
    from a2f_b200 import modules, ops, trainer as tr
    from oracle import inputs as oin, weights as ow

    if not torch.cuda.is_available():
        raise SystemExit("song2face_train_step: needs a CUDA device")
    dev = torch.device("cuda:0")
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)      # 256 MB > 126 MB of L2
    sd = ow.make_state_dict("song2face", seed=14)

    calls = None                                     # list of (kind, start, end) while instrumented

    def timed(kind, fn):
        def wrapper(*a, **k):
            if calls is None:
                return fn(*a, **k)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = fn(*a, **k)
            e.record()
            calls.append((kind, s, e))
            return out
        return wrapper

    ops.lstm_recurrence_train = timed("rec", ops.lstm_recurrence_train)
    ops.lstm_bptt = timed("bptt", ops.lstm_bptt)

    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:  # noqa: BLE001
        gpu = torch.cuda.get_device_name(0) + " (power limit not read)"
    lines = [
        "eager Song2Face training step (trainer.ConvModelTrainer: train-mode forward, VocaLoss, backward, fused Adam), fp32,",
        f"features [B, 52, 32] given; L2 flushed before every step; {args.steps} steps per set after {args.warmup} warm-up steps",
        f"GPU: {gpu}",
    ]
    for B in args.batches:
        m = modules.Song2Face(15069, 12)
        m.load_state_dict(sd, strict=True)
        m = m.to(dev)
        t = tr.ConvModelTrainer(m, lr=1e-4)
        tp = oin.batch_templates(B, 5)
        d_in = [oin.a2m_features(B, 5).to(dev), oin.one_hot(B, 12, 5).to(dev), tp.to(dev),
                oin.gt_like((B, 5023, 3), tp, 6).to(dev)]
        for _ in range(args.warmup):
            t.step(*d_in)
        torch.cuda.synchronize()

        def run_set():
            per_step = []
            for _ in range(args.steps):
                flush.zero_()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                t.step(*d_in)
                e.record()
                per_step.append((s, e))
            torch.cuda.synchronize()
            return [s.elapsed_time(e) for s, e in per_step]

        plain = run_set()
        calls = []
        inst = run_set()
        rec = [s.elapsed_time(e) for k, s, e in calls if k == "rec"]
        bptt = [s.elapsed_time(e) for k, s, e in calls if k == "bptt"]
        calls = None
        n = args.steps
        ms = statistics.median(plain)
        rec_step, bptt_step = sum(rec) / n, sum(bptt) / n
        rest = statistics.mean(inst) - rec_step - bptt_step
        lines += [
            f"B = {B} windows: {ms:.3f} ms per step (median; min {min(plain):.3f}, max {max(plain):.3f}) = "
            f"{1000.0 * B / ms:.0f} windows/s",
            f"  instrumented set, mean per step {statistics.mean(inst):.3f} ms: forward recurrences (2 calls) {rec_step:.3f} ms, "
            f"a2f_lstm_bptt (2 calls) {bptt_step:.3f} ms, everything else {rest:.3f} ms",
            f"  per call: a2f_lstm_recurrence_train median {statistics.median(rec):.3f} ms, a2f_lstm_bptt median "
            f"{statistics.median(bptt):.3f} ms; BPTT / forward recurrence = {statistics.median(bptt) / statistics.median(rec):.2f}",
        ]
        del t, m
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
