#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 audio->mesh hot path (DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
                    [--workload faceformer|faceformer_train|audio2mesh|voca|voca_audio]   (configs[2] | [3] | [1] | [0]-shaped |
                                                                              raw audio windows -> MFCC -> VOCA)
    (configs[4], the long-sequence sweep: tools/sweep_long.py)

--dump-outputs DIR writes the vertices the timed path returned in its last timed step to DIR/vertices.npy (float32,
[n, 5023, 3]): a fixed, seeded sample of DUMP_MESHES meshes of the output, or all of them when it has fewer.  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.

Workload (BASELINE.json configs[2], the largest single-GPU inference configuration): FaceFormer inference,
random-init wav2vec2-base encoder + 1-layer biased causal decoder, batch 32 x 5 s synthetic 16 kHz audio at 30 fps,
5023-vertex FLAME output.  One "step" = one forward of the drop-in module over one batch.  Metric: mesh frames/sec.

For N > 1 the driver launches this file under torch.distributed.run (one rank per GPU, NCCL); the path shards over
independent utterances, so there is no data-path collective (weak scaling: 32 utterances per GPU); only the timing
reduction (max over ranks) uses the process group.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# FLOP model of SURVEY.md App. C (2*MAC, KV-cached decode, no padding)
def ff_flops_per_utt(n_samples: int, T: int) -> float:
    L = [(n_samples - 10) // 5 + 1]
    for k in (3, 3, 3, 3, 2, 2):
        L.append((L[-1] - k) // 2 + 1)
    fe = 2 * 512 * (10 * L[0] + 512 * 3 * sum(L[1:5]) + 512 * 2 * (L[5] + L[6]))
    proj = 2 * 512 * 768 * T
    pos = 2 * 768 * 48 * 128 * T
    enc_lin = 12 * (8 * 768 ** 2 + 4 * 768 * 3072) * T
    enc_att = 12 * 4 * 768 * T * T
    afm = 2 * 768 * 64 * T
    dec = 81920 * T + 256 * T * (T + 1) / 2
    head = 2 * (2 * 64 * 15069 * T)
    return float(fe + proj + pos + enc_lin + enc_att + afm + dec + head)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_burst": d["bf16_tflops"], "bf16_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


_SD_CACHE = {}
DUMP_MESHES = 512          # 512 x 5023 x 3 float32 = 31 MB


def sample_meshes(out):
    """--dump-outputs: the same DUMP_MESHES meshes of a [..., 5023, 3] output on every run (seeded choice over the
    flattened leading dimensions, kept in order), as a float32 numpy array."""
    import numpy as np
    import torch
    meshes = out.reshape(-1, 5023, 3)
    n = meshes.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_MESHES), replace=False))
    return meshes[torch.from_numpy(idx).to(meshes.device)].float().cpu().numpy()


def deglitch(prof):
    """The instrumented pass runs the step twice; entry i of both runs is the same launch.  Keep the smaller of the two
    event-pair times for every launch (a host hiccup that lets the device run ahead of the enqueue inflates one pair) and
    return [(kind, flops, seconds)] for BOTH runs again, so that callers keep dividing by two."""
    rows = [(k, f, s.elapsed_time(e) * 1e-3) for (k, f, s, e) in prof]
    n = len(rows) // 2
    if n == 0 or len(rows) != 2 * n or [r[0] for r in rows[:n]] != [r[0] for r in rows[n:]]:
        return rows
    best = [(a[0], a[1], min(a[2], b[2])) for a, b in zip(rows[:n], rows[n:])]
    return best + best


# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_frames_per_s(workload: str, fps: int, seconds: float, n_utt: int, threads: int):
    """Times the oracle (CPU restatement of the reference path, reference O(T^2) decode loop included) on the host."""
    import torch
    from oracle import inputs as oin, ref_models as orm, weights as ow

    torch.set_num_threads(threads)
    with torch.set_grad_enabled(workload in ("faceformer_train", "audio2mesh_train")):
        if workload == "faceformer":
            sd = _SD_CACHE.get("faceformer") or _SD_CACHE.setdefault("faceformer", ow.make_state_dict("faceformer", 13))
            n = int(16000 * seconds)
            audio, oh, tp = oin.audio(n_utt, n, 1), oin.one_hot(n_utt, 12, 1), oin.batch_templates(n_utt, 1, scale=100.0)
            orm.faceformer_forward(sd, audio[:1, :16000], oh[:1], tp[:1], fps)          # warm-up
            t0 = time.perf_counter()
            frames = 0
            for b in range(n_utt):
                y = orm.faceformer_forward(sd, audio[b:b + 1], oh[b:b + 1], tp[b:b + 1], fps)
                frames += y.shape[1]
            dt = time.perf_counter() - t0
            return frames / dt, f"{n_utt} utterance(s) x {seconds:g} s @ {fps} fps, fp32, reference O(T^2) decode loop"
        if workload == "faceformer_train":
            from oracle import ref_train as ort
            sd = _SD_CACHE.get("faceformer") or _SD_CACHE.setdefault("faceformer", ow.make_state_dict("faceformer", 13))
            n = int(16000 * seconds)
            T = n * fps // 16000
            audio, oh, tp = oin.audio(1, n, 1), oin.one_hot(1, 12, 1), oin.batch_templates(1, 1, scale=100.0)
            gt = oin.gt_like((1, T, 5023, 3), tp[:, None], 2, scale=100.0)
            t0 = time.perf_counter()
            ort.faceformer_loss_and_grads(sd, audio, oh, tp, gt, fps)
            dt = time.perf_counter() - t0
            return T / dt, (f"1 utterance x {seconds:g} s @ {fps} fps: forward + FaceFormerLoss + autograd backward, fp32, "
                            "reference O(T^2) decode loop (no optimizer step)")
        if workload == "song2face":
            sd = ow.make_state_dict("song2face", 14)
            B = 64
            x, oh, tp = oin.a2m_features(B, 1), oin.one_hot(B, 12, 1), oin.batch_templates(B, 1)
            orm.song2face_forward(sd, x[:4], oh[:4], tp[:4])
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < 8.0:
                orm.song2face_forward(sd, x, oh, tp)
                reps += 1
            dt = time.perf_counter() - t0
            return reps * B / dt, f"{reps} x {B} windows, fp32, eval-mode BatchNorm, LSTM as a Python loop over torch ops (oracle port)"
        if workload == "audio2mesh_train":
            from oracle import ref_mfcc as omf, ref_train as ort
            cfg = omf.CONFIGS["audio2mesh"]
            sd, bufs = ow.make_state_dict("audio2mesh", 12), omf.make_buffers(cfg[0], cfg[1], cfg[3], cfg[5])
            B = 128
            x, oh, tp = oin.speech_like_windows(B, seed=1), oin.one_hot(B, 12, 1), oin.batch_templates(B, 1)
            gt = oin.gt_like((B, 5023, 3), tp, 2)

            def run():
                with torch.no_grad():
                    feat = omf.mfcc_forward(bufs, x, cfg[2], cfg[3], cfg[4], cfg[5])
                ort.conv_loss_and_grads("audio2mesh", sd, feat, oh, tp, gt)
            run()
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < 8.0:
                run()
                reps += 1
            dt = time.perf_counter() - t0
            return reps * B / dt, (f"{reps} x {B} windows: MFCC + Audio2Mesh train-mode forward + VocaLoss + autograd backward, fp32 "
                                   "(no optimizer step)")
        if workload == "voca_config0":
            import numpy as np
            from oracle import ref_audio as ora, ref_mfcc as omf
            z0 = np.load(os.path.join(ROOT, "tests", "golden", "config0_voca.npz"))
            cfg = omf.CONFIGS["voca"]
            sd, bufs = ow.make_state_dict("voca", int(z0["weight_seed"])), omf.make_buffers(cfg[0], cfg[1], cfg[3], cfg[5])
            F_ = int(z0["n_frames"])
            oh = torch.zeros(F_, 12)
            oh[:, 0] = 1.0
            tp = oin.flame_like_template(int(z0["template_seed"]))[None].expand(F_, -1, -1).contiguous()

            def run():
                win = ora.fragments(z0["clip"], F_)
                return orm.voca_forward(sd, omf.mfcc_forward(bufs, win, cfg[2], cfg[3], cfg[4], cfg[5]), oh, tp)
            run()
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < 4.0:
                run()
                reps += 1
            dt = time.perf_counter() - t0
            return reps * F_ / dt, (f"{reps} x the 348-window clip: get_audio_fragment loop + MFCC (torch stft path) + VOCA, fp32 "
                                    "(the configuration BASELINE.json configs[0] says runs on CPU)")
        if workload == "voca_audio":
            from oracle import ref_mfcc as omf
            cfg = omf.CONFIGS["voca"]
            sd, bufs = ow.make_state_dict("voca", 11), omf.make_buffers(cfg[0], cfg[1], cfg[3], cfg[5])
            B = 512
            x, oh, tp = oin.speech_like_windows(B, seed=1), oin.one_hot(B, 12, 1), oin.batch_templates(B, 1)
            run = lambda: orm.voca_forward(sd, omf.mfcc_forward(bufs, x, cfg[2], cfg[3], cfg[4], cfg[5]), oh, tp)  # noqa: E731
            run()
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < 5.0:
                run()
                reps += 1
            dt = time.perf_counter() - t0
            return reps * B / dt, f"{reps} x {B} windows of 11440 samples: MFCC (torch stft path) + VOCA, fp32"
        if workload == "audio2mesh":
            sd = ow.make_state_dict("audio2mesh", 12)
            B = 64
            x, oh, tp = oin.a2m_features(B, 1), oin.one_hot(B, 12, 1), oin.batch_templates(B, 1)
            orm.audio2mesh_forward(sd, x, oh, tp)
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < 5.0:
                orm.audio2mesh_forward(sd, x, oh, tp)
                reps += 1
            dt = time.perf_counter() - t0
            return reps * B / dt, f"{reps} x {B} windows, fp32, eval-mode BatchNorm"
        sd = ow.make_state_dict("voca", 11)
        B = 4096
        x, oh, tp = oin.voca_features(B, 1), oin.one_hot(B, 12, 1), oin.batch_templates(B, 1)
        orm.voca_forward(sd, x[:64], oh[:64], tp[:64])
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 5.0:
            orm.voca_forward(sd, x, oh, tp)
            reps += 1
        dt = time.perf_counter() - t0
        return reps * B / dt, f"{reps} x {B} windows, fp32"


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the reference itself does not
    import: ref:src/model/lightning_model.py:14 needs a missing module, and /root/reference is absent on the GPU box)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    vals = []
    sample = ""
    if args.warmup > 0:        # one untimed pass (thread pool, allocator, lazily built oracle state); more would only repeat it
        cpu_reference_frames_per_s(args.workload, args.fps, min(args.seconds, 1.0), 1, threads)
    for _ in range(max(1, args.steps)):
        v, sample = cpu_reference_frames_per_s(args.workload, args.fps, args.seconds, 1, threads)
        vals.append(v)
    value = statistics.mean(vals)
    T = int(16000 * args.seconds) * args.fps // 16000
    line = {
        "impl": "reference", "metric": "mesh frames/sec (5023-vert FLAME)", "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * (T / value if args.workload.startswith("faceformer") else 4096 / value),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args), reference_arm=(
            "oracle port (oracle/ref_models.py: plain torch fp32 restatement, pinned to the live reference by tests/golden) on all "
            "host cores; each step is a bounded sample of the workload (one utterance / one timed batch loop); one untimed "
            "warm-up pass whatever --warmup says; conservative: the real reference also materialises and returns 12 x "
            "[12,T,T] attention maps (ref:src/model/wav2vec.py:101), does a D2H+H2D round trip for the processor, and "
            "cannot be imported on the GPU box (ref:src/model/lightning_model.py:14 needs a missing module)")),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args):
    if args.workload == "faceformer":
        T = int(16000 * args.seconds) * args.fps // 16000
        return {"workload": f"faceformer_inference_b{args.batch}x{args.seconds:g}s_{args.fps}fps (BASELINE.json configs[2])",
                "batch_per_gpu": args.batch, "audio_seconds": args.seconds, "sample_rate": 16000, "fps": args.fps,
                "frames_per_utterance": T, "vertices": 5023, "weights": "random-init (oracle.weights seed 13, heads de-zeroed)",
                "l2": "flushed between timed steps (256 MiB device memset outside the per-step event pairs)",
                "template_units": "centimetres (x100, ref lightning_model.py:145-148)",
                "launch": "eager" if args.no_graph else "one CUDA graph per forward (modules.GraphedForward); the vertex head runs "
                          "on a forked stream of that graph, concurrently with the decoder rollout"}
    if args.workload == "faceformer_train":
        T = int(16000 * args.seconds) * args.fps // 16000
        return {"workload": f"faceformer_train_step_b{args.batch}_per_gpu_x{args.seconds:g}s_{args.fps}fps (BASELINE.json configs[3])",
                "batch_per_gpu": args.batch, "audio_seconds": args.seconds, "sample_rate": 16000, "fps": args.fps,
                "frames_per_utterance": T, "vertices": 5023, "precision": "bf16 tensor-core GEMMs, fp32 master weights/grads/Adam",
                "step": "forward + FaceFormerLoss (rec + 10 vel) + backward (BPTT through the free rollout) + gradient "
                        "all-reduce (NCCL, overlapped with the backward) + fused Adam(lr 1e-4, wd 1e-5)",
                "stochastic_ops": "off (dropout / LayerDrop / SpecAugment; eval-mode arithmetic, DESIGN.md)",
                "weights": "random-init (oracle.weights seed 13, heads de-zeroed)",
                "l2": "flushed between timed steps (256 MiB device memset outside the per-step event pairs)",
                "template_units": "centimetres (x100, ref lightning_model.py:145-148)",
                "launch": "eager" if args.no_graph else "one CUDA graph per optimisation step (the line's `launch` says if capture fell back)"}
    if args.workload == "audio2mesh":
        return {"workload": f"audio2mesh_inference_b{args.batch}_windows (BASELINE.json configs[1])", "batch_per_gpu": args.batch,
                "window": "52 x 32 MFCC", "vertices": 5023, "weights": "random-init (oracle.weights seed 12, randomised BatchNorm stats)",
                "l2": "flushed between timed steps (256 MiB device memset outside the per-step event pairs)",
                "launch": "eager" if args.no_graph else "one CUDA graph per forward (modules.GraphedForward)"}
    if args.workload == "song2face":
        return {"workload": f"song2face_inference_b{args.batch}_windows (registry entry song2face, SURVEY.md 8(f) rank 4)",
                "batch_per_gpu": args.batch, "window": "52 x 32 MFCC", "vertices": 5023,
                "weights": "random-init (oracle.weights seed 14, randomised BatchNorm stats)",
                "l2": "flushed between timed steps (256 MiB device memset outside the per-step event pairs)",
                "launch": "eager" if args.no_graph else "one CUDA graph per forward (modules.GraphedForward)"}
    if args.workload == "audio2mesh_train":
        return {"workload": f"audio2mesh_train_step_b{args.batch}_windows (the reference's own config.yaml: modelname audio2mesh, "
                            "feature_extractor mfcc, batch 128; BASELINE.json configs[1] shape, training)",
                "batch_per_gpu": args.batch, "window_samples": 11440, "sample_rate": 22000,
                "mfcc": "n_mfcc 32, out_dim 52, win 440, hop 220, n_fft 1024 (ref config.yaml)", "vertices": 5023,
                "step": "MFCC extractor (tcgen05 bf16x3 DFT) + train-mode forward (batch-statistics BatchNorm) + VocaLoss + "
                        "backward + gradient all-reduce + fused Adam(lr 1e-4, wd 1e-5)",
                "precision": "fp32 SIMT GEMMs for the model's forward / backward (the 1e-5 parity path)",
                "weights": "random-init (oracle.weights seed 12)",
                "l2": "flushed between timed steps (256 MiB device memset outside the per-step event pairs)", "launch": "eager"}
    if args.workload == "voca_config0":
        return {"workload": "voca_inference_audio_sample_348_windows (BASELINE.json configs[0], literal shape)",
                "input": "the reference's assets/audio_sample.npy (int16, 22 kHz, 127 600 samples; carried by tests/golden/config0_voca.npz)",
                "step": "clip -> 348 windows of 11 440 samples (get_audio_fragment / normalize_audio) -> MFCC(16 x 29) -> Voca -> [348,5023,3]",
                "batch_per_gpu": 348, "vertices": 5023, "weights": "random-init (oracle.weights seed 11)", "template": "one per window (module interface)",
                "check": "assets/verts_sample.npy is absent from the reference checkout; parity is against the live reference modules (fixture)",
                "l2": "flushed between timed steps (256 MiB device memset outside the per-step event pairs)",
                "launch": "eager" if args.no_graph else "one CUDA graph per forward (modules.GraphedForward)"}
    if args.workload == "voca_audio":
        return {"workload": f"mfcc_plus_voca_b{args.batch}_windows (BASELINE.json configs[0] from raw audio: SURVEY.md 8(f) rank 1 + a18)",
                "batch_per_gpu": args.batch, "window_samples": 11440, "sample_rate": 22000,
                "mfcc": "n_mfcc 16, win 790, hop 395, n_fft 1024, 128 mels, top_db 80 (ref config.yaml)", "vertices": 5023,
                "weights": "random-init (oracle.weights seed 11)",
                "l2": "flushed between timed steps (256 MiB device memset outside the per-step event pairs)",
                "launch": "eager" if args.no_graph else "one CUDA graph per forward (modules.GraphedForward)"}
    return {"workload": f"voca_inference_b{args.batch} (BASELINE.json configs[0] shape)", "batch_per_gpu": args.batch,
            "vertices": 5023, "weights": "random-init (oracle.weights seed 11)",
            "l2": "flushed between timed steps (256 MiB device memset outside the per-step event pairs)"}



class Ctx:
    """One process per GPU: rank / device / process group are set up ONCE in main() and shared by every workload leg."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        from a2f_b200 import lib as L
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1 and not dist.is_initialized():
            # the gradient all-reduce of the training leg runs UNDER the backward kernels: cap NCCL's CTAs so that the
            # persistent GEMM kernels keep their SMs (NVLS / NVSwitch needs few; override with the environment)
            os.environ.setdefault("NCCL_MAX_CTAS", "16")
            dist.init_process_group("nccl", device_id=self.dev)
        self.lib = L.load()
        L.check(self.lib.a2f_device_check(), "a2f_device_check")
        self.cpu_binding = self._bind_local_cpus()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)

    def _bind_local_cpus(self) -> str:
        """Bind this rank to the CPUs NVML reports as local to its GPU BEFORE any pinned staging buffer is allocated
        (first touch places the pages on that NUMA node; tools/d2h_ceiling.py measures what the box then gives)."""
        if self.world == 1:
            return "unchanged (one rank: every core stays available to the cpu_baseline leg)"
        try:
            import pynvml
            pynvml.nvmlInit()
            before = len(os.sched_getaffinity(0))
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(self.local))
            cpus = sorted(os.sched_getaffinity(0))
            return f"{before} -> {len(cpus)} cpus ({cpus[0]}..{cpus[-1]})"
        except Exception as exc:  # noqa: BLE001
            return f"unchanged ({type(exc).__name__})"

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        import torch
        import torch.distributed as dist
        if self.world == 1:
            return vals
        t = torch.tensor(list(vals), device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return tuple(float(x) for x in t)

    def close(self):
        import torch.distributed as dist
        if self.world > 1 and dist.is_initialized():
            dist.destroy_process_group()

# ---------------------------------------------------------------------------------------------------------------
def run_ours(args, ctx):
    """Inference workloads (configs[2] headline, configs[0], configs[1], ...).  Returns the JSON line (rank 0) or None."""
    import torch

    import a2f_b200  # noqa: F401
    from a2f_b200 import modules, ops
    from oracle import inputs as oin, weights as ow       # input / weight generators only (not the timed path)

    world, rank, local, dev, lib = ctx.world, ctx.rank, ctx.local, ctx.dev, ctx.lib

    B = args.batch
    if args.workload == "faceformer":
        n = int(16000 * args.seconds)
        T = n * args.fps // 16000
        model = modules.Faceformer(15069, 12)
        model.load_state_dict(ow.make_state_dict("faceformer", 13), strict=True)
        model = model.to(dev).eval().set_precision("bf16")
        h_in = [oin.audio(B, n, 100 + rank).pin_memory(), oin.one_hot(B, 12, 100 + rank).pin_memory(),
                oin.batch_templates(B, 100 + rank, scale=100.0).pin_memory()]
        units = B * T
        flops_step = B * ff_flops_per_utt(n, T)
        call = lambda a, o, t: model(a, o, t, fps=args.fps)      # noqa: E731
        out_shape = (B, T, 5023, 3)
    elif args.workload == "audio2mesh":
        model = modules.Audio2Mesh(15069, 12)
        model.load_state_dict(ow.make_state_dict("audio2mesh", 12), strict=True)
        model = model.to(dev).eval().set_precision("bf16")
        h_in = [oin.a2m_features(B, 100 + rank).pin_memory(), oin.one_hot(B, 12, 100 + rank).pin_memory(),
                oin.batch_templates(B, 100 + rank).pin_memory()]
        units = B
        flops_step = B * 131.0e6                                 # SURVEY.md 8d: 131.0 MFLOP per window
        call = lambda a, o, t: model(a, o, t)                    # noqa: E731
        out_shape = (B, 5023, 3)
    elif args.workload == "song2face":
        model = modules.Song2Face(15069, 12)
        model.load_state_dict(ow.make_state_dict("song2face", 14), strict=True)
        model = model.to(dev).eval().set_precision("bf16")
        h_in = [oin.a2m_features(B, 100 + rank).pin_memory(), oin.one_hot(B, 12, 100 + rank).pin_memory(),
                oin.batch_templates(B, 100 + rank).pin_memory()]
        units = B
        # convs (k=5,5,3,3,3 along W; 4 x k=3 along the resized axis), LSTM projections + recurrences, MLP + head
        conv = 2.0 * 64 * (16 * 72 * 5 + 8 * 108 * 360 + 4 * 162 * 324 + 2 * 243 * 486 + 256 * 729) + 2.0 * 256 * 768 * (16 + 8 + 4 + 1)
        lstm = 2.0 * 256 * 1024 * (64 + 256) + 2 * (2.0 * 256 * 1024 * 256)
        flops_step = B * (conv + lstm + 1.6e6)
        call = lambda a, o, t: model(a, o, t)                    # noqa: E731
        out_shape = (B, 5023, 3)
    elif args.workload == "voca_audio":
        from a2f_b200 import features
        voca = modules.Voca(15069, 12)
        voca.load_state_dict(ow.make_state_dict("voca", 11), strict=True)
        model = features.ExtractAndPredict(features.MFCCExtractor(22000, 16, 29, 790, None, 1024), voca).to(dev).eval()
        model.set_precision("bf16")
        h_in = [oin.speech_like_windows(B, seed=100 + rank).pin_memory(), oin.one_hot(B, 12, 100 + rank).pin_memory(),
                oin.batch_templates(B, 100 + rank).pin_memory()]
        units = B
        flops_step = B * (2.0 * 29 * 1026 * 790 + 1.679e6)       # DFT as a GEMM over the window support + VOCA
        call = lambda a, o, t: model(a, o, t)                    # noqa: E731
        out_shape = (B, 5023, 3)
    elif args.workload == "voca_config0":
        # BASELINE.json configs[0] at its literal shape: the reference's assets/audio_sample.npy (int16, 22 kHz, 127 600
        # samples; carried by tests/golden/config0_voca.npz together with the live reference's vertices) -> 348 windows
        # -> MFCC -> VOCA.  One step = the whole clip.
        import numpy as np
        from a2f_b200 import features
        z0 = np.load(os.path.join(ROOT, "tests", "golden", "config0_voca.npz"))
        voca = modules.Voca(15069, 12)
        voca.load_state_dict(ow.make_state_dict("voca", int(z0["weight_seed"])), strict=True)
        model = features.ClipToVerts(features.MFCCExtractor(22000, 16, 29, 790, None, 1024), voca).to(dev).eval()
        model.set_precision("bf16")
        B = args.batch = int(z0["n_frames"])
        oh0 = torch.zeros(B, 12)
        oh0[:, 0] = 1.0
        h_in = [torch.from_numpy(z0["clip"]).pin_memory(), oh0.pin_memory(),
                oin.flame_like_template(int(z0["template_seed"]))[None].expand(B, -1, -1).contiguous().pin_memory()]
        units = B
        flops_step = B * (2.0 * 29 * 1026 * 790 + 1.679e6)
        call = lambda a, o, t: model(a, o, t)                    # noqa: E731
        out_shape = (B, 5023, 3)
    else:
        model = modules.Voca(15069, 12)
        model.load_state_dict(ow.make_state_dict("voca", 11), strict=True)
        model = model.to(dev).eval().set_precision("bf16")
        h_in = [oin.voca_features(B, 100 + rank).pin_memory(), oin.one_hot(B, 12, 100 + rank).pin_memory(),
                oin.batch_templates(B, 100 + rank).pin_memory()]
        units = B
        flops_step = B * 1.679e6
        call = lambda a, o, t: model(a, o, t)                    # noqa: E731
        out_shape = (B, 5023, 3)
    d_in = [t.to(dev) for t in h_in]
    flush, barrier = ctx.flush, ctx.barrier

    with torch.no_grad():
        # the product's fixed-shape fast path: one forward captured as a CUDA graph (modules.GraphedForward)
        step = call if args.no_graph else model.graphed(*d_in, **({"fps": args.fps} if args.workload == "faceformer" else {}))
        n0 = lib.a2f_launch_count()
        call(*d_in)
        launches_per_step = int(lib.a2f_launch_count() - n0)
        # device-resident leg: the inputs live in the graph's captured input buffers (GraphedForward.static_in), so a
        # replay reads them in place; passing other tensors would add a device-to-device copy of every input per step
        # (1 GB of per-sample templates at the VOCA shape).  The e2e leg uploads straight into the same buffers.
        d_run = d_in if args.no_graph else step.static_in
        for _ in range(max(3, args.warmup)):
            out = step(*d_run)
        barrier()
        # ------------------------------ device-resident timing (value) ------------------------------
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()
        for s, e in ev:
            flush.zero_()                       # L2 flush, outside the event pair
            s.record()
            out = step(*d_run)
            e.record()
        barrier()
        launches = launches_per_step * args.steps   # kernels of liba2f_sm100.so executed in the timed region
        dev_s = sum(s.elapsed_time(e) for s, e in ev) * 1e-3
        n_par = {"faceformer": 1, "voca": 64}.get(args.workload, B)     # samples of the LAST TIMED step kept for the parity check
        timed_out = out[:n_par].detach().cpu() if rank == 0 else None
        dump = sample_meshes(out) if rank == 0 and args.dump_outputs else None
        # ------------------------------ end-to-end timing (host buffers) ----------------------------
        # every step: H2D of the step's inputs from pinned memory, forward, D2H of the step's result into pinned
        # memory.  Copies run on a side stream so that step i's D2H overlaps step i+1's compute (double-buffered).
        h_out = [torch.empty(out_shape, dtype=torch.float32).pin_memory() for _ in range(2)]
        d_stage = [torch.empty(out_shape, dtype=torch.float32, device=dev) for _ in range(2)]
        copy_stream = torch.cuda.Stream()
        comp = torch.cuda.current_stream()
        done = [torch.cuda.Event(), torch.cuda.Event()]
        outs = [None, None]
        barrier()
        t_e2e0 = torch.cuda.Event(enable_timing=True)
        t_e2e1 = torch.cuda.Event(enable_timing=True)
        t_e2e0.record()
        for i in range(args.steps):
            slot = i & 1
            comp.wait_event(done[slot])                         # the slot's previous D2H has drained
            if args.no_graph:
                di = [t.to(dev, non_blocking=True) for t in h_in]   # H2D of this step's inputs
            else:
                di = step.static_in                                 # H2D straight into the captured input buffers
                for dst, src in zip(di, h_in):
                    dst.copy_(src, non_blocking=True)
            d_stage[slot].copy_(step(*di))                      # graph output buffer is reused by the next replay
            outs[slot] = d_stage[slot]
            ready = torch.cuda.Event()
            ready.record(comp)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ready)
                h_out[slot].copy_(outs[slot], non_blocking=True)
                done[slot].record(copy_stream)
        comp.wait_stream(copy_stream)
        t_e2e1.record()
        barrier()
        e2e_s = t_e2e0.elapsed_time(t_e2e1) * 1e-3
        # clocks are sampled through both timed legs (device-resident and end-to-end): the first alone can be
        # shorter than two nvidia-smi sampling periods
        clocks = sampler.stop() if rank == 0 else None
        # ------------------------------ per-kernel roofline pass (instrumented, untimed) -------------
        # The GPU is parked on a spin kernel first so that the host has enqueued every launch and event of the pass
        # before the device starts: the event pairs then bracket kernels that run back to back (no host-side gaps).
        torch.cuda.synchronize()
        torch.cuda._sleep(int(0.08 * 1.9e9))
        ops.PROFILE = []
        # per-kernel pass: the vertex head is launched AFTER the rollout here (in the timed legs it runs concurrently with
        # it on a side stream, where an event pair around it would mostly measure its waiting for frames)
        had_stream_head = getattr(model, "stream_head", None)
        if had_stream_head is not None:
            model.stream_head = False
        for _ in range(2):
            call(*d_in)
        torch.cuda.synchronize()
        if had_stream_head is not None:
            model.stream_head = had_stream_head
        prof = deglitch(ops.PROFILE)
        ops.PROFILE = None

    dev_s, e2e_s = ctx.max_over_ranks(dev_s, e2e_s)
    del model, step
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    pk = peaks()
    total_units = units * world
    value = total_units * args.steps / dev_s
    e2e_value = total_units * args.steps / e2e_s
    h2d = sum(t.numel() * t.element_size() for t in h_in)
    d2h = 1
    for d in out_shape:
        d2h *= d
    d2h *= 4

    if args.workload == "faceformer":
        # dominant kernel: the tcgen05 GEMM (all bf16 launches of one forward)
        gem = [(f, t) for (kind, f, t) in prof if kind == "gemm_tc"]
        g_flops = sum(f for f, _ in gem)
        g_time = sum(t for _, t in gem)
        achieved = g_flops / g_time / 1e12
        # DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum, mean over the step's tcgen05 GEMM launches)
        # from the committed ncu pass of this same shape; null for any other shape
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r2_traffic_infer.json")
        if os.path.exists(tpath) and B == 32 and args.fps == 30 and args.seconds == 5.0:
            tj = json.load(open(tpath))
            traffic = tj["gemm_tc_all"]["dram_bytes_per_launch"]
            traffic_src = "profiles/r2_traffic_infer.json (bytes per launch, mean over %d launches)" % tj["gemm_tc_all"]["launches"]
        roofline = {"bound": "tensor", "kernel": "a2f::enc_block_kernel / gemm_tc2_kernel / gemm_tc_kernel / posconv_tc_kernel (tcgen05/TMEM/TMA "
                                                 "GEMMs incl. the one-kernel encoder blocks with their LayerNorms, all launches of a step)",
                    "achieved": achieved, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": achieved / pk["bf16_sustained"],
                    "traffic": traffic, "traffic_source": traffic_src, "peak_source": pk["source"] + ", sustained bf16",
                    "launches_per_step": len(gem) // 2, "kernel_share_of_step": (g_time / 2) / (dev_s / args.steps),
                    "whole_step_tflops": flops_step * world * args.steps / dev_s / 1e12,
                    "whole_step_frac": flops_step * world * args.steps / dev_s / 1e12 / (pk["bf16_sustained"] * world)}
    elif args.workload == "audio2mesh":
        # the ten convolutions (and the vertex head) run on tcgen05 as explicit-im2col GEMMs over the error-compensated
        # bf16x3 split; algorithmic FLOPs = 131 MFLOP per window (SURVEY.md 8d), so the 3-term split and the K padding to
        # multiples of 64 cap frac near 0.25; `executed_tflops` counts what the tensor cores actually did
        gem = [(f, t) for (kind, f, t) in prof if kind == "gemm_tc"]
        g_exec, g_time = sum(f for f, _ in gem), sum(t for _, t in gem)
        achieved = 2 * flops_step / g_time / 1e12            # two instrumented forwards
        roofline = {"bound": "tensor", "kernel": "a2f::gemm_tc2_kernel / gemm_tc_kernel (conv stack + vertex head as bf16x3-split GEMMs, "
                                                 "all launches of a step)",
                    "achieved": achieved, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": achieved / pk["bf16_sustained"],
                    "traffic": None, "peak_source": pk["source"] + ", sustained bf16", "launches_per_step": len(gem) // 2,
                    "executed_tflops": g_exec / g_time / 1e12,
                    "kernel_share_of_step": (g_time / 2) / (dev_s / args.steps),
                    "whole_step_tflops": flops_step * world * args.steps / dev_s / 1e12,
                    "note": "B=64 windows is launch / latency bound (27 launches, ~0.39 ms); --batch 1024 reaches ~0.5 M windows/s"}
    elif args.workload == "song2face":
        # dominant kernel: the two fp32 LSTM recurrences (256 dependent steps each; W_hh re-read from L2 every step by
        # B/4 CTAs) -- timed by difference: whole step minus the GEMM launches the instrumented pass sees
        gem = [(f, t) for (kind, f, t) in prof if kind in ("gemm_tc", "gemm_simt")]
        g_time = sum(t for _, t in gem) / 2
        rec_flops = B * 2 * (2.0 * 256 * 1024 * 256)
        rec_time = max(dev_s / args.steps - g_time, 1e-9)
        fp32_peak = 148 * 128 * 2 * 1.965e-3
        roofline = {"bound": "tensor", "kernel": "a2f::lstm_recurrence_kernel (fp32 SIMT; time = step minus the GEMM launches, so it "
                                                 "also carries the im2col / transpose / resize launches)",
                    "achieved": rec_flops / rec_time / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                    "frac": rec_flops / rec_time / 1e12 / fp32_peak, "traffic": None,
                    "peak_source": "fp32 FMA peak of the SIMT path (148 SMs x 128 lanes x 2 x 1.965 GHz)",
                    "gemm_share_of_step": g_time / (dev_s / args.steps),
                    "whole_step_tflops": flops_step * world * args.steps / dev_s / 1e12}
    elif args.workload == "voca_audio":
        # dominant kernel: the DFT GEMM (frames x window-folded cos|sin basis) on the bf16x3 split -- the first tcgen05
        # launch of a forward; algorithmic FLOPs = 2 * rows * 1026 * 790 (un-padded, un-split), so the 3-term split and
        # the K padding to 832 cap frac at 0.32
        gem = [(f, t) for (kind, f, t) in prof if kind == "gemm_tc"]
        dft = gem[0::2]
        g_time = sum(t for _, t in dft)
        alg = 2.0 * B * 29 * 1026 * 790 * len(dft)
        achieved = alg / g_time / 1e12
        roofline = {"bound": "tensor", "kernel": "a2f::gemm_tc2_kernel (DFT of the MFCC extractor as a bf16x3-split GEMM)",
                    "achieved": achieved, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": achieved / pk["bf16_sustained"],
                    "traffic": None, "peak_source": pk["source"] + ", sustained bf16", "launches_per_step": 1,
                    "executed_tflops": sum(f for f, _ in dft) / g_time / 1e12,
                    "kernel_share_of_step": (g_time / len(dft)) / (dev_s / args.steps)}
    elif args.workload == "voca_config0":
        # 348 windows: 42.6 MB of algorithmic traffic per step (SURVEY.md 8d: 122 456 B per window) in 6 launches -- a
        # latency-bound step; the roofline line is the WHOLE step against HBM, the head launch is listed beside it
        gem = [(f, t) for (kind, f, t) in prof if kind == "gemm_tc"]
        head = gem[1::2]
        byts = B * 122456 + h_in[0].numel() * 2
        achieved = byts / (dev_s / args.steps) / 1e9
        roofline = {"bound": "hbm", "kernel": "whole step (a2f_audio_fragments, mfcc_frames, DFT gemm_tc2, mfcc_mel_db, mfcc_dct_resize, "
                                              "voca_trunk, vertex-head gemm_tc)",
                    "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"], "traffic": None,
                    "algorithmic_bytes_per_step": byts, "launches_per_step": launches_per_step,
                    "head_launch_us": 1e6 * sum(t for _, t in head) / max(len(head), 1),
                    "head_launch_gbs": 2 * (B * 15069 * 4) * len(head) / max(sum(t for _, t in head), 1e-12) / 1e9,
                    "peak_source": pk["source"]}
    else:
        head = [(f, t) for (kind, f, t) in prof if kind == "gemm_tc"]
        byts = 2 * (B * 15069 * 4) * len(head)            # template read + vertex write per launch
        t_head = sum(t for _, t in head)
        achieved = byts / t_head / 1e9
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r1_traffic_voca.json")
        if args.workload == "voca" and B == 16384 and os.path.exists(tpath):   # the committed ncu pass is of this shape
            tj = json.load(open(tpath))
            traffic = tj["gemm_tc_all"]["dram_bytes_per_launch"]
            traffic_src = "profiles/r1_traffic_voca.json (dram bytes read + written per launch, mean over %d launches)" % tj["gemm_tc_all"]["launches"]
        roofline = {"bound": "hbm", "kernel": "a2f::gemm_tc_kernel<256,float,scalar> (vertex head + template add)",
                    "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
                    "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": byts // max(len(head), 1),
                    "kernel_share_of_step": (t_head / max(len(head), 1)) / (dev_s / args.steps),
                    "peak_source": pk["source"]}

    threads = os.cpu_count() or 1
    if world == 1 and not args.no_cpu_baseline:
        v, sample = cpu_reference_frames_per_s(args.workload, args.fps, args.seconds, 2, threads)
        cpu_baseline = {"value": v, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample}
    else:
        cpu_baseline = None

    line = {
        "metric": "mesh frames/sec (5023-vert FLAME)", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": 1e3 * dev_s / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args),
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "note": "pinned host buffers in and out through the drop-in module; D2H of step i overlaps step i+1",
                "cpu_binding": ctx.cpu_binding},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "parity": infer_parity(args, timed_out, h_in),
    }
    if dump is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "vertices.npy"), dump)
    return line


def infer_parity(args, timed_out, h_in):
    """The oracle as the CHECKER of the timed output (rank 0's last timed step), never as the thing measured: max error of
    the first sample(s) against the CPU restatement (configs[0] literal: against the live-reference fixture)."""
    import numpy as np
    import torch
    from oracle import ref_models as orm, weights as ow

    n = timed_out.shape[0]
    a, oh, tp = h_in[0], h_in[1][:n], h_in[2][:n]
    if args.workload != "voca_config0":
        a = a[:n]
    with torch.no_grad():
        if args.workload == "faceformer":
            want = orm.faceformer_forward(_SD_CACHE.get("faceformer") or _SD_CACHE.setdefault("faceformer", ow.make_state_dict("faceformer", 13)),
                                          a, oh, tp, args.fps)
            err = float((timed_out - want).abs().max()) / 100.0               # centimetres -> metres
            off = float((want - tp[:, None]).abs().max()) / 100.0
            return {"checked": f"utterance 0 of the last timed step vs oracle.faceformer_forward (fp32 CPU), {want.shape[1]} frames",
                    "max_abs_err_m": err, "tol_m": 5e-4, "err_rel_to_max_offset": err / off, "ok": bool(err < 5e-4)}
        if args.workload == "voca_config0":
            z0 = np.load(os.path.join(ROOT, "tests", "golden", "config0_voca.npz"))
            err = float(np.abs(timed_out.reshape(-1)[:: int(z0["verts_step"])].numpy() - z0["verts_sub"]).max())
            return {"checked": "all 348 windows of the last timed step vs the LIVE reference's vertices for assets/audio_sample.npy "
                               "(tests/golden/config0_voca.npz, sub-sampled)", "max_abs_err": err, "tol": 5e-4,
                    "err_rel_to_max_offset": err / float(z0["offset_absmax"]), "ok": bool(err < 5e-4)}
        if args.workload == "voca":
            want = orm.voca_forward(ow.make_state_dict("voca", 11), a, oh, tp)
            tol = 5e-5
        elif args.workload == "audio2mesh":
            want = orm.audio2mesh_forward(ow.make_state_dict("audio2mesh", 12), a, oh, tp)
            tol = 2e-4
        elif args.workload == "song2face":
            want = orm.song2face_forward(ow.make_state_dict("song2face", 14), a, oh, tp)
            tol = 2e-4
        else:
            return None
        err = float((timed_out - want).abs().max())
        off = float((want - tp).abs().max())
        return {"checked": f"first {n} windows of the last timed step vs the oracle (fp32 CPU)", "max_abs_err": err, "tol": tol,
                "err_rel_to_max_offset": err / off, "ok": bool(err < tol)}


def run_train(args, ctx):
    """BASELINE.json configs[3]: FaceFormer bf16 training step, data-parallel, batch 8 per GPU.  Under torchrun the step's
    gradient all-reduce (NCCL) is inside the timed region."""
    import torch

    from a2f_b200 import modules, ops, trainer as tr, training
    from oracle import inputs as oin, weights as ow       # input / weight generators only (not the timed path)

    world, rank, local, dev, lib = ctx.world, ctx.rank, ctx.local, ctx.dev, ctx.lib
    B, n = args.batch, int(16000 * args.seconds)
    T = n * args.fps // 16000
    model = modules.Faceformer(15069, 12)
    model.load_state_dict(ow.make_state_dict("faceformer", 13), strict=True)
    model = model.to(dev).eval().set_precision("bf16")
    trainer = tr.FaceformerTrainer(model, lr=1e-4, fps=args.fps, wire=args.wire, n_buckets=args.buckets)
    tp = oin.batch_templates(B, 100 + rank, scale=100.0)
    h_in = [oin.audio(B, n, 100 + rank).pin_memory(), oin.one_hot(B, 12, 100 + rank).pin_memory(), tp.pin_memory(),
            oin.gt_like((B, T, 5023, 3), tp[:, None], 200 + rank, scale=100.0).pin_memory()]
    d_in = [t.to(dev) for t in h_in]
    flush, barrier = ctx.flush, ctx.barrier
    units = B * T
    flops_step = 3.0 * B * ff_flops_per_utt(n, T)        # fwd + dgrad + wgrad (SURVEY.md 8d)

    # parity of the path about to be timed (rank 0): the taped forward of this batch at the initial weights, utterance 0's
    # FaceFormerLoss from the loss kernel vs the oracle's forward + loss (checker only)
    parity = None
    if rank == 0:
        with torch.no_grad():
            out0, _tape = training.forward_train(model, d_in[0], d_in[1], d_in[2].reshape(B, -1), args.fps)
            Te = T - (T % 2)
            l_gpu = ops.voca_loss_fwd(out0[0, :Te].reshape(Te, -1).contiguous(), d_in[3][0, :Te].reshape(Te, -1).contiguous(), Te,
                                      15069, 1.0, 10.0).cpu()
            del out0, _tape
        parity = train_parity(args, l_gpu, h_in)

    n0 = lib.a2f_launch_count()
    loss0 = float(trainer.step(*d_in)["loss"])
    launches_per_step = int(lib.a2f_launch_count() - n0)
    # the product's fixed-shape fast path: the whole optimisation step (re-pack, forward, fused head + loss, backward, gradient
    # all-reduce, Adam) captured as ONE CUDA graph (trainer.GraphedTrainStep); --no-graph = eager launches
    step_fn, launch_mode = trainer.step, "eager"
    if not args.no_graph:
        try:
            gstep = trainer.graphed(*d_in)
            step_fn, launch_mode = gstep, "one CUDA graph per optimisation step (trainer.GraphedTrainStep)"
            launches_per_step = gstep.launches_per_replay
        except Exception as exc:  # noqa: BLE001
            launch_mode = f"eager (graph capture failed: {type(exc).__name__}: {str(exc)[:120]})"
            torch.cuda.synchronize()
    for _ in range(max(3, args.warmup) - 1):
        step_fn(*d_in)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for s, e in ev:
        flush.zero_()
        s.record()
        out = step_fn(*d_in)
        e.record()
    barrier()
    dev_s = sum(s.elapsed_time(e) for s, e in ev) * 1e-3
    loss_last = float(out["loss"])
    # end to end: every step uploads its batch (audio, one-hot, template, ground-truth vertices) from pinned host
    # memory and reads the loss back
    # memory and reads the loss back.  The upload of step i+1 runs on a copy stream into the other half of a
    # double-buffered device batch while step i computes (the usual prefetching loader); all copies are inside the
    # timed region.
    h_loss = torch.empty(3, dtype=torch.float32).pin_memory()
    d_buf = [[torch.empty_like(t, device=dev) for t in h_in] for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    comp = torch.cuda.current_stream()
    up_done = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def upload(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])              # the step that last read this slot has finished
            for d, h in zip(d_buf[slot], h_in):
                d.copy_(h, non_blocking=True)
            up_done[slot].record(copy_stream)

    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    copy_stream.wait_event(t0)
    upload(0)
    for i in range(args.steps):
        slot = i & 1
        if i + 1 < args.steps:
            upload(slot ^ 1)
        comp.wait_event(up_done[slot])
        o = step_fn(*d_buf[slot])
        consumed[slot].record(comp)
        h_loss.copy_(torch.stack([o["loss"], o["rec_loss"], o["vel_loss"]]), non_blocking=True)
    t1.record()
    barrier()
    e2e_s = t0.elapsed_time(t1) * 1e-3
    # clocks are sampled through both timed legs (device-resident and end-to-end): the first alone can be
    # shorter than two nvidia-smi sampling periods
    clocks = sampler.stop() if rank == 0 else None
    # per-kernel roofline pass (instrumented, untimed)
    torch.cuda.synchronize()
    torch.cuda._sleep(int(0.3 * 1.9e9))      # park the GPU while the host enqueues the instrumented steps (see run_ours)
    ops.PROFILE = []
    for _ in range(2):
        trainer.step(*d_in)
    torch.cuda.synchronize()
    prof, ops.PROFILE = deglitch(ops.PROFILE), None

    dev_s, e2e_s = ctx.max_over_ranks(dev_s, e2e_s)
    comm = {"world": world, "gradient_bytes_fp32": int(trainer.flat.total) * 4, "wire": trainer.wire_description()}
    del trainer, model
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    pk = peaks()
    total_units = units * world
    gem = [(f, t) for (kind, f, t) in prof if kind in ("gemm_tc", "wgrad_tc")]
    g_flops, g_time = sum(f for f, _ in gem), sum(t for _, t in gem)
    achieved = g_flops / g_time / 1e12
    roofline = {"bound": "tensor", "kernel": "a2f::gemm_tc_kernel + a2f::wgrad_tc_kernel (tcgen05 forward / data-gradient / "
                                             "weight-gradient GEMMs, all launches of a step)",
                "achieved": achieved, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": achieved / pk["bf16_sustained"],
                "traffic": None, "peak_source": pk["source"] + ", sustained bf16", "launches_per_step": len(gem) // 2,
                "kernel_share_of_step": (g_time / 2) / (dev_s / args.steps),
                "whole_step_tflops": flops_step * world * args.steps / dev_s / 1e12,
                "whole_step_frac": flops_step * args.steps / dev_s / 1e12 / pk["bf16_sustained"]}
    threads = os.cpu_count() or 1
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        v, sample = cpu_reference_frames_per_s("faceformer_train", args.fps, min(args.seconds, 2.0), 1, threads)
        cpu_baseline = {"value": v, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample}
    line = {
        "metric": "mesh frames/sec (5023-vert FLAME)", "value": total_units * args.steps / dev_s, "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": 1e3 * dev_s / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args),
        "e2e": {"value": total_units * args.steps / e2e_s, "unit": "frames/s",
                "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in h_in), "d2h_bytes_per_step": 12,
                "note": "pinned host batch (audio, one-hot, template, ground-truth vertices) in, loss scalars out; the upload of step i+1 overlaps step i (copy stream, double-buffered device batch)"},
        "gpu_launches": int(launches_per_step * args.steps), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
        "loss_first_step": float(loss0), "loss_last_timed_step": loss_last, "parity": parity, "gradient_exchange": comm,
        "launch": launch_mode,
    }
    return line


def train_parity(args, l_gpu, h_in):
    import torch
    from oracle import ref_models as orm, weights as ow
    sd = _SD_CACHE.get("faceformer") or _SD_CACHE.setdefault("faceformer", ow.make_state_dict("faceformer", 13))
    with torch.no_grad():
        want = orm.faceformer_loss(orm.faceformer_forward(sd, h_in[0][:1], h_in[1][:1], h_in[2][:1], args.fps), h_in[3][:1])
    rel = {k: abs(float(l_gpu[j]) - float(want[k])) / abs(float(want[k])) for j, k in enumerate(("loss", "rec_loss", "vel_loss"))}
    return {"checked": "utterance 0 of the timed batch at the initial weights: taped bf16 forward + loss kernel vs the oracle's fp32 "
                       "forward + FaceFormerLoss", "loss_gpu": float(l_gpu[0]), "loss_oracle": float(want["loss"]),
            "rel_err": rel, "tol_rel": {"loss": 1e-4, "rec_loss": 5e-4, "vel_loss": 5e-4},
            "note": "loss (the optimised quantity): north_star's 1e-4; its components sit on the bf16 noise floor of the 12-layer "
                    "post-LN encoder at T=300 (2e-4 .. 3e-4 in a pure-oracle emulation of bf16 operands, tools/bf16_noise_floor.py)",
            "ok": bool(rel["loss"] < 1e-4 and rel["rec_loss"] < 5e-4 and rel["vel_loss"] < 5e-4)}


def run_conv_train(args, ctx):
    """The reference's default configuration (ref:config.yaml): Audio2Mesh + MFCC extractor, batch 128, one training step."""
    import torch

    from a2f_b200 import features, modules, ops, trainer as tr
    from oracle import inputs as oin, weights as ow       # input / weight generators only (not the timed path)

    world, rank, local, dev, lib = ctx.world, ctx.rank, ctx.local, ctx.dev, ctx.lib
    B = args.batch
    model = modules.Audio2Mesh(15069, 12)
    model.load_state_dict(ow.make_state_dict("audio2mesh", 12), strict=True)
    model = model.to(dev)
    ext = features.MFCCExtractor(22000, 32, 52, 440, None, 1024).to(dev).set_precision("bf16")
    trainer = tr.ConvModelTrainer(model, ext, lr=1e-4)
    tp = oin.batch_templates(B, 100 + rank)
    h_in = [oin.speech_like_windows(B, seed=100 + rank).pin_memory(), oin.one_hot(B, 12, 100 + rank).pin_memory(), tp.pin_memory(),
            oin.gt_like((B, 5023, 3), tp, 200 + rank).pin_memory()]
    d_in = [t.to(dev) for t in h_in]
    flush, barrier = ctx.flush, ctx.barrier
    flops_step = 3.0 * B * 131.0e6 + B * 2.0 * 53 * 1026 * 440      # fwd + dgrad + wgrad of the model, DFT of the extractor

    n0 = lib.a2f_launch_count()
    loss0 = float(trainer.step(*d_in)["loss"])
    launches_per_step = int(lib.a2f_launch_count() - n0)
    for _ in range(max(3, args.warmup) - 1):
        trainer.step(*d_in)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for s, e in ev:
        flush.zero_()
        s.record()
        out = trainer.step(*d_in)
        e.record()
    barrier()
    dev_s = sum(s.elapsed_time(e) for s, e in ev) * 1e-3
    loss_last = float(out["loss"])
    h_loss = torch.empty(3, dtype=torch.float32).pin_memory()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        di = [t.to(dev, non_blocking=True) for t in h_in]
        o = trainer.step(*di)
        h_loss.copy_(torch.stack([o["loss"], o["rec_loss"], o["vel_loss"]]), non_blocking=True)
    t1.record()
    barrier()
    e2e_s = t0.elapsed_time(t1) * 1e-3
    # clocks are sampled through both timed legs (device-resident and end-to-end): the first alone can be
    # shorter than two nvidia-smi sampling periods
    clocks = sampler.stop() if rank == 0 else None
    torch.cuda.synchronize()
    torch.cuda._sleep(int(0.3 * 1.9e9))
    ops.PROFILE = []
    for _ in range(2):
        trainer.step(*d_in)
    torch.cuda.synchronize()
    prof, ops.PROFILE = deglitch(ops.PROFILE), None
    dev_s, e2e_s = ctx.max_over_ranks(dev_s, e2e_s)
    del trainer, model
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    gem = [(f, t) for (kind, f, t) in prof if kind == "gemm_simt"]
    g_flops, g_time = sum(f for f, _ in gem), sum(t for _, t in gem)
    fp32_peak = 148 * 128 * 2 * 1.965e-3
    roofline = {"bound": "tensor", "kernel": "a2f::gemm_simt_kernel (fp32 forward / data-gradient GEMMs of the conv stack; weight "
                                             "gradients run in the SIMT wgrad kernel)",
                "achieved": g_flops / g_time / 1e12, "peak": fp32_peak, "unit": "TFLOP/s", "frac": g_flops / g_time / 1e12 / fp32_peak,
                "traffic": None, "peak_source": "fp32 FMA peak of the SIMT path (148 SMs x 128 lanes x 2 x 1.965 GHz)",
                "launches_per_step": len(gem) // 2, "kernel_share_of_step": (g_time / 2) / (dev_s / args.steps),
                "whole_step_tflops": flops_step * world * args.steps / dev_s / 1e12}
    threads = os.cpu_count() or 1
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        v, sample = cpu_reference_frames_per_s("audio2mesh_train", args.fps, args.seconds, 1, threads)
        cpu_baseline = {"value": v, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample}
    line = {
        "metric": "mesh frames/sec (5023-vert FLAME)", "value": B * world * args.steps / dev_s, "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": 1e3 * dev_s / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "e2e": {"value": B * world * args.steps / e2e_s, "unit": "frames/s",
                "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in h_in), "d2h_bytes_per_step": 12,
                "note": "pinned host batch (audio windows, one-hot, template, ground-truth vertices) in, loss scalars out"},
        "gpu_launches": int(launches_per_step * args.steps), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
        "loss_first_step": loss0, "loss_last_timed_step": loss_last,
    }
    return line


def run_sweep(args, ctx):
    """BASELINE.json configs[4] in brief (the full grid is tools/sweep_long.py): FaceFormer autoregressive decode of long
    utterances at 60 fps, TOTAL batch fixed per point (strong scaling: B_total / n_gpus utterances per rank, at least one --
    ranks beyond B_total run replicas and are not counted), eager launches, bf16."""
    import torch

    from a2f_b200 import modules
    from oracle import inputs as oin, weights as ow       # input / weight generators only (not the timed path)

    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    m = modules.Faceformer(15069, 12)
    m.load_state_dict(ow.make_state_dict("faceformer", 13), strict=True)
    m = m.to(dev).eval().set_precision("bf16")
    pk = peaks()
    rows = []
    steps = args.steps
    for L_s, B_total in ((10.0, 128), (30.0, 32), (60.0, 8)):
        n = int(16000 * L_s)
        T = n * 60 // 16000
        Bp = max(1, B_total // world)
        counted = min(world, B_total)                       # ranks holding distinct utterances
        audio = oin.audio(1, n, 7 + rank).to(dev).expand(Bp, n).contiguous()
        audio *= torch.linspace(0.7, 1.3, Bp, device=dev)[:, None]
        oh = oin.one_hot(Bp, 12, 7).to(dev)
        tp = oin.batch_templates(1, 7, scale=100.0).to(dev).expand(Bp, 5023, 3).contiguous()
        with torch.no_grad():
            for _ in range(2):
                out = m(audio, oh, tp, fps=60)
            finite = bool(torch.isfinite(out[:, -1]).all())
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            ctx.barrier()
            for s_, e_ in ev:
                ctx.flush.zero_()
                s_.record()
                out = m(audio, oh, tp, fps=60)
                e_.record()
            ctx.barrier()
        sec, = ctx.max_over_ranks(sum(s_.elapsed_time(e_) for s_, e_ in ev) * 1e-3)
        del out, audio, tp
        torch.cuda.empty_cache()
        frames = counted * Bp * T * steps / sec
        tfl = counted * Bp * ff_flops_per_utt(n, T) * steps / sec / 1e12
        rows.append({"seconds": L_s, "batch_total": counted * Bp, "batch_per_gpu": Bp, "gpus_with_work": counted,
                     "frames_per_utterance": T, "ms_per_step": 1e3 * sec / steps, "frames_per_s": frames, "tflops": tfl,
                     "frac_of_bf16_sustained": tfl / (pk["bf16_sustained"] * counted), "finite": finite})
    del m
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    return {"metric": "mesh frames/sec (5023-vert FLAME)", "unit": "frames/s", "n_gpus": world, "steps": steps, "warmup": 2,
            "scaling": "strong (total batch fixed per point)", "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "faceformer_long_sequence_sweep_60fps (BASELINE.json configs[4], three points; full grid: "
                                   "tools/sweep_long.py -> profiles/)", "launch": "eager",
                       "l2": "flushed between timed steps (256 MiB device memset outside the per-step event pairs)"},
            "points": rows, "value": max(r["frames_per_s"] for r in rows)}


EXTRA_WORKLOADS = (          # (key, workload, batch, fps) -- legs the default invocation runs after the headline
    ("voca_config0", "voca_config0", 348, None),
    ("voca_b16384", "voca", 16384, None),
    ("audio2mesh_b64", "audio2mesh", 64, None),
    ("faceformer_train_b8", "faceformer_train", 8, 60),
    ("long_sweep", "sweep", None, 60),
)


def run_one(args, ctx):
    if args.workload == "faceformer_train":
        return run_train(args, ctx)
    if args.workload == "audio2mesh_train":
        return run_conv_train(args, ctx)
    if args.workload == "sweep":
        return run_sweep(args, ctx)
    return run_ours(args, ctx)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=["faceformer", "voca", "voca_config0", "voca_audio", "audio2mesh",
                                                         "faceformer_train", "audio2mesh_train", "song2face", "sweep"],
                    help="one workload only; default: the headline (faceformer, BASELINE.json configs[2]) followed by the "
                         "other BASELINE configs as `extra_workloads` of the same JSON line")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--seconds", type=float, default=5.0)
    ap.add_argument("--fps", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="default invocation: skip the extra workloads")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of the CUDA-graph fast path")
    ap.add_argument("--wire", default=None, choices=["fp32", "bf16"], help="faceformer_train: gradient all-reduce wire format "
                                                                             "(default: bf16 for the bf16 step)")
    ap.add_argument("--buckets", type=int, default=7, help="faceformer_train: all-reduce buckets per step (14 = one per stage)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="inference workloads: write the last timed step's vertices (a fixed sample of at most "
                         f"{DUMP_MESHES} meshes) to DIR/vertices.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    with_extras = args.workload is None and not args.no_extra and args.impl == "ours"
    if args.workload is None:
        args.workload = "faceformer"
    if args.dump_outputs and (args.impl != "ours" or args.workload in ("faceformer_train", "audio2mesh_train", "sweep")):
        ap.error("--dump-outputs applies to the inference workloads of --impl ours")
    defaults = {"faceformer": 32, "faceformer_train": 8, "voca": 16384, "voca_config0": 348, "voca_audio": 4096, "audio2mesh": 64,
                "audio2mesh_train": 128, "song2face": 64, "sweep": 0}
    if args.fps is None:
        args.fps = 60 if args.workload in ("faceformer_train", "sweep") else 30
    if args.batch is None:
        args.batch = defaults[args.workload]
    if args.impl == "reference":
        run_reference(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun when called directly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    ctx = Ctx()
    line = run_one(args, ctx)
    if with_extras:
        extras = {}
        for key, wl, batch, fps in EXTRA_WORKLOADS:
            sub = argparse.Namespace(**vars(args))
            sub.workload, sub.batch, sub.fps = wl, batch, fps if fps is not None else 30
            sub.seconds = 5.0
            sub.dump_outputs = None                 # the dump is the headline workload's output
            try:
                extras[key] = run_one(sub, ctx)
            except Exception as exc:  # noqa: BLE001  (an extra leg must never take the headline line down with it)
                import traceback
                extras[key] = {"error": f"{type(exc).__name__}: {exc}", "traceback": traceback.format_exc()[-1500:]}
        if line is not None:
            line["extra_workloads"] = extras
    if line is not None:
        print(json.dumps(line))
    ctx.close()


if __name__ == "__main__":
    main()
