"""Data-parallel FaceFormer training step on the sm_100a kernels (BASELINE.json configs[3]).

Mirrors what Lightning does around the reference model (ref:src/model/lightning_model.py:145-161 training_step,
:209-213 configure_optimizers = Adam(lr, weight_decay=lr/10); ref:train.py:48-60 Trainer -> implicit DDP, SURVEY.md
2.1): one process per GPU, every rank holds a replica and a shard of the utterances, and exactly ONE exchange per
step -- the gradient all-reduce (NCCL over NVLink/NVSwitch).

B200-first layout: parameters, gradients and the two Adam moments live in four FLAT fp32 buffers (the nn.Parameters
are re-pointed at views of them, state_dict keys unchanged).  The flat order is the order in which the explicit
backward pass (training.backward) finishes gradients, cut into 14 contiguous stages which are grouped into a few
BUCKETS: as soon as the last stage of a bucket is final, the bucket is handed to ncclAllReduce, which runs on NCCL's
stream underneath the remaining backward kernels.  Wire format: with precision "bf16" the bucket is cast to a flat
bf16 mirror first (one kernel) and reduced in bf16 -- half the bytes on NVLink (193 MB instead of 386 MB for
FaceFormer; the round-1 limiter at 8 GPUs, VERDICT r1 weak #8); the fused Adam kernel (a2f_adam_step_bf16g) reads
the reduced bf16 gradient directly, masters / moments / update stay fp32, the 1/world average is folded in.
Same trade as torch DDP's bf16_compress_hook; wire="fp32" keeps the exact fp32 sum.

FlatBuffers is device-agnostic host logic (it is covered by world_size-2 gloo tests on CPU); the compute path is
CUDA only -- there is no CPU fallback.
"""
from __future__ import annotations

from typing import Callable, Dict, Iterable, List, Optional, Tuple

import torch
import torch.distributed as dist

from . import lib as L

ALIGN = 64          # every parameter starts on a 256-byte boundary of the flat buffers (TMA reduce-add / float4 access)


def _world() -> int:
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def default_buckets(n_stages: int, n_buckets: int = 7) -> List[List[int]]:
    """Group the backward's stages (0 = finished first) into at most n_buckets all-reduce buckets of consecutive stages.
    The LAST stage (the front end, final only when the backward ends) always travels alone so that nothing else waits
    for it; the others are split evenly: [[0,1,2], [3,4], [5,6], [7,8], [9,10], [11,12], [13]] for FaceFormer's 14 stages
    with the default of 7 -- measured best at 8 GPUs (profiles/r2_train_scaling_8gpu.txt: 7 buckets 13.07 ms, 14 buckets
    13.27 ms, 4 buckets 15.20 ms: a bucket of four encoder layers starts too late to hide under the backward)."""
    if n_stages <= 1 or n_buckets <= 1:
        return [list(range(n_stages))]
    n_buckets = min(n_buckets, n_stages)
    head = list(range(n_stages - 1))
    k = n_buckets - 1
    out, i = [], 0
    for j in range(k):
        size = (len(head) - i + (k - j) - 1) // (k - j)
        out.append(head[i:i + size])
        i += size
    return [b for b in out if b] + [[n_stages - 1]]


class FlatBuffers:
    """Flat parameter / gradient storage cut into all-reduce stages.

    named_params: iterable of (name, nn.Parameter); stage_of(name) -> int in [0, n_stages).  Parameters are laid out
    stage by stage (original order inside a stage); `p.data` and `p.grad` become views into `params` / `grads`.
    wire: "fp32" (exact sum) or "bf16" (the exchange runs on a bf16 mirror `grads_wire`; `reduced_grads()` is what the
    optimizer reads).  buckets: lists of consecutive stages reduced by one collective each (default: one per stage)."""

    def __init__(self, named_params: Iterable[Tuple[str, torch.nn.Parameter]], stage_of: Callable[[str], int],
                 n_stages: int, skip: Iterable[str] = (), order_in_stage: Optional[Callable[[str], int]] = None,
                 wire: str = "fp32", buckets: Optional[List[List[int]]] = None):
        skip = set(skip)
        items = [(n, p) for n, p in named_params if n not in skip and p.requires_grad]
        if not items:
            raise ValueError("no trainable parameters")
        if wire not in ("fp32", "bf16"):
            raise ValueError("wire must be 'fp32' or 'bf16'")
        dev = items[0][1].device
        for n, p in items:
            if p.dtype != torch.float32 or p.device != dev:
                raise ValueError(f"{n}: flat buffers hold fp32 parameters of one device")
        # order_in_stage(name): optional rank inside a stage (ties keep the original order); used to make q/k/v weight
        # (and bias) gradients adjacent so that one fused weight-gradient GEMM / column sum writes all three
        rank = order_in_stage if order_in_stage is not None else (lambda n: 0)
        order = sorted(range(len(items)), key=lambda i: (stage_of(items[i][0]), rank(items[i][0]), i))
        self.entries: List[Tuple[str, torch.nn.Parameter, int, int, int]] = []
        self.stage_ranges: List[Tuple[int, int]] = []
        off = 0
        cur = 0
        lo = 0
        for i in order:
            name, p = items[i]
            st = stage_of(name)
            if not 0 <= st < n_stages:
                raise ValueError(f"{name}: stage {st} out of range")
            while cur < st:
                self.stage_ranges.append((lo, off))
                lo, cur = off, cur + 1
            self.entries.append((name, p, off, p.numel(), st))
            off += (p.numel() + ALIGN - 1) // ALIGN * ALIGN
        while cur < n_stages:
            self.stage_ranges.append((lo, off))
            lo, cur = off, cur + 1
        self.total = off
        self.params = torch.zeros(off, dtype=torch.float32, device=dev)
        self.grads = torch.zeros(off, dtype=torch.float32, device=dev)
        self.wire = wire
        self.grads_wire = torch.zeros(off, dtype=torch.bfloat16, device=dev) if wire == "bf16" else None
        with torch.no_grad():
            for name, p, o, n, _ in self.entries:
                self.params[o:o + n].copy_(p.detach().reshape(-1))
                p.data = self.params[o:o + n].view(p.shape)
                p.grad = self.grads[o:o + n].view(p.shape)
        self.buckets = [list(b) for b in buckets] if buckets is not None else [[s] for s in range(n_stages)]
        flat = [s for b in self.buckets for s in b]
        if flat != list(range(n_stages)):
            raise ValueError("buckets must list every stage once, in order, as runs of consecutive stages")
        self._bucket_of = {s: i for i, b in enumerate(self.buckets) for s in b}
        self._pending: List = []
        self._ready = [False] * n_stages
        self._sent = [False] * len(self.buckets)

    # -- gradient exchange ---------------------------------------------------------------------------------------
    def zero_grads(self) -> None:
        self.grads.zero_()
        self._ready = [False] * len(self.stage_ranges)
        self._sent = [False] * len(self.buckets)

    def bucket_range(self, b: int) -> Tuple[int, int]:
        return self.stage_ranges[self.buckets[b][0]][0], self.stage_ranges[self.buckets[b][-1]][1]

    def _send_bucket(self, b: int, group=None) -> None:
        lo, hi = self.bucket_range(b)
        self._sent[b] = True
        if hi <= lo or _world() == 1:
            return
        if self.wire == "bf16":
            src, dst = self.grads[lo:hi], self.grads_wire[lo:hi]
            if src.is_cuda:
                from . import ops
                ops.cast_into(src, dst)                 # one kernel on the compute stream, ordered after the backward so far
            else:
                dst.copy_(src)                          # host-logic tests (gloo, CPU tensors)
            buf = dst
        else:
            buf = self.grads[lo:hi]
        self._pending.append(dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group, async_op=True))

    def all_reduce_stage(self, stage: int, group=None) -> None:
        """Mark one stage's gradients final; when that completes a bucket, start its (asynchronous) sum all-reduce.
        With NCCL the collective is ordered after everything already enqueued on the current stream and runs on NCCL's
        own stream, i.e. under the backward kernels launched afterwards."""
        self._ready[stage] = True
        b = self._bucket_of[stage]
        if not self._sent[b] and all(self._ready[s] for s in self.buckets[b]):
            self._send_bucket(b, group)

    def finish_all_reduce(self, group=None) -> None:
        """Reduce every bucket that was not started during the backward, then make the current stream wait for all."""
        for b, done in enumerate(self._sent):
            if not done:
                self._send_bucket(b, group)
        for h in self._pending:
            h.wait()
        self._pending = []

    def reduced_grads(self) -> torch.Tensor:
        """The flat gradient the optimizer reads after finish_all_reduce(): the bf16 wire mirror when the exchange ran
        in bf16 on more than one rank, else the fp32 buffer."""
        return self.grads_wire if (self.wire == "bf16" and _world() > 1) else self.grads

    def broadcast_params(self, src: int = 0, group=None) -> None:
        if _world() > 1:
            dist.broadcast(self.params, src=src, group=group)

    def bump_versions(self) -> None:
        """The fused optimizer writes through raw pointers; tell torch (and the modules' derived-weight caches, which
        key on the version counters) that the parameters changed."""
        for _, p, _, _, _ in self.entries:
            torch.autograd.graph.increment_version(p)

    def named_grads(self) -> Dict[str, torch.Tensor]:
        return {name: self.grads[o:o + n].view(p.shape) for name, p, o, n, _ in self.entries}


class FaceformerTrainer:
    """One process per GPU.  `step(audio, one_hot, template, gt)` = forward + FaceFormerLoss + backward + gradient
    all-reduce + Adam, in the units it is given; `training_step(batch)` applies the reference's x100 scaling first
    (ref:src/model/lightning_model.py:145-148).  Eval-mode arithmetic by default (dropout / LayerDrop / SpecAugment off,
    DESIGN.md); `model.encoder_dropout = True` in train() mode turns on the wav2vec2 encoder's dropout and LayerDrop.
    The rank is folded into the dropout key (replicas draw independent masks); LayerDrop draws from the seed alone
    (every replica skips the same layers).  A layer skipped by LayerDrop gets no gradient, and like torch.optim.Adam
    for `grad is None`, its parameters, moments and step count stay untouched that step.

    Frozen parameters (requires_grad False when the trainer is constructed, e.g. after
    `model.audio_encoder.freeze_feature_encoder()`) are not trained: they stay out of the flat buffers (no gradient, no
    Adam moments, `.grad` stays None), the backward stops at the lowest trainable op, and only the packed operands of
    trainable parameters are re-derived after each update.  Changing the trainable set later raises at the next step.

    Batch semantics (extension; the reference is batch-1): loss = mean over the utterances of the per-utterance
    FaceFormerLoss; across ranks the gradient is the average of the per-rank gradients (DDP semantics)."""

    def __init__(self, model, lr: float = 1e-4, weight_decay: Optional[float] = None, betas=(0.9, 0.999), eps: float = 1e-8,
                 fps: int = 60, overlap: bool = True, group=None, wire: Optional[str] = None, n_buckets: int = 7):
        from . import training
        if not next(model.parameters()).is_cuda:
            raise L.A2FError("FaceformerTrainer runs on CUDA (sm_100a) only; there is no CPU fallback")
        self.model = model
        self.lr = float(lr)
        self.weight_decay = float(lr / 10 if weight_decay is None else weight_decay)    # ref lightning_model.py:99
        self.betas, self.eps = betas, float(eps)
        self.fps = int(fps)
        self.overlap = overlap
        self.group = group
        # wire format of the gradient exchange: bf16 for the bf16 tensor-core step, exact fp32 for the fp32 parity path
        self.wire = wire if wire is not None else ("bf16" if getattr(model, "precision", "fp32") == "bf16" else "fp32")
        self.flat = FlatBuffers(model.named_parameters(), training.grad_stage_of, training.N_GRAD_STAGES,
                                skip=training.no_grad_params(model), order_in_stage=training.grad_order_in_stage,
                                wire=self.wire, buckets=default_buckets(training.N_GRAD_STAGES, n_buckets))
        # the flat buffers hold the parameters that require grad now: freezing or unfreezing one later would leave them wrong
        self._requires_grad = frozenset(n for n, p in model.named_parameters() if p.requires_grad)
        self.exp_avg = torch.zeros_like(self.flat.params)
        self.exp_avg_sq = torch.zeros_like(self.flat.params)
        self.steps = 0
        self.flat.broadcast_params(0, group)
        self.flat.bump_versions()
        self._ws = None
        self._step_dev = torch.zeros(1, dtype=torch.int32, device=self.flat.params.device)
        if _world() > 1:
            # one dropout seed for all replicas (rank 0's, drawn there if unset): LayerDrop must skip the same layers on
            # every rank, and the rank is folded into the Philox key so that the dropout masks differ
            seed = torch.tensor([-1 if model.dropout_seed is None else int(model.dropout_seed)], dtype=torch.int64,
                                device=self.flat.params.device)
            if dist.get_rank(group) == 0 and model.dropout_seed is None:
                seed.fill_(int(torch.randint(0, 2 ** 62, (1,)).item()))
            dist.broadcast(seed, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            model.dropout_seed = int(seed.item())
        training.set_dropout_rank(model, dist.get_rank() if _world() > 1 else 0)
        self._skipped_stages = frozenset()      # stages of the layers LayerDrop skipped in the last forward
        self._stage_steps = None                # per-stage Adam step counts once LayerDrop has skipped a stage
        self._dy = None
        self._ws_head = None

    # -- one optimisation step -------------------------------------------------------------------------------------
    def forward_backward(self, audio, one_hot, template, gt) -> torch.Tensor:
        """Gradients of the local shard into the flat buffer (all-reduce started, not yet waited).  Returns the
        device tensor {loss, rec_loss, vel_loss} [3] of the local shard."""
        from . import ops, training
        m = self.model
        now = frozenset(n for n, p in m.named_parameters() if p.requires_grad)
        if now != self._requires_grad:
            diff = sorted(now ^ self._requires_grad)
            raise L.A2FError(f"FaceformerTrainer: the set of trainable parameters changed after construction ({len(diff)} "
                             f"parameters, e.g. {diff[0]}); freeze before constructing the trainer, or build a new one")
        audio = audio.contiguous().float()
        B = audio.shape[0]
        one_hot = one_hot.reshape(B, -1).contiguous().float()
        tmpl = template.reshape(B, -1).contiguous().float()
        self.flat.zero_grads()
        self._skipped_stages = frozenset()
        hook = (lambda st: self.flat.all_reduce_stage(st, self.group)) if (self.overlap and _world() > 1) else None
        T = audio.shape[1] * self.fps // 16000
        if m.precision == "bf16" and T >= 2 and T % 2 == 0:
            # tensor-core path, even clip length: the vertex head runs with the losses fused into its epilogue
            # (a2f_vertex_head_loss): gt is read once, dL/dy leaves as bf16 in the layout the backward GEMMs read, the
            # 60 KB/frame prediction is never written.  (Odd clips drop their last frame from the loss, ref loss.py:12-15,
            # and take the unfused path below.)
            with torch.no_grad():
                _, tape = training.forward_train(m, audio, one_hot, tmpl, self.fps, with_head=False)
                self._note_skips(tape)
                V3, M = m.vertice_dim, B * T
                g = gt.reshape(M, V3)
                if g.dtype != torch.float32 or not g.is_contiguous():
                    g = g.contiguous().float()
                if self._dy is None or tuple(self._dy.shape) != (M, training.V3PAD):
                    self._dy = torch.zeros((M, training.V3PAD), dtype=torch.bfloat16, device=audio.device)   # pad columns stay 0
                if self._ws_head is None:
                    n = L.load().a2f_vertex_head_loss_workspace_bytes()
                    self._ws_head = torch.empty((n + 7) // 8, dtype=torch.float64, device=audio.device)
                z3 = ops.split_bf16x3(tape["D"].view(M, 64), False)
                out3 = ops.vertex_head_loss(z3, m._head_operand(m.vertice_map_r.weight, 64), m.vertice_map_r.bias.detach(), tmpl, T,
                                            g, self._dy, 1.0, 10.0, ws=self._ws_head)
                training.backward(m, tape, None, on_ready=hook, dYb=self._dy)
            return out3
        with torch.no_grad():
            out, tape = training.forward_train(m, audio, one_hot, tmpl, self.fps)
            self._note_skips(tape)
            T, V3 = out.shape[1], m.vertice_dim
            Te = T - (T % 2)                                  # ref loss.py:12-15: an odd last frame is dropped
            if Te < 2:
                raise L.A2FError("FaceFormerLoss needs at least two frames")
            pred = out.view(B, T, V3)
            g = gt.reshape(B, -1, V3)
            if Te != T:
                pred_l, g_l = pred[:, :Te].contiguous(), g[:, :Te].contiguous().float()
            else:
                pred_l, g_l = pred, g.contiguous().float()
            rows = B * Te
            if self._ws is None:
                self._ws = ops.loss_workspace(audio.device)
            out3 = ops.voca_loss_fwd(pred_l.view(rows, V3), g_l.view(rows, V3), rows, V3, 1.0, 10.0, self._ws)
            dpred = torch.empty((B, Te, V3), dtype=torch.float32, device=audio.device)
            ops.voca_loss_bwd(pred_l.view(rows, V3), g_l.view(rows, V3), rows, V3, 1.0, 10.0, None, dpred.view(rows, V3))
            if Te != T:
                dfull = torch.zeros((B, T, V3), dtype=torch.float32, device=audio.device)
                dfull[:, :Te] = dpred
                dpred = dfull
            training.backward(m, tape, dpred, on_ready=hook)
        return out3

    def _note_skips(self, tape) -> None:
        from . import training
        drop = tape.get("drop")
        if drop and drop["skip"]:
            self._skipped_stages = frozenset(training.grad_stage_of(f"audio_encoder.encoder.layers.{l}.") for l in drop["skip"])

    def _adam_per_stage(self) -> None:
        """Adam over the stages that received gradients, each run of consecutive stages with equal step counts in one
        launch (eager only: the counts are host-side)."""
        from . import ops
        n = len(self.flat.stage_ranges)
        if self._stage_steps is None:
            self._stage_steps = [self.steps - 1] * n
        g = self.flat.reduced_grads()
        runs = []
        for st in range(n):
            if st in self._skipped_stages:
                continue
            self._stage_steps[st] += 1
            if runs and runs[-1][1] == st - 1 and self._stage_steps[runs[-1][0]] == self._stage_steps[st]:
                runs[-1][1] = st
            else:
                runs.append([st, st])
        for s0, s1 in runs:
            lo, hi = self.flat.stage_ranges[s0][0], self.flat.stage_ranges[s1][1]
            if hi > lo:
                ops.adam_step(self.flat.params[lo:hi], g[lo:hi], self.exp_avg[lo:hi], self.exp_avg_sq[lo:hi], self.lr,
                              self.betas[0], self.betas[1], self.eps, self.weight_decay, self._stage_steps[s0],
                              grad_scale=1.0 / _world())

    def optimizer_step(self) -> None:
        from . import ops
        self.flat.finish_all_reduce(self.group)
        self.steps += 1
        if self._skipped_stages or self._stage_steps is not None:
            # LayerDrop skipped a layer (now or earlier): per-parameter step counts differ, as in torch.optim.Adam
            self._step_dev.add_(1)
            self._adam_per_stage()
            self.flat.bump_versions()
            return
        # the step count lives on the device (incremented on the stream) so that the whole step can be replayed as a graph
        self._step_dev.add_(1)
        ops.adam_step(self.flat.params, self.flat.reduced_grads(), self.exp_avg, self.exp_avg_sq, self.lr, self.betas[0],
                      self.betas[1], self.eps, self.weight_decay, self._step_dev, grad_scale=1.0 / _world())
        self.flat.bump_versions()

    def wire_description(self) -> str:
        f = self.flat
        mb = f.total * (2 if f.wire == "bf16" else 4) / 1e6
        return (f"{len(f.buckets)} NCCL all-reduce buckets per step (stages {f.buckets}), {f.wire} on the wire = {mb:.0f} MB, "
                "started from inside the backward; 1/world folded into the fused Adam kernel")

    def step(self, audio, one_hot, template, gt) -> Dict[str, torch.Tensor]:
        out3 = self.forward_backward(audio, one_hot, template, gt)
        self.optimizer_step()
        return {"loss": out3[0], "rec_loss": out3[1], "vel_loss": out3[2]}

    def training_step(self, batch: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """batch keys as produced by the reference's dataset (ref:src/dataset/vocaset.py:72-77)."""
        verts, tmpl = batch["verts"] * 100, batch["template_vert"] * 100        # ref lightning_model.py:145-148
        return self.step(batch["audio"], batch["one_hot"], tmpl, verts)

    def graphed(self, audio, one_hot, template, gt) -> "GraphedTrainStep":
        """Capture one whole optimisation step for these shapes as a CUDA graph (see GraphedTrainStep)."""
        return GraphedTrainStep(self, audio, one_hot, template, gt)


class GraphedTrainStep:
    """One FaceformerTrainer.step -- weight re-packing, forward, fused head + loss, backward, the bucketed gradient
    all-reduce and the fused Adam update -- captured as ONE CUDA graph for fixed shapes.  A step is ~330 launches of mostly
    small kernels; replaying the graph takes the Python / ctypes launch path (15-25 us per launch on the host) off the
    critical path.  Call it like `step`: inputs are copied into the captured buffers; the returned loss tensors are the
    captured outputs (overwritten by the next replay).  Requirements: no host-side draw inside the step (SpecAugment and
    LayerDrop off; encoder dropout is fine, each replay draws fresh masks) and shapes equal to the captured ones."""

    def __init__(self, trainer: "FaceformerTrainer", audio, one_hot, template, gt, warmup: int = 2):
        from . import training
        if training.spec_augment_active(trainer.model):
            raise L.A2FError("GraphedTrainStep: SpecAugment draws its mask on the host every step; capture needs it off")
        m = trainer.model
        if training.encoder_dropout_active(m) and float({**training.DROPOUT_DEFAULTS, **(m.dropout_p or {})}["layerdrop"]) > 0:
            raise L.A2FError("GraphedTrainStep: LayerDrop draws the skipped layers on the host every step; capture needs "
                             "dropout_p['layerdrop'] = 0 (dropout alone is captured: its offset advances on the device)")
        if trainer._stage_steps is not None:
            raise L.A2FError("GraphedTrainStep: LayerDrop left per-stage Adam step counts; capture needs a trainer that never "
                             "skipped a layer")
        self.trainer = trainer
        self.static_in = [audio.clone(), one_hot.clone(), template.clone(), gt.clone()]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):          # allocator pools, packed-operand caches, NCCL channels
                trainer.step(*self.static_in)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        n0 = L.load().a2f_launch_count()
        with torch.cuda.graph(self.graph):
            self.static_out = trainer.step(*self.static_in)
        self.launches_per_replay = int(L.load().a2f_launch_count() - n0)

    def __call__(self, audio, one_hot, template, gt) -> Dict[str, torch.Tensor]:
        for dst, src in zip(self.static_in, (audio, one_hot, template, gt)):
            if dst.data_ptr() != src.data_ptr():
                dst.copy_(src, non_blocking=True)
        self.graph.replay()
        self.trainer.steps += 1                      # host-side bookkeeping; the Adam kernel reads the device-side counter
        return self.static_out


class ConvModelTrainer:
    """Training step of the convolutional models (Voca / Audio2Mesh / Song2Face) with an optional feature extractor in front:
    the reference's default configuration (ref:config.yaml: modelname audio2mesh, feature_extractor mfcc, batch 128)
    as Lightning runs it (ref:src/model/lightning_model.py:111-117 forward, :145-161 training_step, :209-213 Adam).

    One process per GPU; parameters / gradients / Adam moments in flat fp32 buffers, one all-reduce of the whole
    gradient (2.2 M floats for Audio2Mesh) and the fused Adam kernel.  BatchNorm statistics stay per replica (the
    reference has no SyncBN).

    freeze_bn=True puts every nn.BatchNorm2d in eval() after model.train(): the fine-tuning recipe that normalises with
    the running statistics and keeps them unchanged (conv_training._bn_fwd).  Parameters with requires_grad False (e.g.
    frozen BatchNorm affines) are not trained."""

    def __init__(self, model, feature_extractor=None, lr: float = 1e-4, weight_decay: Optional[float] = None,
                 betas=(0.9, 0.999), eps: float = 1e-8, group=None, freeze_bn: bool = False):
        from . import modules
        if not next(model.parameters()).is_cuda:
            raise L.A2FError("ConvModelTrainer runs on CUDA (sm_100a) only; there is no CPU fallback")
        self.model, self.feature_extractor = model.train(), feature_extractor
        if freeze_bn:
            for mod in model.modules():
                if isinstance(mod, torch.nn.BatchNorm2d):
                    mod.eval()
        self.loss = modules.VocaLoss()
        self.lr = float(lr)
        self.weight_decay = float(lr / 10 if weight_decay is None else weight_decay)
        self.betas, self.eps, self.group = betas, float(eps), group
        self.flat = FlatBuffers(model.named_parameters(), lambda name: 0, 1)
        self.exp_avg = torch.zeros_like(self.flat.params)
        self.exp_avg_sq = torch.zeros_like(self.flat.params)
        self.steps = 0
        self.flat.broadcast_params(0, group)
        self.flat.bump_versions()

    def step(self, x, one_hot, template, gt) -> Dict[str, torch.Tensor]:
        from . import ops
        self.flat.zero_grads()
        with torch.no_grad():
            feat = self.feature_extractor(x).detach() if self.feature_extractor is not None else x
        with torch.enable_grad():
            out = self.loss(self.model(feat, one_hot, template), gt)
            out["loss"].backward()
        self.flat.finish_all_reduce(self.group)
        self.steps += 1
        ops.adam_step(self.flat.params, self.flat.grads, self.exp_avg, self.exp_avg_sq, self.lr, self.betas[0], self.betas[1],
                      self.eps, self.weight_decay, self.steps, grad_scale=1.0 / _world())
        self.flat.bump_versions()
        return {k: v.detach() for k, v in out.items()}

    def training_step(self, batch: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        verts, tmpl = batch["verts"] * 100, batch["template_vert"] * 100        # ref lightning_model.py:145-148
        return self.step(batch["audio"], batch["one_hot"], tmpl, verts)
