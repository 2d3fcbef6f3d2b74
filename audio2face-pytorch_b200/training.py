"""FaceFormer training step on the sm_100a kernels: the forward that keeps what the backward needs, and the explicit
backward pass (ref: torch.autograd over ref:src/model/faceformer.py:139-188 + HF Wav2Vec2Model inside Lightning's
training_step, ref:src/model/lightning_model.py:150-161).

Semantics: eval-mode arithmetic by default (dropout and LayerDrop are inactive -- stated in DESIGN.md).  With
`model.encoder_dropout = True` a training forward in train() mode applies the wav2vec2 encoder's dropout sites and
LayerDrop (see encoder_dropout_active); its masks follow the RNG contract of include/a2f.h, so oracle/philox.py can
regenerate them exactly.  SpecAugment, whose randomness is host-side numpy in
the reference, is available with `model.spec_augment = True` and reproduces the reference's masks draw for draw
(spec_augment.py).  Every parameter of the reference receives a gradient; `audio_encoder.masked_spec_embed` only with
SpecAugment on (same in the reference: unused otherwise, SURVEY.md App. B.2).  Parameter gradients are ACCUMULATED into `param.grad` (allocated as zeros when
missing), exactly where torch.optim / a flat-buffer trainer expects them.

precision "fp32": true-fp32 SIMT GEMMs everywhere (the tight-tolerance parity path);
precision "bf16": tcgen05 GEMMs for forward, data gradients (W^T operands) and weight gradients (MN-major operands
read in place), bf16 activations / activation gradients, fp32 LayerNorm / softmax statistics, fp32 decoder, fp32
parameter gradients.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np
import torch

from . import lib as L
from . import ops
from . import spec_augment

GELU = L.ACT_GELU
V3PAD = 15072          # 15069 rounded up to a multiple of 8 (16-byte bf16 rows for TMA)


_WARNED_DROPOUT = False

# wav2vec2 encoder dropout (modules.Faceformer.dropout_p): the 960h checkpoint config the reference loads
DROPOUT_DEFAULTS = {"hidden": 0.1, "attention": 0.1, "activation": 0.1, "feat_proj": 0.1, "layerdrop": 0.1}
N_ENC_LAYERS = 12
_RANK_MIX = 0x9E3779B97F4A7C15          # replicas' Philox keys: seed ^ (rank * _RANK_MIX) mod 2^64
_GRAD_SINK = None      # set by collect_grads(): id(param) -> buffer the explicit backward accumulates into instead of .grad


def _grad(p: torch.nn.Parameter) -> torch.Tensor:
    """Where the explicit backward accumulates dL/dp: the parameter's .grad (allocated as zeros when missing -- the flat
    gradient buffer under trainer.FlatBuffers), or the sink of an enclosing collect_grads()."""
    if _GRAD_SINK is not None:
        _GRAD_SINK.touched.add(id(p))
        return _GRAD_SINK.bufs[id(p)]
    if p.grad is None:
        p.grad = torch.zeros_like(p, memory_format=torch.contiguous_format)
    return p.grad


class collect_grads:
    """Context manager for the torch.autograd glue: inside it the explicit backward writes every parameter gradient into
    views of ONE fresh zero-filled flat buffer (parameters in the order given, each on a 256-byte boundary, so the fused
    q|k|v weight-gradient GEMM still applies) instead of touching `.grad`.  `grads()` then hands them to autograd as the
    Function's outputs: AccumulateGrad (and with it torch DDP's reducer hooks, Lightning's gradient clipping, hooks
    registered by the user) sees them exactly as it sees the reference's gradients."""

    def __init__(self, params, order_key=None):
        self.params = list(params)
        self.touched = set()
        order = sorted(range(len(self.params)), key=(lambda i: (order_key(i), i)) if order_key else None)
        offs, off = {}, 0
        for i in order:
            offs[i] = off
            off += (self.params[i].numel() + 63) // 64 * 64
        dev = self.params[0].device if self.params else None
        self.flat = torch.zeros(off, dtype=torch.float32, device=dev)
        self.bufs = {id(p): self.flat[offs[i]:offs[i] + p.numel()].view(p.shape) for i, p in enumerate(self.params)}

    def __enter__(self):
        global _GRAD_SINK
        if _GRAD_SINK is not None:
            raise L.A2FError("nested backward passes are not supported")
        _GRAD_SINK = self
        return self

    def __exit__(self, *exc):
        global _GRAD_SINK
        _GRAD_SINK = None
        return False

    def grads(self):
        """One entry per parameter: its gradient, or None when the backward never wrote it / it does not require grad."""
        return tuple(self.bufs[id(p)] if (id(p) in self.touched and p.requires_grad) else None for p in self.params)


def encoder_dropout_active(model) -> bool:
    """Encoder dropout / LayerDrop run in a training forward when `model.encoder_dropout` is True and the module is in
    train() mode.  A no-grad forward (Faceformer.forward under torch.no_grad) is the inference path and keeps eval
    arithmetic either way."""
    return bool(getattr(model, "encoder_dropout", False)) and model.training


def _i64(v: int) -> int:
    v &= (1 << 64) - 1
    return v - (1 << 64) if v >= 1 << 63 else v


def dropout_key(seed: int, rank: int = 0) -> int:
    """64-bit Philox key of a replica: the seed itself on rank 0, so replicas draw independent masks."""
    return (int(seed) ^ (int(rank) * _RANK_MIX)) & ((1 << 64) - 1)


def _dropout_state(model, dev) -> torch.Tensor:
    """The model's device int64 {key, offset}, plus the host generator of the LayerDrop draws (seeded with the seed alone,
    so every replica skips the same layers without a collective).  Created at first use (seed drawn from torch's default
    generator when model.dropout_seed is None); a new model.dropout_seed starts a new stream (offset 0, generator
    reseeded), a new rank a new key, and a device move carries the offset over."""
    if getattr(model, "dropout_seed", None) is None:
        model.dropout_seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    seed, rank = int(model.dropout_seed), getattr(model, "_dropout_rank", 0)
    st, meta = getattr(model, "_drop_state", None), getattr(model, "_drop_meta", None)
    if st is not None and meta == (seed, rank, dev):
        return st
    offset = 0
    if st is not None and meta[0] == seed:
        offset = int(st[1])                      # same stream on a new device or under a new rank
    else:
        model._layerdrop_gen = torch.Generator().manual_seed(seed)
    st = torch.tensor([_i64(dropout_key(seed, rank)), offset], dtype=torch.int64, device=dev)
    model._drop_state, model._drop_meta = st, (seed, rank, dev)
    return st


def set_dropout_rank(model, rank: int) -> None:
    """Fold the data-parallel rank into the model's dropout key (FaceformerTrainer does this at construction)."""
    model._dropout_rank = int(rank)


def _draw_layerdrop(model, p: float) -> frozenset:
    """Layers skipped by this forward: one host uniform per layer, like HF's `torch.rand([]) < layerdrop`."""
    if p <= 0:
        return frozenset()
    u = torch.rand(N_ENC_LAYERS, generator=model._layerdrop_gen)
    return frozenset(i for i in range(N_ENC_LAYERS) if float(u[i]) < p)


def _dropout_plan(model, dev) -> Optional[Dict]:
    """Snapshot (seed, offset) for this forward and its backward, advance the model's offset on the stream, draw
    LayerDrop.  None when encoder dropout is off."""
    if not encoder_dropout_active(model):
        return None
    p = dict(DROPOUT_DEFAULTS)
    p.update(getattr(model, "dropout_p", None) or {})
    for k, v in p.items():
        if not 0.0 <= float(v) < 1.0:
            raise L.A2FError(f"dropout_p[{k!r}] = {v} must lie in [0, 1)")
    st = _dropout_state(model, dev)
    so = st.clone()
    st[1:].add_(1)
    return {"so": so, "hidden": float(p["hidden"]), "activation": float(p["activation"]), "attention": float(p["attention"]),
            "feat_proj": float(p["feat_proj"]), "skip": _draw_layerdrop(model, float(p["layerdrop"]))}


def conv_lengths(n_samples: int) -> List[int]:
    Ls = [(n_samples - 10) // 5 + 1]
    for k in (3, 3, 3, 3, 2, 2):
        Ls.append((Ls[-1] - k) // 2 + 1)
    return Ls


# ---------------------------------------------------------------------------------------------------------------
# derived weights of the backward pass (W^T operands); rebuilt when a parameter changes, never saved
# ---------------------------------------------------------------------------------------------------------------
def packed_backward_weights(model) -> Dict:
    bf = model.precision == "bf16"
    dt = torch.bfloat16 if bf else torch.float32
    ae = model.audio_encoder

    def build():
        dev = model.audio_feature_map.weight.device
        plan = ops.PackPlan(dev)
        new = lambda *shape: torch.empty(shape, dtype=dt, device=dev)                # noqa: E731

        def T_(w, dtype=None):                                                       # [N,K] -> [K,N]
            w = w.detach()
            o = torch.empty((w.shape[1], w.shape[0]), dtype=dtype or dt, device=dev)
            plan.transpose(w, o)
            return o

        P = {}
        convs = []
        cl = ae.feature_extractor.conv_layers
        for i, k in zip(range(1, 7), (3, 3, 3, 3, 2, 2)):
            w = cl[i].conv.weight.detach()                           # [co, ci, k]
            if k == 3:
                even = new(512, 1024)                                # [ci, (tap2 co | tap0 co)]
                plan.transpose(w, even, ldo=1024, dst_off=0, R=512, Cc=512, ld_r=1536, ld_c=3, src_off=2)
                plan.transpose(w, even, ldo=1024, dst_off=512, R=512, Cc=512, ld_r=1536, ld_c=3, src_off=0)
                odd = new(512, 512)
                plan.transpose(w, odd, R=512, Cc=512, ld_r=1536, ld_c=3, src_off=1)
                convs.append((even, odd))
            else:
                both = new(1024, 512)                                # [(tap, ci), co]
                plan.transpose(w, both, ldo=512, dst_off=0, R=512, Cc=512, ld_r=1024, ld_c=2, src_off=0)
                plan.transpose(w, both, ldo=512, dst_off=512 * 512, R=512, Cc=512, ld_r=1024, ld_c=2, src_off=1)
                convs.append((both,))
        P["convs"] = convs
        P["proj_t"] = T_(ae.feature_projection.projection.weight)             # [512,768]
        pz = ae.encoder.pos_conv_embed.conv.parametrizations.weight
        _, pshape = ops.posconv_weight_shape(dt)
        P["pos_fwd"], P["pos_bwd"] = new(*pshape), new(*pshape)
        lay = []
        for blk in ae.encoder.layers:
            a = blk.attention
            qkv_t = new(768, 2304)
            for j, lin in enumerate((a.q_proj, a.k_proj, a.v_proj)):
                plan.transpose(lin.weight.detach(), qkv_t, ldo=2304, dst_off=768 * j)
            lay.append({"qkv_t": qkv_t, "o_t": T_(a.out_proj.weight),
                        "f1_t": T_(blk.feed_forward.intermediate_dense.weight),     # [768,3072]
                        "f2_t": T_(blk.feed_forward.output_dense.weight)})          # [3072,768]
        P["layers"] = lay
        P["afm_t"] = T_(model.audio_feature_map.weight)                              # [768,64]
        wr = model.vertice_map_r.weight.detach()                                     # [15069,64]
        if bf:
            wr_t = torch.zeros((64, V3PAD), dtype=dt, device=dev)
            plan.transpose(wr, wr_t, ldo=V3PAD)
        else:
            wr_t = new(64, wr.shape[0])                                              # [64,15069]
            plan.transpose(wr, wr_t)
        P["head_t"] = wr_t
        d = model.transformer_decoder.layers[0]
        P["ca_out_t"] = T_(d.multihead_attn.out_proj.weight, torch.float32)
        P["ca_v_t"] = torch.empty((64, 64), dtype=torch.float32, device=dev)
        plan.transpose(d.multihead_attn.in_proj_weight.detach(), P["ca_v_t"], R=64, Cc=64, ld_r=64, src_off=128 * 64)
        plan.finalize()
        P["_plan"] = plan

        def refresh():
            plan.run()
            ops.pack_posconv_weights_train(pz.original0.detach().reshape(-1), pz.original1.detach(), dt,
                                           out=(P["pos_fwd"], P["pos_bwd"]))

        P["_refresh"] = refresh
        refresh()
        return P

    srcs = list(model.parameters())
    return model._cache.get("ffbwd_" + model.precision, srcs, build)


# ---------------------------------------------------------------------------------------------------------------
# forward with tape
# ---------------------------------------------------------------------------------------------------------------
def forward_train(model, audio: torch.Tensor, one_hot: torch.Tensor, tmpl: torch.Tensor, fps: int, with_head: bool = True):
    """Same arithmetic as Faceformer.forward; returns (out [B,T,5023,3] fp32, tape).  with_head=False stops at the decoder
    states (tape["D"]) and returns out = None: the caller runs the vertex head fused with the loss (ops.vertex_head_loss)."""
    global _WARNED_DROPOUT
    if model.training and not _WARNED_DROPOUT:
        # the reference's train() mode also enables dropout 0.1 (PPE, decoder layer, wav2vec2 hidden / activation / attention)
        # and LayerDrop 0.1.  Said once, loudly, because a drop-in must not hide what is missing.
        import warnings
        if encoder_dropout_active(model):
            msg = ("a2f_b200 Faceformer in train() mode with encoder_dropout: SpecAugment and the wav2vec2 encoder's dropout "
                   "and LayerDrop are applied, but the decoder / PPE dropout is NOT (INTEGRATION.md 2c)")
        else:
            msg = ("a2f_b200 Faceformer in train() mode: SpecAugment is applied like the reference's, but dropout (p=0.1) and "
                   "LayerDrop are NOT -- the training kernels run eval-mode arithmetic for those ops unless "
                   "model.encoder_dropout is set (INTEGRATION.md 2c)")
        warnings.warn(msg, RuntimeWarning, stacklevel=3)
        _WARNED_DROPOUT = True
    P = model._packed()
    bf = model.precision == "bf16"
    dt = torch.bfloat16 if bf else torch.float32
    be = model._backend()
    ae = model.audio_encoder
    B, N = audio.shape
    T = N * fps // 16000
    dev = audio.device
    tp: Dict = {"B": B, "N": N, "T": T, "audio": audio, "one_hot": one_hot}
    drop = _dropout_plan(model, dev)
    tp["drop"] = drop
    ph = drop["hidden"] if drop else 0.0
    pa = drop["activation"] if drop else 0.0

    stats = ops.audio_stats(audio)
    gn = ae.feature_extractor.conv_layers[0].layer_norm
    a0, ws0 = ops.conv0_gn_gelu_train(audio, stats, P["conv0_w"], gn.weight.detach(), gn.bias.detach(), dt)
    tp["stats"], tp["ws0"] = stats, ws0
    A, Z = [a0], [None]
    x, L_in = a0, a0.shape[1]
    for i, k in enumerate((3, 3, 3, 3, 2, 2)):
        L_out = (L_in - k) // 2 + 1
        z = torch.empty((B, L_out, 512), dtype=dt, device=dev)
        y = ops.padded_rows(B, L_out, 512, dt, dev)                               # read by the next layer's wgrad
        if bf and L_out > 128:
            # tensor-core path: ONE launch writes the pre-activation z (kept for the GELU backward) and gelu(z)
            ops.gemm(x, P["convs"][i], z, act=GELU, out2=y, backend=be, M=B * L_out, K=k * 512, a_row_stride=1024,
                     a_batch_stride=L_in * 512, rows_per_batch=L_out, ldc=512)
        else:
            ops.gemm(x, P["convs"][i], z, backend=be, M=B * L_out, K=k * 512, a_row_stride=1024, a_batch_stride=L_in * 512,
                     rows_per_batch=L_out, ldc=512)
            ops.act_fwd(z, GELU, out=y)
        Z.append(z)
        A.append(y)
        x, L_in = y, L_out
    tp["A"], tp["Z"] = A, Z
    fp = ae.feature_projection
    xi = ops.interp_ln(x, fp.layer_norm.weight.detach(), fp.layer_norm.bias.detach(), T, dt)       # [B,T,512]
    M = B * T
    h0 = torch.empty((M, 768), dtype=dt, device=dev)
    ops.gemm(xi.view(M, 512), P["proj_w"], h0, bias=fp.projection.bias.detach(), backend=be)
    if drop and drop["feat_proj"] > 0:
        ops.dropout_apply(h0, drop["feat_proj"], L.DROP_FEAT_PROJ, drop["so"], out=h0)
    if spec_augment_active(model):
        # SpecAugment (ref:src/model/wav2vec.py:149-162): the mask is drawn on the host with the reference's numpy
        # sequence (spec_augment.py), applied and back-propagated by the a2f_spec_mask_* kernels
        mask = spec_augment.time_mask(B, T)
        tp["spec_mask"] = torch.from_numpy(mask.reshape(-1).astype(np.uint8)).to(dev)
        ops.spec_mask_fwd(h0, tp["spec_mask"], ae.masked_spec_embed.detach())
    PB = packed_backward_weights(model)
    pc = ops.posconv_pre(h0, PB["pos_fwd"], ae.encoder.pos_conv_embed.conv.bias.detach(), B, T, be)
    pre = ops.act_fwd(pc, GELU, resid=h0)
    h = torch.empty((M, 768), dtype=dt, device=dev)
    ops.layernorm(pre, ae.encoder.layer_norm.weight.detach(), ae.encoder.layer_norm.bias.detach(), h)
    if ph > 0:
        ops.dropout_apply(h, ph, L.DROP_ENC_IN, drop["so"], out=h)
    tp.update(xi=xi, h0=h0, pc=pc, pre=pre)
    layers = []
    # the dropout sites of a layer run unfused: GEMM + a2f_dropout_apply (+ the separate LayerNorm)
    fuse_ln = bf and getattr(model, "fuse_layernorm", True) and ph == 0
    for li, (blk, W) in enumerate(zip(ae.encoder.layers, P["layers"])):
        if drop and li in drop["skip"]:
            layers.append(None)                   # LayerDrop: the layer is the identity and launches nothing
            continue
        s = {"h_in": h}
        qkv = torch.empty((M, 2304), dtype=dt, device=dev)
        ops.gemm(h, W["qkv_w"], qkv, bias=W["qkv_b"], backend=be)
        att = torch.empty((M, 768), dtype=dt, device=dev)
        lse = torch.empty((B, 12, T), dtype=torch.float32, device=dev)
        att32 = torch.empty((M, 768), dtype=torch.float32, device=dev) if bf else None
        adrop = (drop["attention"], 8 * li + L.DROP_ATTN_PROB, drop["so"]) if drop and drop["attention"] > 0 else None
        ops.mha_lse(qkv, att, lse, B, T, out_f32=att32, dropout=adrop)
        pre1 = torch.empty((M, 768), dtype=dt, device=dev)
        h1 = torch.empty((M, 768), dtype=dt, device=dev)
        if fuse_ln:      # LayerNorm in the GEMM epilogue; the pre-LN sum is written once (bf16) for the backward
            ops.gemm_ln(att, W["o_w"], blk.attention.out_proj.bias.detach(), h, blk.layer_norm.weight.detach(),
                        blk.layer_norm.bias.detach(), h1, pre_out=pre1)
        elif ph > 0:
            ops.gemm(att, W["o_w"], pre1, bias=blk.attention.out_proj.bias.detach(), backend=be)
            ops.dropout_apply(pre1, ph, 8 * li + L.DROP_ATTN_OUT, drop["so"], resid=h, out=pre1)
            ops.layernorm(pre1, blk.layer_norm.weight.detach(), blk.layer_norm.bias.detach(), h1)
        else:
            ops.gemm(att, W["o_w"], pre1, bias=blk.attention.out_proj.bias.detach(), resid=h, backend=be)
            ops.layernorm(pre1, blk.layer_norm.weight.detach(), blk.layer_norm.bias.detach(), h1)
        fpre = torch.empty((M, 3072), dtype=dt, device=dev)
        if bf and M > 128:
            f = torch.empty((M, 3072), dtype=dt, device=dev)
            ops.gemm(h1, W["f1_w"], fpre, bias=blk.feed_forward.intermediate_dense.bias.detach(), act=GELU, out2=f, backend=be)
        else:
            ops.gemm(h1, W["f1_w"], fpre, bias=blk.feed_forward.intermediate_dense.bias.detach(), backend=be)
            f = ops.act_fwd(fpre, GELU)
        if pa > 0:
            ops.dropout_apply(f, pa, 8 * li + L.DROP_FFN_ACT, drop["so"], out=f)
        pre2 = torch.empty((M, 768), dtype=dt, device=dev)
        h = torch.empty((M, 768), dtype=dt, device=dev)
        if fuse_ln:
            ops.gemm_ln(f, W["f2_w"], blk.feed_forward.output_dense.bias.detach(), h1, blk.final_layer_norm.weight.detach(),
                        blk.final_layer_norm.bias.detach(), h, pre_out=pre2)
        elif ph > 0:
            ops.gemm(f, W["f2_w"], pre2, bias=blk.feed_forward.output_dense.bias.detach(), backend=be)
            ops.dropout_apply(pre2, ph, 8 * li + L.DROP_FFN_OUT, drop["so"], resid=h1, out=pre2)
            ops.layernorm(pre2, blk.final_layer_norm.weight.detach(), blk.final_layer_norm.bias.detach(), h)
        else:
            ops.gemm(f, W["f2_w"], pre2, bias=blk.feed_forward.output_dense.bias.detach(), resid=h1, backend=be)
            ops.layernorm(pre2, blk.final_layer_norm.weight.detach(), blk.final_layer_norm.bias.detach(), h)
        s.update(qkv=qkv, att=att, att32=att32, lse=lse, pre1=pre1, h1=h1, fpre=fpre, f=f, pre2=pre2)
        layers.append(s)
    tp["layers"], tp["hs"] = layers, h
    memory = torch.empty((M, 64), dtype=torch.float32, device=dev)
    ops.gemm(h, P["afm_w"], memory, bias=model.audio_feature_map.bias.detach(), backend=be)
    D, dtape = ops.decoder_rollout_train(P["dec"][0], memory, one_hot, model.period, B, T)
    tp["memory"], tp["D"], tp["dtape"] = memory, D, dtape
    if not with_head:
        return None, tp
    out = model._vertex_head(D.view(M, 64), model.vertice_map_r.weight, model.vertice_map_r.bias, tmpl, T, 64)
    return out.view(B, T, -1, 3), tp


# ---------------------------------------------------------------------------------------------------------------
# backward
# ---------------------------------------------------------------------------------------------------------------
def backward(model, tp: Dict, dout: Optional[torch.Tensor], on_ready=None, dYb: Optional[torch.Tensor] = None) -> None:
    """dout: dL/d(out) [B,T,5023,3] fp32 -- or, on the bf16 path, dYb: the same gradient already as bf16 [B*T, V3PAD] with
    zero pad columns (what the fused head + loss epilogue writes).  Accumulates dL/d(parameter) into every parameter's .grad.

    on_ready(stage): called (host side, after the stage's kernels are enqueued) when every gradient of a stage is
    final -- stage 0 = vertex head + decoder + audio_feature_map, 1..12 = encoder layers 11..0, 13 = the rest (the
    front end).  The data-parallel trainer starts that stage's gradient all-reduce from it (see grad_stage_of)."""
    P = model._packed()
    PB = packed_backward_weights(model)
    bf = model.precision == "bf16"
    dt = torch.bfloat16 if bf else torch.float32
    be = model._backend()
    S = L.SIMT_F32
    ae = model.audio_encoder
    B, N, T = tp["B"], tp["N"], tp["T"]
    M = B * T
    V3 = model.vertice_dim
    D = tp["D"].view(M, 64)
    dev = D.device
    dtape = tp["dtape"]
    wr, br = model.vertice_map_r.weight, model.vertice_map_r.bias
    wm, bm = model.vertice_map.weight, model.vertice_map.bias

    # ---- vertex head: Y = D Wr^T + br + template ----
    if dYb is not None:
        if not bf or tuple(dYb.shape) != (M, V3PAD) or dYb.dtype != torch.bfloat16:
            raise L.A2FError("backward: dYb is the bf16 path's [B*T, V3PAD] gradient")
        ops.colsum(dYb, _grad(br), cols=V3)
        dY32 = None
    else:
        dY32 = dout.reshape(M, V3)
        if not dY32.is_contiguous():
            dY32 = dY32.contiguous()
        ops.colsum(dY32, _grad(br))
    gD = torch.empty((M, 64), dtype=torch.float32, device=dev)
    if bf:
        if dYb is None:
            dYb = ops.cast_rows(dY32, torch.bfloat16, V3PAD)
        Db = ops.cast_rows(D, torch.bfloat16, 64)
        ops.gemm_wgrad(dYb, Db, _grad(wr), backend=be, N=V3)
        ops.gemm(dYb, PB["head_t"], gD, backend=be)
        del dYb
    else:
        ops.gemm_wgrad(dY32, D, _grad(wr), backend=S)
        ops.gemm(dY32, PB["head_t"], gD, backend=S)

    # ---- decoder rollout (BPTT) ----
    G = ops.decoder_rollout_bwd(P["dec"][0], dtape, gD, model.period)
    d = model.transformer_decoder.layers[0]
    sa, ca = d.self_attn, d.multihead_attn
    ops.gemm_wgrad(G["GQKV"], dtape.X, _grad(sa.in_proj_weight), backend=S)
    ops.colsum(G["GQKV"], _grad(sa.in_proj_bias))
    ops.gemm_wgrad(G["G1"], dtape.CTX, _grad(sa.out_proj.weight), backend=S)
    ops.colsum(G["G1"], _grad(sa.out_proj.bias))
    ops.gemm_wgrad(G["G3"], dtape.HID, _grad(d.linear2.weight), backend=S)
    ops.colsum(G["G3"], _grad(d.linear2.bias))
    ops.gemm_wgrad(G["GHID"], dtape.Y2, _grad(d.linear1.weight), backend=S)
    ops.colsum(G["GHID"], _grad(d.linear1.bias))
    ops.ln64_param_grad(G["GD"], dtape.Y3PRE, _grad(d.norm3.weight), _grad(d.norm3.bias))
    ops.ln64_param_grad(G["GY2"], dtape.Y2PRE, _grad(d.norm2.weight), _grad(d.norm2.bias))
    ops.ln64_param_grad(G["G2"], dtape.Y1PRE, _grad(d.norm1.weight), _grad(d.norm1.bias))
    # cross-attention under the diagonal memory mask: ca = out_proj(v_proj(mem)) (q/k rows get exact zeros)
    ops.gemm_wgrad(G["G2"], dtape.TMP, _grad(ca.out_proj.weight), backend=S)
    ops.colsum(G["G2"], _grad(ca.out_proj.bias))
    dTMP = torch.empty((M, 64), dtype=torch.float32, device=dev)
    ops.gemm(G["G2"], PB["ca_out_t"], dTMP, backend=S)
    gw, gb = _grad(ca.in_proj_weight), _grad(ca.in_proj_bias)
    ops.gemm_wgrad(dTMP, tp["memory"], gw[128:192], backend=S)
    ops.colsum(dTMP, gb[128:192])
    dMEM = torch.empty((M, 64), dtype=torch.float32, device=dev)
    ops.gemm(dTMP, PB["ca_v_t"], dMEM, backend=S)
    # feedback e_{i+1} = Wc d_i + bc + style,  Wc = Wm Wr,  bc = Wm br + bm
    dWc = torch.zeros((64, 64), dtype=torch.float32, device=dev)
    dbc = torch.zeros((64,), dtype=torch.float32, device=dev)
    ops.gemm_wgrad(G["DEFB"], D, dWc, backend=S, M=M, rows_per_batch=T, dy_batch_stride=T * 64, x_batch_stride=T * 64,
                   x_rows=T, segs=[(-1, 0)])
    ops.colsum(G["DEFB"], dbc)
    gwm = _grad(wm)
    ops.gemm(dWc, wr.detach(), gwm, resid=gwm, backend=S)                             # += dWc Wr^T
    ops.gemm(dbc.view(64, 1), br.detach().view(V3, 1), gwm, resid=gwm, backend=S)     # += dbc br^T
    ops.colsum(G["DEFB"], _grad(bm))
    ops.gemm_wgrad(wm.detach(), dWc, _grad(wr), backend=S)                            # += Wm^T dWc
    ops.gemm_wgrad(wm.detach(), dbc.view(64, 1), _grad(br).view(V3, 1), backend=S)    # += Wm^T dbc
    ops.gemm_wgrad(G["DSTYLE"], tp["one_hot"], _grad(model.obj_vector.weight), backend=S)

    # ---- audio_feature_map ----
    afm = model.audio_feature_map
    ops.colsum(dMEM, _grad(afm.bias))
    dMEMc = ops.cast_rows(dMEM, dt, 64) if bf else dMEM
    ops.gemm_wgrad(dMEMc, tp["hs"], _grad(afm.weight), backend=be)
    dh = torch.empty((M, 768), dtype=dt, device=dev)
    ops.gemm(dMEMc, PB["afm_t"], dh, backend=be)
    if on_ready is not None:
        on_ready(0)

    # ---- encoder layers ----
    # dropout (tp["drop"]): the same a2f_dropout_apply with the forward's (seed, offset) snapshot masks a gradient; the
    # residual branch of a site keeps the unmasked gradient, its Linear (weight, bias, data gradient) gets the masked one
    drop = tp.get("drop")
    ph = drop["hidden"] if drop else 0.0
    pa = drop["activation"] if drop else 0.0
    stage = 0
    n_layers = len(tp["layers"])
    for i, (blk, W, s) in enumerate(zip(reversed(list(ae.encoder.layers)), reversed(PB["layers"]), reversed(tp["layers"]))):
        li = n_layers - 1 - i
        stage += 1
        if s is None:                             # skipped by LayerDrop: no launch, no gradient
            if on_ready is not None:
                on_ready(stage)
            continue
        a, ff = blk.attention, blk.feed_forward
        dpre2 = ops.layernorm_bwd(dh, s["pre2"], blk.final_layer_norm.weight.detach(), _grad(blk.final_layer_norm.weight),
                                  _grad(blk.final_layer_norm.bias), None if ph > 0 else _grad(ff.output_dense.bias))
        g2 = dpre2
        if ph > 0:
            g2 = ops.dropout_apply(dpre2, ph, 8 * li + L.DROP_FFN_OUT, drop["so"])
            ops.colsum(g2, _grad(ff.output_dense.bias))
        ops.gemm_wgrad(g2, s["f"], _grad(ff.output_dense.weight), backend=be)
        dfpre = torch.empty((M, 3072), dtype=dt, device=dev)
        if pa > 0:
            df = torch.empty((M, 3072), dtype=dt, device=dev)
            ops.gemm(g2, W["f2_t"], df, backend=be)
            ops.dropout_apply(df, pa, 8 * li + L.DROP_FFN_ACT, drop["so"], out=df)
            dfpre = ops.act_bwd(df, s["fpre"], GELU)
            del df
        else:
            ops.gemm(g2, W["f2_t"], dfpre, act=GELU, resid=s["fpre"], resid_mode=L.RESID_DACT, backend=be)
        ops.gemm_wgrad(dfpre, s["h1"], _grad(ff.intermediate_dense.weight), backend=be)
        ops.colsum(dfpre, _grad(ff.intermediate_dense.bias))
        dh1 = torch.empty((M, 768), dtype=dt, device=dev)
        ops.gemm(dfpre, W["f1_t"], dh1, resid=dpre2, backend=be)
        dpre1 = ops.layernorm_bwd(dh1, s["pre1"], blk.layer_norm.weight.detach(), _grad(blk.layer_norm.weight),
                                  _grad(blk.layer_norm.bias), None if ph > 0 else _grad(a.out_proj.bias))
        g1 = dpre1
        if ph > 0:
            g1 = ops.dropout_apply(dpre1, ph, 8 * li + L.DROP_ATTN_OUT, drop["so"])
            ops.colsum(g1, _grad(a.out_proj.bias))
        ops.gemm_wgrad(g1, s["att"], _grad(a.out_proj.weight), backend=be)
        datt = torch.empty((M, 768), dtype=dt, device=dev)
        ops.gemm(g1, W["o_t"], datt, backend=be)
        adrop = (drop["attention"], 8 * li + L.DROP_ATTN_PROB, drop["so"]) if drop and drop["attention"] > 0 else None
        dqkv = ops.mha_bwd(s["qkv"], s["att"], datt, s["lse"], B, T, out_f32=s["att32"], dropout=adrop)
        gw = [_grad(lin.weight) for lin in (a.q_proj, a.k_proj, a.v_proj)]
        gb = [_grad(lin.bias) for lin in (a.q_proj, a.k_proj, a.v_proj)]
        if _adjacent(gw):
            # flat gradient buffer (trainer.FlatBuffers orders q | k | v back to back): one fused [2304, 768] GEMM
            ops.gemm_wgrad(dqkv, s["h_in"], gw[0].as_strided((2304, 768), (768, 1)), backend=be)
        else:
            for j in range(3):
                ops.gemm_wgrad(dqkv, s["h_in"], gw[j], backend=be, N=768, dy_offset=768 * j)
        if _adjacent(gb):
            ops.colsum(dqkv, gb[0].as_strided((2304,), (1,)))
        else:
            ops.colsum3(dqkv, gb)
        dh = torch.empty((M, 768), dtype=dt, device=dev)
        ops.gemm(dqkv, W["qkv_t"], dh, resid=dpre1, backend=be)
        if on_ready is not None:
            on_ready(stage)

    # ---- encoder.layer_norm, positional conv, feature projection ----
    if ph > 0:
        ops.dropout_apply(dh, ph, L.DROP_ENC_IN, drop["so"], out=dh)
    dpre = ops.layernorm_bwd(dh, tp["pre"], ae.encoder.layer_norm.weight.detach(), _grad(ae.encoder.layer_norm.weight),
                             _grad(ae.encoder.layer_norm.bias))
    pcv = ae.encoder.pos_conv_embed.conv
    dpc = ops.act_bwd(dpre, tp["pc"], GELU)
    ops.colsum(dpc, _grad(pcv.bias))
    dwp = ops.posconv_wgrad(dpc, tp["h0"], B, T, be)
    pz = pcv.parametrizations.weight
    ops.weight_norm_bwd(dwp, pz.original1.detach(), pz.original0.detach().reshape(-1), _grad(pz.original1),
                        _grad(pz.original0).view(-1))
    dh0 = ops.posconv_dgrad(dpc, PB["pos_bwd"], dpre, B, T, be)
    if tp.get("spec_mask") is not None:
        ops.spec_mask_bwd(dh0, tp["spec_mask"], _grad(ae.masked_spec_embed))
    if drop and drop["feat_proj"] > 0:
        ops.dropout_apply(dh0, drop["feat_proj"], L.DROP_FEAT_PROJ, drop["so"], out=dh0)
    fp = ae.feature_projection
    ops.gemm_wgrad(dh0, tp["xi"].view(M, 512), _grad(fp.projection.weight), backend=be)
    ops.colsum(dh0, _grad(fp.projection.bias))
    dxi = torch.empty((M, 512), dtype=dt, device=dev)
    ops.gemm(dh0, PB["proj_t"], dxi, backend=be)
    A, Z = tp["A"], tp["Z"]
    da6 = ops.interp_ln_bwd(A[6], dxi.view(B, T, 512), fp.layer_norm.weight.detach(), _grad(fp.layer_norm.weight),
                            _grad(fp.layer_norm.bias))
    dz = ops.act_bwd(da6, Z[6], GELU, out_dtype=dt)                       # [B,L6,512]

    # ---- conv stack 6..1 (weight gradient in place on the strided view, data gradient as gather GEMMs) ----
    cl = ae.feature_extractor.conv_layers
    for i, k in zip(range(6, 0, -1), (2, 2, 3, 3, 3, 3)):
        x = A[i - 1]
        L_in, L_out = x.shape[1], dz.shape[1]
        dwp = torch.zeros((512, k * 512), dtype=torch.float32, device=dev)
        ops.gemm_wgrad(dz, x, dwp, backend=be, M=B * L_out, N=512, K=512, dy_row_stride=512, dy_batch_stride=L_out * 512,
                       x_row_stride=1024, x_batch_stride=L_in * 512, rows_per_batch=L_out, x_rows=(L_in + 1) // 2,
                       segs=[(0, 0), (0, 512), (1, 0)][:k])
        ops.add_strided3(dwp, _grad(cl[i].conv.weight), (512, k, 512), (k * 512, 512, 1), (512 * k, 1, k))
        dx = torch.zeros((B, L_in, 512), dtype=dt, device=dev)
        last = i == 1                      # conv0's GELU backward lives in a2f_conv0_bwd (its pre-activation is never stored)
        kw = {} if last else dict(act=GELU, resid=Z[i - 1], resid_mode=L.RESID_DACT, ldr=1024, r_batch_stride=L_in * 512)
        Wd = PB["convs"][i - 1]
        if k == 3:
            U = min(L_out + 1, (L_in + 1) // 2)
            ops.gemm(dz, Wd[0], dx, backend=be, M=B * U, K=1024, N=512, a_row_stride=512, a_batch_stride=L_out * 512,
                     rows_per_batch=U, a_rows=L_out, segs=[(-1, 0), (0, 0)], ldc=1024, c_batch_stride=L_in * 512, **kw)
            kw2 = dict(kw)
            if not last:
                kw2["r_offset"] = 512
            ops.gemm(dz, Wd[1], dx, backend=be, M=B * L_out, K=512, N=512, a_row_stride=512, a_batch_stride=L_out * 512,
                     rows_per_batch=L_out, ldc=1024, c_batch_stride=L_in * 512, c_offset=512, **kw2)
        else:
            ops.gemm(dz, Wd[0], dx, backend=be, M=B * L_out, K=512, N=1024, a_row_stride=512, a_batch_stride=L_out * 512,
                     rows_per_batch=L_out, ldc=1024, c_batch_stride=L_in * 512, **kw)
        dz = dx
    gn = cl[0].layer_norm
    ops.conv0_bwd(tp["audio"], tp["stats"], P["conv0_w"], gn.weight.detach(), gn.bias.detach(), tp["ws0"], dz,
                  _grad(cl[0].conv.weight).view(512, 10), _grad(gn.weight), _grad(gn.bias))
    if on_ready is not None:
        on_ready(N_GRAD_STAGES - 1)


N_GRAD_STAGES = 14
NO_GRAD_PARAMS = ("audio_encoder.masked_spec_embed",)     # unused without SpecAugment: grad is None in the reference too


def spec_augment_active(model) -> bool:
    """SpecAugment runs when `model.spec_augment` is True, or -- left at None -- whenever the module is in train mode: the
    reference applies it under `self.training` (HF config apply_spec_augment=True, mask_time_prob=0.05,
    ref:src/model/wav2vec.py:149-162)."""
    sa = getattr(model, "spec_augment", None)
    return bool(model.training if sa is None else sa)


def no_grad_params(model) -> tuple:
    """Parameters that receive no gradient from backward() for this model configuration."""
    return () if spec_augment_active(model) else NO_GRAD_PARAMS


def grad_stage_of(name: str) -> int:
    """Backward stage (see backward()) in which the gradient of Faceformer parameter `name` becomes final."""
    if name.startswith("audio_encoder.encoder.layers."):
        return 12 - int(name.split(".")[3])
    if name.startswith("audio_encoder."):
        return N_GRAD_STAGES - 1
    return 0


_QKV_RANK = {"attention.q_proj.weight": 0, "attention.k_proj.weight": 1, "attention.v_proj.weight": 2,
             "attention.q_proj.bias": 3, "attention.k_proj.bias": 4, "attention.v_proj.bias": 5}


def grad_order_in_stage(name: str) -> int:
    """Rank of a parameter inside its stage of the flat gradient buffer: q, k, v projection weights first and adjacent
    (then their biases), so that backward() can write all three gradients with ONE [2304, 768] weight-gradient GEMM."""
    for suffix, r in _QKV_RANK.items():
        if name.endswith(suffix):
            return r
    return 6


def _adjacent(ts) -> bool:
    """True when the tensors are contiguous and laid out back to back in one storage (the flat gradient buffer)."""
    for a, b in zip(ts[:-1], ts[1:]):
        if not (a.is_contiguous() and b.is_contiguous()) or a.untyped_storage().data_ptr() != b.untyped_storage().data_ptr() \
                or b.data_ptr() != a.data_ptr() + a.numel() * a.element_size():
            return False
    return True


class FaceformerTrainFn(torch.autograd.Function):
    """Glue to torch.autograd.  Every parameter of the model is an INPUT of the Function and its gradient an output of
    backward(), so AccumulateGrad runs per parameter: `.grad` accumulates like the reference's, and torch DDP (what the
    reference's Lightning Trainer wraps the model in on a multi-GPU box, ref:train.py:48-60) sees every gradient in its
    reducer hooks.  (trainer.FaceformerTrainer is the fast path: flat buffers, bucketed all-reduce started from inside the
    backward, fused Adam -- it calls forward_train / backward directly and never comes through here.)"""

    @staticmethod
    def forward(ctx, model, audio, one_hot, tmpl, fps, *params):
        out, tape = forward_train(model, audio, one_hot, tmpl, fps)
        ctx.model, ctx.tape = model, tape
        return out

    @staticmethod
    def backward(ctx, dout):
        model = ctx.model
        names = {id(p): n for n, p in model.named_parameters()}
        params = list(model.parameters())
        key = lambda i: (grad_stage_of(names[id(params[i])]), grad_order_in_stage(names[id(params[i])]))   # noqa: E731
        with collect_grads(params, key) as sink:
            backward(model, ctx.tape, dout.contiguous().float())
        ctx.tape = None
        return (None, None, None, None, None) + sink.grads()

    @staticmethod
    def run(model, audio, one_hot, tmpl, fps):
        return FaceformerTrainFn.apply(model, audio, one_hot, tmpl, fps, *model.parameters())
