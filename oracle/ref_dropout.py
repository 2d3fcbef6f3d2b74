"""TEST INFRASTRUCTURE -- CPU restatement of FaceFormer's training step with the wav2vec2 encoder in TRAIN-mode dropout
(HF modeling_wav2vec2.py, post-LN layers, as reached through ref:src/model/wav2vec.py:147-180), under GIVEN masks.

The masks come from oracle/philox.py (the RNG contract of include/a2f.h), so this reproduces the arithmetic of the
sm_100a training step with `encoder_dropout=True`.  Sites (drop(x) = keep ? x / (1 - p) : 0):
    feat_proj   h0  = drop(LN(x) Wp^T + bp)                       (before SpecAugment)
    enc_in      h   = drop(LN(h0 + gelu(posconv(h0))))
    attn_prob   att = drop(softmax(Q K^T / 8)) V
    attn_out    h1  = LN(h + drop(att Wo^T + bo))
    ffn_act     f   = drop(gelu(h1 W1^T + b1))
    ffn_out     h'  = LN(h1 + drop(f W2^T + b2))
    LayerDrop   a skipped layer is the identity (its masks are None in the mask set)
Everything else is oracle/ref_models.py unchanged (decoder and PPE dropout stay off).
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

from . import philox
from . import ref_models as orm


def _drop(x: torch.Tensor, keep: np.ndarray, p: float) -> torch.Tensor:
    if p == 0:
        return x
    k = torch.as_tensor(keep, dtype=torch.bool).view(x.shape)
    return torch.where(k, x * float(philox.scale(p)), torch.zeros((), dtype=x.dtype))


def encoder(sd, h: torch.Tensor, drop: Dict) -> torch.Tensor:
    """oracle/ref_models.encoder for one utterance [1,T,768] with the masks of philox.utterance()."""
    e = "audio_encoder.encoder."
    ph, pa, pt = drop["p"].get("hidden", 0.0), drop["p"].get("activation", 0.0), drop["p"].get("attention", 0.0)
    pos = F.conv1d(h.transpose(1, 2), orm.pos_conv_weight(sd), sd[e + "pos_conv_embed.conv.bias"], padding=64, groups=16)
    pos = F.gelu(pos[:, :, :-1]).transpose(1, 2)
    h = h + pos
    h = F.layer_norm(h, (768,), sd[e + "layer_norm.weight"], sd[e + "layer_norm.bias"], 1e-5)
    h = _drop(h, drop["enc_in"], ph)
    B, T, _ = h.shape
    for l in range(12):
        dl = drop["layers"][l]
        if dl is None:                                                   # LayerDrop
            continue
        p = e + f"layers.{l}."
        q = F.linear(h, sd[p + "attention.q_proj.weight"], sd[p + "attention.q_proj.bias"]).view(B, T, 12, 64).transpose(1, 2)
        k = F.linear(h, sd[p + "attention.k_proj.weight"], sd[p + "attention.k_proj.bias"]).view(B, T, 12, 64).transpose(1, 2)
        v = F.linear(h, sd[p + "attention.v_proj.weight"], sd[p + "attention.v_proj.bias"]).view(B, T, 12, 64).transpose(1, 2)
        w = _drop(torch.softmax(torch.matmul(q, k.transpose(2, 3)) * (64 ** -0.5), dim=-1), dl["attn_prob"], pt)
        a = torch.matmul(w, v).transpose(1, 2).reshape(B, T, 768)
        a = F.linear(a, sd[p + "attention.out_proj.weight"], sd[p + "attention.out_proj.bias"])
        h = F.layer_norm(h + _drop(a, dl["attn_out"], ph), (768,), sd[p + "layer_norm.weight"], sd[p + "layer_norm.bias"], 1e-5)
        f = F.gelu(F.linear(h, sd[p + "feed_forward.intermediate_dense.weight"], sd[p + "feed_forward.intermediate_dense.bias"]))
        f = _drop(f, dl["ffn_act"], pa)
        f = F.linear(f, sd[p + "feed_forward.output_dense.weight"], sd[p + "feed_forward.output_dense.bias"])
        h = F.layer_norm(h + _drop(f, dl["ffn_out"], ph), (768,), sd[p + "final_layer_norm.weight"],
                         sd[p + "final_layer_norm.bias"], 1e-5)
    return h


def faceformer_forward(sd, audio: torch.Tensor, one_hot: torch.Tensor, template: torch.Tensor, fps: int,
                       drop: Dict) -> torch.Tensor:
    """oracle/ref_models.faceformer_forward for one utterance (no SpecAugment) with the encoder masks `drop`."""
    frame_num = audio.shape[1] * fps // 16000
    audio_n = orm.processor_normalize(audio.squeeze(0))[None]
    template = template.reshape(1, 1, -1)
    h = orm.feature_extractor(sd, audio_n).transpose(1, 2)
    h = orm.linear_interpolation(h, frame_num)
    h = orm.feature_projection(sd, h)
    h = _drop(h, drop["feat_proj"], drop["p"].get("feat_proj", 0.0))
    hs = encoder(sd, h, drop)
    memory = F.linear(hs, sd["audio_feature_map.weight"], sd["audio_feature_map.bias"])
    vertice_out = orm.faceformer_decode(sd, memory, one_hot, frame_num)
    return (vertice_out + template).view(1, frame_num, -1, 3)


def faceformer_loss_and_grads(sd, audio, one_hot, template, gt, fps: int = 60, drop: Optional[Dict] = None
                              ) -> Tuple[Dict[str, float], Dict[str, torch.Tensor]]:
    """oracle/ref_train.faceformer_loss_and_grads with the batch masks of philox.encoder_dropout_masks() (sliced per
    utterance by global batch index; None = every p zero).  Parameters that received no gradient (LayerDrop) map to
    None."""
    params = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and k != "PPE.pe" else v)
              for k, v in sd.items()}
    B = audio.shape[0]
    tot = {"loss": 0.0, "rec_loss": 0.0, "vel_loss": 0.0}
    loss_sum = None
    with torch.enable_grad():
        for b in range(B):
            d = philox.utterance(drop, b) if drop is not None else _NO_DROP
            out = faceformer_forward(params, audio[b:b + 1], one_hot[b:b + 1], template[b:b + 1], fps, d)
            l = orm.faceformer_loss(out, gt[b:b + 1])
            for k in tot:
                tot[k] += float(l[k]) / B
            loss_sum = l["loss"] if loss_sum is None else loss_sum + l["loss"]
        (loss_sum / B).backward()
    grads = {k: p.grad for k, p in params.items() if isinstance(p, torch.Tensor) and p.requires_grad}
    return tot, grads


_NO_DROP = {"p": {}, "feat_proj": None, "enc_in": None, "layers": [{"attn_prob": None, "attn_out": None, "ffn_act": None, "ffn_out": None}] * 12}
