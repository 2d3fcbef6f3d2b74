"""TEST INFRASTRUCTURE -- CPU restatement (oracle) of the Audio2Mesh / Song2Face training step with some BatchNorms
FROZEN: the model in `train()`, the named BatchNorm2d layers put in `eval()` (the usual fine-tuning recipe).  torch's
per-layer rule: a frozen layer normalises with its running statistics and leaves them alone, a training layer uses
batch statistics and updates them.

Only tests/ may import this package.  Every layer is oracle/ref_models.py's (`_bn` with the layer's own train flag,
`lstm_forward`, `voca_loss`); with no layer frozen the forwards are ref_models.audio2mesh_forward(train_bn=True) /
ref_song2face_train.song2face_forward(train_bn=True), with every layer frozen the eval-mode ref_models forwards
(tests/test_frozen_bn.py checks both, and a mixed pattern against the drop-in module's own torch layers).
"""
from __future__ import annotations

from typing import Collection, Dict, Optional

import torch
import torch.nn.functional as F

from . import ref_models as orm

SD = Dict[str, torch.Tensor]

A2M_BN = tuple(f"analysis_net.{3 * i + 1}" for i in range(5)) + tuple(f"articulation_net.{i}" for i in (1, 4, 7, 9, 12))
S2F_BN = tuple(f"vocal_encoder_nn.{i}.1" for i in range(5)) + tuple(f"regression_net.{i}.1" for i in range(3))
BN_PREFIXES = {"audio2mesh": A2M_BN, "song2face": S2F_BN}


def audio2mesh_forward(sd: SD, x: torch.Tensor, one_hot: torch.Tensor, template: torch.Tensor,
                       frozen: Collection[str] = (), running: Optional[SD] = None) -> torch.Tensor:
    """ref:src/model/audio2face.py:57-66 in train mode; the BatchNorms named in `frozen` in eval mode"""
    def bn(prefix, h):
        return orm._bn(sd, prefix, h, prefix not in frozen, running)

    bs = x.size(0)
    emb = one_hot.repeat(1, 32).view(bs, 1, -1, 32)                     # audio2face.py:59
    h = torch.cat((x.unsqueeze(1), emb), 2)                             # audio2face.py:60-62 -> [bs,1,64,32]
    for i in range(5):                                                  # audio2face.py:13-29 conv -> BN -> ReLU
        h = F.conv2d(h, sd[f"analysis_net.{3 * i}.weight"], sd[f"analysis_net.{3 * i}.bias"], stride=(1, 2), padding=(0, 1))
        h = F.relu(bn(f"analysis_net.{3 * i + 1}", h))
    for conv_idx, bn_idx in ((0, 1), (3, 4), (6, 7)):                   # audio2face.py:31-40 conv -> BN -> ReLU
        h = F.conv2d(h, sd[f"articulation_net.{conv_idx}.weight"], sd[f"articulation_net.{conv_idx}.bias"],
                     stride=(2, 1), padding=(1, 0))
        h = F.relu(bn(f"articulation_net.{bn_idx}", h))
    h = bn("articulation_net.9", h)                                     # audio2face.py:41-43 BN -> conv -> ReLU
    h = F.relu(F.conv2d(h, sd["articulation_net.10.weight"], sd["articulation_net.10.bias"], stride=(2, 1), padding=(1, 0)))
    h = bn("articulation_net.12", h)                                    # audio2face.py:44-46
    h = F.relu(F.conv2d(h, sd["articulation_net.13.weight"], sd["articulation_net.13.bias"], stride=(4, 1)))
    return _output_net(sd, h.view(bs, -1), one_hot, template)


def song2face_forward(sd: SD, x: torch.Tensor, one_hot: torch.Tensor, template: torch.Tensor,
                      frozen: Collection[str] = (), running: Optional[SD] = None) -> torch.Tensor:
    """ref:src/model/song2face.py:63-76 in train mode; the BatchNorms named in `frozen` in eval mode"""
    bs = x.size(0)
    emb = one_hot.repeat(1, 32).view(bs, 1, -1, 32)                     # song2face.py:65
    h = torch.cat((x.unsqueeze(1), emb), 2)                             # :66-67 -> [bs,1,64,32]
    for i, (kw, pad) in enumerate(((5, 2), (5, 2), (3, 1), (3, 1), (3, 1))):        # :33-39 conv -> BN -> ReLU
        p = f"vocal_encoder_nn.{i}."
        h = F.conv2d(h, sd[p + "0.weight"], sd[p + "0.bias"], stride=(1, 2), padding=(0, pad))
        h = F.relu(orm._bn(sd, p + "1", h, p + "1" not in frozen, running))
    h = h.squeeze(3)                                                    # :68 -> [bs, 256, 64]
    for name in ("vocal_encoder_lstm1", "vocal_encoder_lstm2"):         # :69-70: 256 steps of 64 / 256 features
        h = orm.lstm_forward(h, sd[name + ".weight_ih_l0"], sd[name + ".weight_hh_l0"], sd[name + ".bias_ih_l0"],
                             sd[name + ".bias_hh_l0"])
    h = F.interpolate(h.unsqueeze(3), size=(32, 1), mode="bilinear")    # :71-72 -> [bs, 256, 32, 1]
    for i in range(4):                                                  # :54-59
        p = f"regression_net.{i}."
        h = F.conv2d(h, sd[p + "0.weight"], sd[p + "0.bias"], stride=(2, 1), padding=(1 if i < 3 else 0, 0))
        if i < 3:
            h = orm._bn(sd, p + "1", h, p + "1" not in frozen, running)
        h = F.relu(h)
    return _output_net(sd, h.squeeze(3).squeeze(2), one_hot, template)  # :74


def _output_net(sd: SD, feat: torch.Tensor, one_hot: torch.Tensor, template: torch.Tensor) -> torch.Tensor:
    """ref:src/model/audio2face.py:49-55,65-66 = ref:src/model/song2face.py:75-76"""
    bs = feat.size(0)
    h = torch.cat((feat, one_hot), 1)
    h = F.linear(h, sd["output_net.0.weight"], sd["output_net.0.bias"])
    h = torch.tanh(F.linear(h, sd["output_net.1.weight"], sd["output_net.1.bias"]))
    h = F.linear(h, sd["output_net.3.weight"], sd["output_net.3.bias"])
    h = F.linear(h, sd["output_net.4.weight"], sd["output_net.4.bias"])
    return h.view(bs, -1, 3) + template


FORWARDS = {"audio2mesh": audio2mesh_forward, "song2face": song2face_forward}


def loss_and_grads(kind: str, sd: SD, x: torch.Tensor, one_hot: torch.Tensor, template: torch.Tensor, gt: torch.Tensor,
                   frozen: Collection[str] = ()):
    """Training step with the BatchNorms named in `frozen` in eval mode (ref:src/model/lightning_model.py:150-161 with
    VocaLoss), the contract of ref_train.conv_loss_and_grads: -> (losses, {param: grad}, running-stat dict after the
    step; the frozen layers' entries unchanged)."""
    params = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and "running_" not in k else v.clone())
              for k, v in sd.items()}
    running = {k: v for k, v in params.items() if "running_" in k or "num_batches" in k}
    with torch.enable_grad():
        out = FORWARDS[kind](params, x, one_hot, template, frozen=frozen, running=running)
        l = orm.voca_loss(out, gt)
        l["loss"].backward()
    grads = {k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in params.items()
             if isinstance(p, torch.Tensor) and p.requires_grad}
    return {k: float(v.detach()) for k, v in l.items()}, grads, running
