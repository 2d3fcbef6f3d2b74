"""TEST INFRASTRUCTURE -- CPU restatement (oracle) of Song2Face's TRAINING step: the reference's `model.train()` forward
(batch-statistics BatchNorm with the running-statistic update) and torch.autograd over it.

Only tests/ may import this package.  The layers, the LSTM and the BatchNorm rule are those of oracle/ref_models.py
(`lstm_forward`, `_bn`); with train_bn=False `song2face_forward` is the eval-mode `ref_models.song2face_forward`, which
tests/golden/song2face.npz pins against the live reference (tests/test_song2face_train.py checks that the two agree,
and checks the train-mode step against the drop-in module's own torch layers).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn.functional as F

from . import ref_models as orm

SD = Dict[str, torch.Tensor]


def song2face_forward(sd: SD, x: torch.Tensor, one_hot: torch.Tensor, template: torch.Tensor,
                      train_bn: bool = False, running: Optional[SD] = None) -> torch.Tensor:
    """ref:src/model/song2face.py:63-76; train_bn: batch-statistics BatchNorm, `running` (<bn>.running_mean / running_var /
    num_batches_tracked) updated in place as nn.BatchNorm2d does (ref_models._bn)."""
    bs = x.size(0)
    emb = one_hot.repeat(1, 32).view(bs, 1, -1, 32)                     # song2face.py:65
    h = torch.cat((x.unsqueeze(1), emb), 2)                             # :66-67 -> [bs,1,64,32]
    for i, (kw, pad) in enumerate(((5, 2), (5, 2), (3, 1), (3, 1), (3, 1))):        # :33-39 conv -> BN -> ReLU
        p = f"vocal_encoder_nn.{i}."
        h = F.conv2d(h, sd[p + "0.weight"], sd[p + "0.bias"], stride=(1, 2), padding=(0, pad))
        h = F.relu(orm._bn(sd, p + "1", h, train_bn, running))
    h = h.squeeze(3)                                                    # :68 -> [bs, 256, 64]
    for name in ("vocal_encoder_lstm1", "vocal_encoder_lstm2"):         # :69-70: 256 steps of 64 / 256 features
        h = orm.lstm_forward(h, sd[name + ".weight_ih_l0"], sd[name + ".weight_hh_l0"], sd[name + ".bias_ih_l0"],
                             sd[name + ".bias_hh_l0"])
    h = F.interpolate(h.unsqueeze(3), size=(32, 1), mode="bilinear")    # :71-72 -> [bs, 256, 32, 1]
    for i in range(4):                                                  # :54-59
        p = f"regression_net.{i}."
        h = F.conv2d(h, sd[p + "0.weight"], sd[p + "0.bias"], stride=(2, 1), padding=(1 if i < 3 else 0, 0))
        if i < 3:
            h = orm._bn(sd, p + "1", h, train_bn, running)
        h = F.relu(h)
    h = h.squeeze(3).squeeze(2)                                         # :74
    h = torch.cat((h, one_hot), 1)                                      # :75
    h = F.linear(h, sd["output_net.0.weight"], sd["output_net.0.bias"])
    h = torch.tanh(F.linear(h, sd["output_net.1.weight"], sd["output_net.1.bias"]))
    h = F.linear(h, sd["output_net.3.weight"], sd["output_net.3.bias"])
    h = F.linear(h, sd["output_net.4.weight"], sd["output_net.4.bias"])
    return h.view(bs, -1, 3) + template                                 # :76


def loss_and_grads(sd: SD, x: torch.Tensor, one_hot: torch.Tensor, template: torch.Tensor, gt: torch.Tensor):
    """Training step of Song2Face (ref:src/model/lightning_model.py:150-161 with VocaLoss, ref:src/loss/loss.py:24-55):
    `pred = model(x, one_hot, template)` in TRAIN mode, `VocaLoss()(pred, gt)`, autograd -- the contract of
    ref_train.conv_loss_and_grads.  -> (losses, {param: grad}, running-stat dict after the step)."""
    params = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and "running_" not in k else v.clone())
              for k, v in sd.items()}
    running = {k: v for k, v in params.items() if "running_" in k or "num_batches" in k}
    with torch.enable_grad():
        out = song2face_forward(params, x, one_hot, template, train_bn=True, running=running)
        l = orm.voca_loss(out, gt)
        l["loss"].backward()
    grads = {k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in params.items()
             if isinstance(p, torch.Tensor) and p.requires_grad}
    return {k: float(v.detach()) for k, v in l.items()}, grads, running
