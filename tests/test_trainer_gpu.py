"""FaceformerTrainer (flat buffers + fused Adam) on one GPU against torch.optim.Adam over the oracle's autograd
(ref:src/model/lightning_model.py:150-161,209-213), and the N-GPU data-parallel check when the box has >= 2 GPUs."""
import os
import subprocess
import sys

import pytest
import torch

from oracle import inputs as oin, ref_models as orm, weights as ow

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_trainer_steps_match_torch_adam_on_the_oracle(a2f_lib, dev):
    from a2f_b200 import modules, trainer as tr
    n, lr = 6400, 1e-4
    audio, oh = oin.audio(1, n, 61), oin.one_hot(1, 12, 61)
    tp = oin.batch_templates(1, 61, scale=100.0)
    gt = oin.gt_like((1, 24, 5023, 3), tp[:, None], 62, scale=100.0)
    sd = ow.make_state_dict("faceformer", seed=13)
    m = modules.Faceformer(15069, 12)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).eval().set_precision("fp32")
    t = tr.FaceformerTrainer(m, lr=lr, fps=60)
    got = [float(t.step(audio.to(dev), oh.to(dev), tp.to(dev), gt.to(dev))["loss"]) for _ in range(2)]
    # oracle: torch.optim.Adam(lr, weight_decay=lr/10) over autograd of the CPU restatement
    params = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and k != "PPE.pe" else v)
              for k, v in sd.items()}
    train = [p for k, p in params.items() if isinstance(p, torch.Tensor) and p.requires_grad
             and k != "audio_encoder.masked_spec_embed"]
    opt = torch.optim.Adam(train, lr=lr, weight_decay=lr / 10)
    want = []
    for _ in range(2):
        opt.zero_grad()
        loss = orm.faceformer_loss(orm.faceformer_forward(params, audio, oh, tp, 60), gt)["loss"]
        loss.backward()
        opt.step()
        want.append(float(loss))
    print("trainer losses", got, "oracle", want)
    for a, b in zip(got, want):
        assert abs(a - b) < 1e-4 * abs(b)
    assert want[1] < want[0]
    # parameters after two steps: each moved by ~lr per step; compare the bulk (sign flips of ~zero gradients excluded)
    new = {k: p.detach().cpu() for k, p in m.named_parameters()}
    assert torch.equal(new["audio_encoder.masked_spec_embed"], sd["audio_encoder.masked_spec_embed"])   # no grad -> untouched
    bad = tot = 0
    for k, p in params.items():
        if not (isinstance(p, torch.Tensor) and p.requires_grad) or k == "audio_encoder.masked_spec_embed":
            continue
        d = (new[k] - p.detach()).abs().reshape(-1)
        bad += int((d > 0.05 * lr).sum())
        tot += d.numel()
    print(f"parameters off by > 0.05*lr after two steps: {bad} of {tot}")
    assert bad < 2e-3 * tot


def test_state_dict_roundtrip_after_flattening(a2f_lib, dev):
    from a2f_b200 import modules, trainer as tr
    sd = ow.make_state_dict("faceformer", seed=13)
    m = modules.Faceformer(15069, 12)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).eval().set_precision("bf16")
    tr.FaceformerTrainer(m)
    out = m.state_dict()
    assert list(out.keys()) == list(sd.keys())
    assert all(torch.equal(out[k].cpu(), sd[k]) for k in sd)
    m.load_state_dict(sd, strict=True)            # loading a checkpoint writes through the flat views


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_data_parallel_two_gpus(a2f_lib, dev, precision):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tests", "dp_check.py"), precision]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0 and "DP_CHECK_OK" in r.stdout
