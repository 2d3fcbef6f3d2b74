"""CPU checks of the frozen-BatchNorm training oracle (oracle/ref_frozen_bn.py) that the GPU step is compared against:
pinned to the existing oracles (and through them to the live-reference fixtures) at the two ends, no layer frozen and
every layer frozen, and checked for a mixed pattern against the drop-in module's own torch layers in float64, with
every other nn.BatchNorm2d put in eval() inside a train() model as a user fine-tuning it would."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import inputs as oin, ref_frozen_bn as ofb, ref_models as orm, ref_song2face_train as ost, weights as ow

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SEED_W = {"audio2mesh": 11, "song2face": 14}


def _running(sd):
    return {k: v.clone() for k, v in sd.items() if "running_" in k or "num_batches" in k}


def test_audio2mesh_oracle_ends_match_existing_oracles_and_fixture():
    z = np.load(os.path.join(G, "audio2mesh.npz"))
    sd = ow.make_state_dict("audio2mesh", seed=int(z["seed_w"]))
    B, s, step = int(z["batch"]), int(z["seed_in"]), int(z["step"])
    x, oh, tp = oin.a2m_features(B, s), oin.one_hot(B, 12, s), oin.batch_templates(B, s)
    with torch.no_grad():
        r_new, r_old = _running(sd), _running(sd)
        y = ofb.audio2mesh_forward(sd, x, oh, tp, frozen=(), running=r_new)
        assert torch.equal(y, orm.audio2mesh_forward(sd, x, oh, tp, train_bn=True, running=r_old))
        assert all(torch.equal(r_new[k], r_old[k]) for k in r_old)
        assert int(r_new["analysis_net.1.num_batches_tracked"]) == int(sd["analysis_net.1.num_batches_tracked"]) + 1
        np.testing.assert_allclose(y.reshape(-1)[::step].numpy(), z["out_train"], rtol=0, atol=5e-6)

        r = _running(sd)
        y = ofb.audio2mesh_forward(sd, x, oh, tp, frozen=ofb.A2M_BN, running=r)
        assert torch.equal(y, orm.audio2mesh_forward(sd, x, oh, tp))
        assert all(torch.equal(r[k], sd[k]) for k in r)
        np.testing.assert_allclose(y.reshape(-1)[::step].numpy(), z["out_eval"], rtol=0, atol=2e-6)


def test_song2face_oracle_ends_match_existing_oracles_and_fixture():
    z = np.load(os.path.join(G, "song2face.npz"))
    sd = ow.make_state_dict("song2face", seed=int(z["seed_w"]))
    B, s, step = int(z["batch"]), int(z["seed_in"]), int(z["step"])
    x, oh, tp = oin.a2m_features(B, s), oin.one_hot(B, 12, s), oin.batch_templates(B, s)
    with torch.no_grad():
        r_new, r_old = _running(sd), _running(sd)
        y = ofb.song2face_forward(sd, x, oh, tp, frozen=(), running=r_new)
        assert torch.equal(y, ost.song2face_forward(sd, x, oh, tp, train_bn=True, running=r_old))
        assert all(torch.equal(r_new[k], r_old[k]) for k in r_old)

        r = _running(sd)
        y = ofb.song2face_forward(sd, x, oh, tp, frozen=ofb.S2F_BN, running=r)
        assert torch.equal(y, orm.song2face_forward(sd, x, oh, tp))
        assert all(torch.equal(r[k], sd[k]) for k in r)
        np.testing.assert_allclose(y.reshape(-1)[::step].numpy(), z["out"], rtol=0, atol=2e-6)


def test_bn_prefixes_are_the_modules_batchnorms():
    from a2f_b200 import modules
    for kind, cls in (("audio2mesh", modules.Audio2Mesh), ("song2face", modules.Song2Face)):
        names = tuple(n for n, mod in cls(15069, 12).named_modules() if isinstance(mod, torch.nn.BatchNorm2d))
        assert sorted(names) == sorted(ofb.BN_PREFIXES[kind]), kind


def _module_forward(kind, m, x, one_hot, template):
    """ref:src/model/audio2face.py:57-66 / ref:src/model/song2face.py:63-76 through the drop-in module's parameter
    containers (plain torch layers, each BatchNorm2d in its own train() / eval() mode)."""
    bs = x.size(0)
    emb = one_hot.repeat(1, 32).view(bs, 1, -1, 32)
    h = torch.cat((x.unsqueeze(1), emb), 2)
    if kind == "audio2mesh":
        h = m.articulation_net(m.analysis_net(h)).view(bs, -1)
    else:
        h = m.vocal_encoder_nn(h).squeeze(3)
        h, _ = m.vocal_encoder_lstm1(h)
        h, _ = m.vocal_encoder_lstm2(h)
        h = F.interpolate(h.unsqueeze(3), size=(32, 1), mode="bilinear")
        h = m.regression_net(h).squeeze(3).squeeze(2)
    h = m.output_net(torch.cat((h, one_hot), 1))
    return h.view(bs, -1, 3) + template


@pytest.mark.parametrize("kind", ["audio2mesh", "song2face"])
def test_mixed_pattern_oracle_matches_torch_layers(kind):
    from a2f_b200 import modules
    B, s = 4, 5                                                 # VocaLoss pairs consecutive windows
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in ow.make_state_dict(kind, seed=SEED_W[kind]).items()}
    x, oh, tp = oin.a2m_features(B, s).double(), oin.one_hot(B, 12, s).double(), oin.batch_templates(B, s).double()
    gt = oin.gt_like((B, 5023, 3), tp, s + 1).double()
    frozen = ofb.BN_PREFIXES[kind][::2]
    want_loss, want, running = ofb.loss_and_grads(kind, sd, x, oh, tp, gt, frozen=frozen)

    m = (modules.Audio2Mesh if kind == "audio2mesh" else modules.Song2Face)(5023 * 3, 12).double()
    m.load_state_dict(sd, strict=True)
    m.train()
    for name in frozen:
        m.get_submodule(name).eval()
    loss = orm.voca_loss(_module_forward(kind, m, x, oh, tp), gt)
    loss["loss"].backward()
    for k in ("loss", "rec_loss", "vel_loss"):
        assert abs(float(loss[k].detach()) - want_loss[k]) <= 1e-10 * abs(want_loss[k]), k
    got = dict(m.named_parameters())
    assert set(got) == set(want)
    for k, g in want.items():
        assert float((got[k].grad - g).abs().max()) <= 1e-9 * (1.0 + float(g.abs().max())), k
    state = m.state_dict()
    assert len(running) == 3 * len(ofb.BN_PREFIXES[kind])
    for k, v in running.items():
        frozen_layer = k.rsplit(".", 1)[0] in frozen
        if v.dtype == torch.int64:
            assert int(state[k]) == int(v) == int(sd[k]) + (0 if frozen_layer else 1), k
        else:
            assert float((state[k] - v).abs().max()) <= 1e-12, k
            assert torch.equal(v, sd[k]) == frozen_layer, k
