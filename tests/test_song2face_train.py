"""CPU checks of the Song2Face training oracle (oracle/ref_song2face_train.py) that the GPU training
step is compared against: the written-out LSTM against torch.nn.LSTM autograd, and the whole train-mode step against a
forward built from the drop-in module's own torch layers (nn.Conv2d / nn.BatchNorm2d / nn.LSTM / nn.Linear called in the
reference's order, ref:src/model/song2face.py:63-76, F.interpolate for the resize)."""
import torch
import torch.nn.functional as F

from oracle import inputs as oin, ref_models as orm, ref_song2face_train as ost, weights as ow


def test_lstm_restatement_gradients_match_torch_lstm():
    g = torch.Generator().manual_seed(21)
    lstm = torch.nn.LSTM(12, 16, 1, batch_first=True).double()
    x = torch.randn(3, 9, 12, generator=g, dtype=torch.float64)
    dh = torch.randn(3, 9, 16, generator=g, dtype=torch.float64)

    def grads(fn):
        xx = x.clone().requires_grad_(True)
        lstm.zero_grad()
        (fn(xx) * dh).sum().backward()
        return [xx.grad] + [p.grad.clone() for p in (lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0)]

    want = grads(lambda xx: lstm(xx)[0])
    got = grads(lambda xx: orm.lstm_forward(xx, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0))
    for a, b in zip(got, want):
        assert float((a - b).abs().max()) <= 1e-10


def test_eval_mode_equals_the_pinned_oracle():
    """with train_bn=False the training oracle is ref_models.song2face_forward (pinned by tests/golden/song2face.npz)"""
    B, s = 3, 2
    sd = ow.make_state_dict("song2face", seed=14)
    x, oh, tp = oin.a2m_features(B, s), oin.one_hot(B, 12, s), oin.batch_templates(B, s)
    with torch.no_grad():
        assert torch.equal(ost.song2face_forward(sd, x, oh, tp), orm.song2face_forward(sd, x, oh, tp))


def _module_forward(m, x, one_hot, template):
    """ref:src/model/song2face.py:63-76 through the drop-in module's parameter containers (plain torch layers)."""
    bs = x.size(0)
    emb = one_hot.repeat(1, 32).view(bs, 1, -1, 32)
    h = torch.cat((x.unsqueeze(1), emb), 2)
    h = m.vocal_encoder_nn(h).squeeze(3)
    h, _ = m.vocal_encoder_lstm1(h)
    h, _ = m.vocal_encoder_lstm2(h)
    h = F.interpolate(h.unsqueeze(3), size=(32, 1), mode="bilinear")
    h = m.regression_net(h).squeeze(3).squeeze(2)
    h = m.output_net(torch.cat((h, one_hot), 1))
    return h.view(bs, -1, 3) + template


def test_train_mode_oracle_matches_torch_layers():
    from a2f_b200 import modules
    B, s = 4, 5                                                 # VocaLoss pairs consecutive windows
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in ow.make_state_dict("song2face", seed=14).items()}
    x, oh, tp = oin.a2m_features(B, s).double(), oin.one_hot(B, 12, s).double(), oin.batch_templates(B, s).double()
    gt = oin.gt_like((B, 5023, 3), tp, s + 1).double()
    want_loss, want, running = ost.loss_and_grads(sd, x, oh, tp, gt)

    m = modules.Song2Face(5023 * 3, 12).double()
    m.load_state_dict(sd, strict=True)
    m.train()
    loss = orm.voca_loss(_module_forward(m, x, oh, tp), gt)
    loss["loss"].backward()
    for k in ("loss", "rec_loss", "vel_loss"):
        assert abs(float(loss[k]) - want_loss[k]) <= 1e-10 * abs(want_loss[k]), k
    got = dict(m.named_parameters())
    assert set(got) == set(want)
    for k, g in want.items():
        assert float((got[k].grad - g).abs().max()) <= 1e-9 * (1.0 + float(g.abs().max())), k
    state = m.state_dict()
    assert len(running) == 3 * 8
    for k, v in running.items():
        if v.dtype == torch.int64:
            assert int(state[k]) == int(v) == int(sd[k]) + 1, k
        else:
            assert float((state[k] - v).abs().max()) <= 1e-12, k
