"""Song2Face training step on the GPU (model.train(): batch-statistics BatchNorm, LSTM backpropagation through time).

Kernels: a2f_lstm_bptt against torch.nn.LSTM autograd (CPU, fp64), a2f_lstm_recurrence_train against the inference
recurrence, a2f_col2im1d / a2f_song2face_resize_bwd as adjoints of their forward ops.  Step: loss, every parameter
gradient and the running statistics against oracle/ref_song2face_train.loss_and_grads (torch autograd over the CPU
restatement, itself checked against torch's own layers in tests/test_song2face_train.py); the module's train() /
eval() routing; torch.optim.Adam and trainer.ConvModelTrainer driving the drop-in module."""
import copy

import pytest
import torch
import torch.nn.functional as F

from oracle import inputs as oin, ref_models as orm, ref_song2face_train as ost, weights as ow

pytestmark = pytest.mark.gpu


def _rel(got, want):
    return float((got.double().cpu() - want.double().cpu()).norm()) / float(want.double().norm())


def _ref_lstm_dgates(lstm64, x, dh):
    """fp64 gradients of the pre-activation gates of torch.nn.LSTM's recurrence (written out, the graph kept per step)"""
    B, T, _ = x.shape
    H = lstm64.weight_hh_l0.shape[1]
    h, c = x.new_zeros(B, H), x.new_zeros(B, H)
    xp = F.linear(x, lstm64.weight_ih_l0, lstm64.bias_ih_l0 + lstm64.bias_hh_l0)
    pre, outs = [], []
    for t in range(T):
        a = xp[:, t] + F.linear(h, lstm64.weight_hh_l0)
        a.retain_grad()
        pre.append(a)
        i, f, g, o = a.chunk(4, 1)
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
        h = torch.sigmoid(o) * torch.tanh(c)
        outs.append(h)
    (torch.stack(outs, 1) * dh).sum().backward()
    return torch.stack([a.grad for a in pre], 1)


@pytest.mark.parametrize("T", [7, 256])
@pytest.mark.parametrize("B", [1, 5, 8, 13])
def test_lstm_bptt_vs_torch_lstm(a2f_lib, dev, B, T):
    """B = 1, 5, 13 leave clusters of 8 windows partly filled."""
    from a2f_b200 import conv_training as ct, ops
    g = torch.Generator().manual_seed(1000 * B + T)
    I = 48
    lstm = torch.nn.LSTM(I, 256, 1, batch_first=True)
    x = torch.randn(B, T, I, generator=g)
    dh = torch.randn(B, T, 256, generator=g)

    ref = copy.deepcopy(lstm).double()
    x64 = x.double().requires_grad_(True)
    out, _ = ref(x64)
    (out * dh.double()).sum().backward()
    dg_ref = _ref_lstm_dgates(copy.deepcopy(lstm).double(), x.double(), dh.double())

    gl = copy.deepcopy(lstm).to(dev)
    _, e = ct.lstm_forward_train(gl, x.to(dev))
    dgates = ops.lstm_bptt(dh.to(dev), e["gates"], e["cell"], gl.weight_hh_l0.detach())
    again = ops.lstm_bptt(dh.to(dev), e["gates"], e["cell"], gl.weight_hh_l0.detach())
    assert torch.equal(dgates, again)
    dx = ct.lstm_backward(gl, e, dh.to(dev))
    torch.cuda.synchronize()

    errs = {"dgates": _rel(dgates, dg_ref), "dx": _rel(dx, x64.grad)}
    for name in ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0"):
        errs[name] = _rel(getattr(gl, name).grad, getattr(ref, name).grad)
    print(f"B={B} T={T}: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    assert max(errs.values()) < 1e-4, errs


@pytest.mark.parametrize("B", [4, 8, 13])
def test_lstm_recurrence_train_matches_inference(a2f_lib, dev, B):
    from a2f_b200 import ops
    g = torch.Generator().manual_seed(77 + B)
    T = 256
    lstm = torch.nn.LSTM(64, 256, 1, batch_first=True)
    x = torch.randn(B, T, 64, generator=g)
    with torch.no_grad():
        xp = F.linear(x, lstm.weight_ih_l0, lstm.bias_ih_l0 + lstm.bias_hh_l0).contiguous()
    whh = lstm.weight_hh_l0.detach().contiguous()
    xp_d, whh_d = xp.to(dev), whh.to(dev)
    h_inf = ops.lstm_recurrence(xp_d, whh_d.t().contiguous(), B, T, 256, whh=whh_d)
    h, gates, cell = ops.lstm_recurrence_train(xp_d, whh_d, B, T, 256)
    torch.cuda.synchronize()
    assert torch.equal(h, h_inf)
    h, gates, cell = h.cpu().double(), gates.cpu().double(), cell.cpu().double()
    hprev = torch.cat([torch.zeros(B, 1, 256, dtype=torch.float64), h[:, :-1]], 1)
    a = xp.double() + hprev @ whh.double().t()
    i, f, gg, o = a.chunk(4, 2)
    want = torch.cat([torch.sigmoid(i), torch.sigmoid(f), torch.tanh(gg), torch.sigmoid(o)], 2)
    assert float((gates - want).abs().max()) < 1e-6
    cprev = torch.cat([torch.zeros(B, 1, 256, dtype=torch.float64), cell[:, :-1]], 1)
    c_want = torch.sigmoid(f) * cprev + torch.sigmoid(i) * torch.tanh(gg)       # one step from the saved c_{t-1}
    assert float((cell - c_want).abs().max()) < 1e-6
    assert float((h - gates[..., 768:] * torch.tanh(cell)).abs().max()) < 1e-6


@pytest.mark.parametrize("taps,stride,pad", [(5, 2, 2), (3, 2, 1), (3, 2, 0)])
def test_col2im1d_is_the_adjoint_of_im2col1d(a2f_lib, dev, taps, stride, pad):
    from a2f_b200 import ops
    g = torch.Generator().manual_seed(taps * 10 + pad)
    for outer, L_, C_, ld in ((6, 13, 7, 9), (4, 32, 256, 256)):
        kpad = (taps * C_ + 7) // 8 * 8
        L_out = (L_ + 2 * pad - taps) // stride + 1
        x = torch.randn(outer, L_, ld, generator=g)
        y = torch.randn(outer * L_out, kpad, generator=g)
        col = ops.im2col1d(x.to(dev), outer, L_ * ld, ld, C_, L_, taps, stride, pad, kpad, False).cpu()
        dx = torch.full((outer, L_, ld), float("nan"))
        dx = ops.col2im1d(y.to(dev), dx.to(dev), outer, L_ * ld, ld, C_, L_, taps, stride, pad).cpu()
        assert torch.isnan(dx[..., C_:]).all() and torch.isfinite(dx[..., :C_]).all()
        lhs = (col.double() * y.double()).sum()
        rhs = (x[..., :C_].double() * dx[..., :C_].double()).sum()
        scale = float((col.double() * y.double()).abs().sum())
        assert abs(float(lhs - rhs)) <= 1e-6 * scale, (float(lhs), float(rhs))


def test_song2face_resize_bwd_is_the_adjoint(a2f_lib, dev):
    from a2f_b200 import ops
    g = torch.Generator().manual_seed(9)
    B, T = 3, 256
    h = torch.randn(B, T, 256, generator=g)
    y = torch.randn(B, 32, T, generator=g)
    out = ops.song2face_resize(h.to(dev), 32).cpu()
    dh = ops.song2face_resize_bwd(y.to(dev), 256).cpu()
    lhs, rhs = (out.double() * y.double()).sum(), (h.double() * dh.double()).sum()
    assert abs(float(lhs - rhs)) <= 1e-6 * float((out.double() * y.double()).abs().sum())
    want = F.interpolate(h.unsqueeze(3), size=(32, 1), mode="bilinear")   # [B, T, 32, 1] (ref song2face.py:71)
    assert float((out - want.squeeze(3).transpose(1, 2)).abs().max()) < 1e-6


def _inputs(B, seed):
    x, oh, tp = oin.a2m_features(B, seed), oin.one_hot(B, 12, seed), oin.batch_templates(B, seed)
    return x, oh, tp, oin.gt_like((B, 5023, 3), tp, seed + 1)


def _compare(grads, want, tol):
    """the rule of tests/test_conv_train_gpu.py: per-tensor relative norm; conv biases in front of a train-mode BatchNorm
    have a mathematically zero gradient and are checked against the largest gradient instead"""
    gmax = max(float(g.norm()) for g in want.values())
    worst, worst_k = 0.0, None
    for k, g in want.items():
        n = float(g.norm())
        if n < 1e-5 * gmax:
            assert float(grads[k].norm()) < 1e-4 * gmax, (k, float(grads[k].norm()), gmax)
            continue
        rel = float((grads[k].double() - g.double()).norm()) / n
        if rel > worst:
            worst, worst_k = rel, k
    assert worst < tol, (worst_k, worst)
    return worst, worst_k


@pytest.mark.parametrize("B,seed", [(4, 7), (14, 7), (64, 17)])
def test_song2face_train_step_vs_oracle(a2f_lib, dev, B, seed):
    """B = 14 (VocaLoss pairs consecutive windows, so B is even) leaves the second LSTM cluster partly filled.  The input
    seeds avoid ReLU ties (see tests/test_conv_train_gpu.py)."""
    from a2f_b200 import modules
    sd = ow.make_state_dict("song2face", seed=14)
    x, oh, tp, gt = _inputs(B, seed)
    want_loss, want, running = ost.loss_and_grads(sd, x, oh, tp, gt)
    m = modules.Song2Face(15069, 12).to(dev)
    m.load_state_dict(sd, strict=True)
    if B == 14:                                  # same fp32 conv / LSTM path; only the vertex head follows the precision
        m.set_precision("bf16")
    m.train()
    loss = modules.VocaLoss()(m(x.to(dev), oh.to(dev), tp.to(dev)), gt.to(dev))
    loss["loss"].backward()
    torch.cuda.synchronize()
    for k in ("loss", "rec_loss", "vel_loss"):
        assert abs(float(loss[k]) - want_loss[k]) < 1e-4 * abs(want_loss[k]), (k, float(loss[k]), want_loss[k])
    grads = {k: p.grad.detach().cpu() for k, p in m.named_parameters()}
    assert set(grads) == set(want)
    worst, k = _compare(grads, want, 2e-3)
    print(f"song2face B={B}: loss {float(loss['loss']):.6f} (oracle {want_loss['loss']:.6f}); worst per-tensor rel grad err "
          f"{worst:.2e} ({k})")
    got = m.state_dict()
    assert len(running) == 3 * 8
    for name, v in running.items():
        if v.dtype == torch.int64:
            assert int(got[name]) == int(v), name
        else:
            assert float((got[name].cpu() - v).abs().max()) < 1e-5 * (1 + float(v.abs().max())), name


def test_train_mode_no_grad_forward_and_eval_after(a2f_lib, dev):
    from a2f_b200 import modules
    B = 6
    sd = ow.make_state_dict("song2face", seed=14)
    x, oh, tp, _ = _inputs(B, 23)
    ref_sd = {k: v.clone() for k, v in sd.items()}
    running = {k: v for k, v in ref_sd.items() if "running_" in k or "num_batches" in k}
    with torch.no_grad():
        want = ost.song2face_forward(ref_sd, x, oh, tp, train_bn=True, running=running)
    m = modules.Song2Face(15069, 12).to(dev)
    m.load_state_dict(sd, strict=True)
    with torch.no_grad():
        m.eval()(x.to(dev), oh.to(dev), tp.to(dev))  # fills the packed-weight cache with the old running stats
        got = m.train()(x.to(dev), oh.to(dev), tp.to(dev)).cpu()
    assert float((got - want).abs().max()) < 1e-5
    state = m.state_dict()
    for k, v in running.items():
        assert float((state[k].cpu().double() - v.double()).abs().max()) < 1e-5 * (1 + float(v.abs().max())), k
    m.eval()
    with torch.no_grad():
        y_eval = m(x.to(dev), oh.to(dev), tp.to(dev)).cpu()
    want_eval = orm.song2face_forward({k: v.cpu() for k, v in m.state_dict().items()}, x, oh, tp)
    assert float((y_eval - want_eval).abs().max()) < 1e-5


def test_eval_mode_gradients_are_refused(a2f_lib, dev):
    import a2f_b200
    from a2f_b200 import modules
    m = modules.Song2Face(15069, 12).to(dev).eval()
    x, oh, tp, _ = _inputs(4, 3)
    with pytest.raises(a2f_b200.A2FError):
        m(x.to(dev), oh.to(dev), tp.to(dev))


def test_torch_adam_reduces_the_loss(a2f_lib, dev):
    from a2f_b200 import modules
    m = modules.Song2Face(15069, 12).to(dev)
    m.load_state_dict(ow.make_state_dict("song2face", seed=14), strict=True)
    m.train()
    x, oh, tp, gt = [t.to(dev) for t in _inputs(16, 9)]
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-4)
    lf = modules.VocaLoss()
    losses = []
    for _ in range(5):
        opt.zero_grad()
        loss = lf(m(x, oh, tp), gt)
        loss["loss"].backward()
        opt.step()
        losses.append(float(loss["loss"]))
    assert losses[-1] < losses[0], losses


def test_conv_model_trainer_with_mfcc_extractor(a2f_lib, dev):
    from a2f_b200 import features, modules, trainer as tr
    from oracle import ref_mfcc as omf
    cfg = omf.CONFIGS["audio2mesh"]
    B = 16
    sd = ow.make_state_dict("song2face", seed=12)
    x, oh, tp = oin.speech_like_windows(B, seed=7), oin.one_hot(B, 12, 7), oin.batch_templates(B, 7)
    gt = oin.gt_like((B, 5023, 3), tp, 8)
    with torch.no_grad():
        feat = omf.mfcc_forward(omf.make_buffers(cfg[0], cfg[1], cfg[3], cfg[5]), x, cfg[2], cfg[3], cfg[4], cfg[5])
    want, _, _ = ost.loss_and_grads(sd, feat, oh, tp, gt)
    m = modules.Song2Face(15069, 12).to(dev)
    m.load_state_dict(sd, strict=True)
    t = tr.ConvModelTrainer(m, features.MFCCExtractor(*cfg).to(dev), lr=1e-3)
    losses = [t.step(x.to(dev), oh.to(dev), tp.to(dev), gt.to(dev)) for _ in range(4)]
    first = {k: float(v) for k, v in losses[0].items()}
    for k in ("loss", "rec_loss", "vel_loss"):
        assert abs(first[k] - want[k]) <= 2e-4 * abs(want[k]), (k, first[k], want[k])
    assert float(losses[-1]["loss"]) < float(losses[0]["loss"])
    assert set(m.state_dict().keys()) == set(sd.keys())
