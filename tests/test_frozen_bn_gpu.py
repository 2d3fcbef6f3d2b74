"""Frozen-BatchNorm fine-tuning on the GPU: Audio2Mesh / Song2Face in train() with some or all of their nn.BatchNorm2d
layers in eval() (running statistics, left unchanged; gradients through the fixed affine map).

Kernels: a2f_bn_frozen_stats against the running statistics, a2f_bn_frozen_bwd against float64 torch autograd of
F.batch_norm(training=False) on both activation layouts.
Step: loss, every parameter gradient and the running statistics against oracle/ref_frozen_bn.loss_and_grads (torch
autograd over the CPU restatement, itself checked against torch's own layers in tests/test_frozen_bn.py), in the
autograd path, in train() under no_grad and in trainer.ConvModelTrainer(freeze_bn=True)."""
import pytest
import torch
import torch.nn.functional as F

from oracle import inputs as oin, ref_frozen_bn as ofb, weights as ow

pytestmark = pytest.mark.gpu
SEED_W = {"audio2mesh": 11, "song2face": 14}


def _inputs(B, seed):
    x, oh, tp = oin.a2m_features(B, seed), oin.one_hot(B, 12, seed), oin.batch_templates(B, seed)
    return x, oh, tp, oin.gt_like((B, 5023, 3), tp, seed + 1)


def _model(kind, dev, frozen):
    from a2f_b200 import modules
    m = (modules.Audio2Mesh if kind == "audio2mesh" else modules.Song2Face)(15069, 12).to(dev)
    m.load_state_dict(ow.make_state_dict(kind, seed=SEED_W[kind]), strict=True)
    m.train()
    for name in frozen:
        m.get_submodule(name).eval()
    return m


def _running(m):
    return {k: v.detach().clone() for k, v in m.state_dict().items() if "running_" in k or "num_batches" in k}


def _compare(grads, want, tol):
    """the rule of tests/test_conv_train_gpu.py: per-tensor relative norm; a tensor whose gradient is mathematically zero
    (a conv bias in front of a train-mode BatchNorm) is checked against the largest gradient instead"""
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


def _step(m, dev, x, oh, tp, gt, between=None):
    from a2f_b200 import modules
    out = m(x.to(dev), oh.to(dev), tp.to(dev))
    if between is not None:
        between()
    loss = modules.VocaLoss()(out, gt.to(dev))
    loss["loss"].backward()
    torch.cuda.synchronize()
    return {k: float(v.detach()) for k, v in loss.items()}


def _check_step(kind, m, loss, want_loss, want, running, before, frozen, label):
    for k in ("loss", "rec_loss", "vel_loss"):
        assert abs(loss[k] - want_loss[k]) < 1e-4 * abs(want_loss[k]), (k, loss[k], want_loss[k])
    grads = {k: p.grad.detach().cpu() for k, p in m.named_parameters() if p.requires_grad}
    worst, wk = _compare(grads, {k: want[k] for k in grads}, 2e-3)
    print(f"{kind} {label}: loss {loss['loss']:.6f} (oracle {want_loss['loss']:.6f}); worst per-tensor rel grad err "
          f"{worst:.2e} ({wk})")
    got = _running(m)
    assert set(got) == set(running)
    for name, v in running.items():
        if name.rsplit(".", 1)[0] in frozen:
            assert torch.equal(got[name], before[name]), name            # bit-unchanged, num_batches_tracked included
        elif v.dtype == torch.int64:
            assert int(got[name]) == int(v), name
        else:
            assert float((got[name].cpu() - v).abs().max()) < 1e-5 * (1 + float(v.abs().max())), name


# ------------------------------------------------------------------------------------------------------------- kernel
def test_bn_frozen_stats_reads_the_running_statistics(a2f_lib, dev):
    from a2f_b200 import ops
    g = torch.Generator().manual_seed(5)
    C, eps = 243, 1e-5
    gamma, beta, rm = torch.randn(C, generator=g), torch.randn(C, generator=g), torch.randn(C, generator=g)
    rv = torch.rand(C, generator=g) + 0.5
    d = [t.to(dev) for t in (gamma, beta, rm, rv)]
    mr, ss = ops.bn_frozen_stats(d[0], d[1], eps, d[2], d[3])
    torch.cuda.synchronize()
    assert torch.equal(d[2].cpu(), rm) and torch.equal(d[3].cpu(), rv)
    rstd = 1.0 / torch.sqrt(rv.double() + eps)
    want_mr = torch.cat((rm.double(), rstd))
    want_ss = torch.cat((gamma.double() * rstd, beta.double() - rm.double() * gamma.double() * rstd))
    assert float((mr.cpu().double() - want_mr).abs().max()) < 1e-6
    assert float((ss.cpu().double() - want_ss).abs().max()) < 1e-6 * (1 + float(want_ss.abs().max()))


@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("layout", ["pad", "rows"])
def test_bn_frozen_bwd_kernel_vs_torch(a2f_lib, dev, relu, layout):
    from a2f_b200 import conv_training as ct, ops
    g = torch.Generator().manual_seed(31 + 2 * relu + (layout == "rows"))
    if layout == "pad":                       # Pad: [nb, L+1, C], row 0 of every block is zero padding
        nb, L_, C = 6, 33, 256
        zp = ct.Pad(nb, L_, C, "cpu")
        zp.buf[:, 1:] = torch.randn(nb, L_, C, generator=g)
        z_live = zp.buf[:, 1:]
        mk = lambda t: ct.Pad(nb, L_, C, dev, buf=t.to(dev)).view()      # noqa: E731
        buf_shape = zp.buf.shape
        z_buf = zp.buf
    else:                                     # _rows: [rows, ld] with ld > C (live columns 0..C-1)
        rows, C, ld = 1037, 243, 244
        z_buf = torch.randn(rows, ld, generator=g)
        z_live = z_buf[:, :C]
        mk = lambda t: ct._rows(t.to(dev), C)                            # noqa: E731
        buf_shape = z_buf.shape
    rm = 0.3 * torch.randn(C, generator=g)
    rv = torch.rand(C, generator=g) + 0.5
    gamma = torch.randn(C, generator=g)
    beta = torch.randn(C, generator=g)
    eps = 1e-5
    dy_buf = torch.randn(buf_shape, generator=g)

    z64 = z_live.double().reshape(-1, C).clone().requires_grad_(True)
    g64, b64 = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    y64 = F.batch_norm(z64, rm.double(), rv.double(), g64, b64, training=False, eps=eps)
    y_buf = None
    if relu:
        y_buf = torch.zeros(buf_shape)
        (y_buf[:, 1:] if layout == "pad" else y_buf[:, :C]).copy_(F.relu(y64).detach().float().view(z_live.shape))
        y64 = F.relu(y64)                     # fp32 rounding keeps every sign, so both sides use the same mask
    dy_live = (dy_buf[:, 1:] if layout == "pad" else dy_buf[:, :C]).double().reshape(-1, C)
    (y64 * dy_live).sum().backward()

    mean_rstd, _ = ops.bn_frozen_stats(gamma.to(dev), beta.to(dev), eps, rm.to(dev), rv.to(dev))
    dz_buf = torch.full(buf_shape, 7.0, device=dev)
    dgamma0, dbeta0 = torch.randn(C, generator=g), torch.randn(C, generator=g)       # accumulate into non-zero buffers
    dgamma, dbeta = dgamma0.to(dev), dbeta0.to(dev)
    ops.bn_frozen_bwd(mk(dy_buf), mk(y_buf) if relu else None, mk(z_buf), mean_rstd, gamma.to(dev),
                      ct.Pad(nb, L_, C, dev, buf=dz_buf).view() if layout == "pad" else ct._rows(dz_buf, C), dgamma, dbeta)
    torch.cuda.synchronize()
    dz_buf = dz_buf.cpu()
    dz_live = (dz_buf[:, 1:] if layout == "pad" else dz_buf[:, :C]).reshape(-1, C)
    rel = lambda a, b: float((a.double() - b).norm() / b.norm())                     # noqa: E731
    errs = {"dz": rel(dz_live, z64.grad), "dgamma": rel(dgamma.cpu() - dgamma0, g64.grad),
            "dbeta": rel(dbeta.cpu() - dbeta0, b64.grad)}
    print(f"layout {layout} relu {relu}: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    assert max(errs.values()) < 1e-6, errs
    rest = dz_buf[:, 0] if layout == "pad" else dz_buf[:, C:]         # padding rows / columns past C: never written
    assert torch.equal(rest, torch.full_like(rest, 7.0))


# --------------------------------------------------------------------------------------------------------- full step
@pytest.mark.parametrize("kind", ["audio2mesh", "song2face"])
@pytest.mark.parametrize("B,seed", [(4, 7), (14, 7), (64, 17)])
def test_every_batchnorm_frozen_step_vs_oracle(a2f_lib, dev, kind, B, seed):
    """B = 14 (VocaLoss needs an even B) leaves Song2Face's second LSTM cluster partly filled.  The input seeds avoid
    ReLU ties (see tests/test_conv_train_gpu.py)."""
    frozen = ofb.BN_PREFIXES[kind]
    x, oh, tp, gt = _inputs(B, seed)
    want_loss, want, running = ofb.loss_and_grads(kind, ow.make_state_dict(kind, seed=SEED_W[kind]), x, oh, tp, gt, frozen)
    m = _model(kind, dev, frozen)
    before = _running(m)
    loss = _step(m, dev, x, oh, tp, gt)
    _check_step(kind, m, loss, want_loss, want, running, before, frozen, f"all frozen B={B}")
    assert all(not m.get_submodule(n).training for n in frozen)


@pytest.mark.parametrize("kind", ["audio2mesh", "song2face"])
@pytest.mark.parametrize("parity", [0, 1])
def test_mixed_modes_step_vs_oracle(a2f_lib, dev, kind, parity):
    """every other BatchNorm frozen (both phases, so each layer of Audio2Mesh, the two in front of a conv included, runs
    frozen once and training once)"""
    frozen = ofb.BN_PREFIXES[kind][parity::2]
    x, oh, tp, gt = _inputs(16, 7)
    want_loss, want, running = ofb.loss_and_grads(kind, ow.make_state_dict(kind, seed=SEED_W[kind]), x, oh, tp, gt, frozen)
    m = _model(kind, dev, frozen)
    before = _running(m)
    loss = _step(m, dev, x, oh, tp, gt)
    _check_step(kind, m, loss, want_loss, want, running, before, frozen, f"mixed {parity}")


@pytest.mark.parametrize("kind", ["audio2mesh", "song2face"])
def test_frozen_train_forward_equals_inference(a2f_lib, dev, kind):
    m = _model(kind, dev, ofb.BN_PREFIXES[kind])
    x, oh, tp, _ = _inputs(12, 23)
    before = _running(m)
    with torch.no_grad():
        y_train = m(x.to(dev), oh.to(dev), tp.to(dev)).cpu()
        y_inf = m.eval()(x.to(dev), oh.to(dev), tp.to(dev)).cpu()
    err = float((y_train - y_inf).abs().max())
    print(f"{kind}: train() with every BatchNorm frozen vs eval() inference, max |diff| {err:.2e} m")
    assert err < 1e-5
    got = _running(m)
    assert all(torch.equal(got[k], before[k]) for k in before)


@pytest.mark.parametrize("kind", ["audio2mesh", "song2face"])
def test_frozen_affine_gets_no_gradient(a2f_lib, dev, kind):
    frozen = ofb.BN_PREFIXES[kind]
    x, oh, tp, gt = _inputs(4, 7)
    want_loss, want, running = ofb.loss_and_grads(kind, ow.make_state_dict(kind, seed=SEED_W[kind]), x, oh, tp, gt, frozen)
    m = _model(kind, dev, frozen)
    for name in frozen:
        m.get_submodule(name).requires_grad_(False)
    before = _running(m)
    loss = _step(m, dev, x, oh, tp, gt)
    for name in frozen:
        bn = m.get_submodule(name)
        assert bn.weight.grad is None and bn.bias.grad is None, name
    _check_step(kind, m, loss, want_loss, want, running, before, frozen, "frozen affine")


@pytest.mark.parametrize("kind", ["audio2mesh", "song2face"])
def test_mode_is_taped_at_forward(a2f_lib, dev, kind):
    """flipping every BatchNorm's mode between forward and backward must not change the gradients"""
    frozen = ofb.BN_PREFIXES[kind][::2]
    x, oh, tp, gt = _inputs(8, 7)
    want_loss, want, running = ofb.loss_and_grads(kind, ow.make_state_dict(kind, seed=SEED_W[kind]), x, oh, tp, gt, frozen)
    m = _model(kind, dev, frozen)
    before = _running(m)

    def flip():
        for name in ofb.BN_PREFIXES[kind]:
            bn = m.get_submodule(name)
            bn.train(not bn.training)
    loss = _step(m, dev, x, oh, tp, gt, between=flip)
    _check_step(kind, m, loss, want_loss, want, running, before, frozen, "flipped before backward")


@pytest.mark.parametrize("kind", ["audio2mesh", "song2face"])
def test_conv_model_trainer_freeze_bn(a2f_lib, dev, kind):
    from a2f_b200 import trainer as tr
    B = 16
    x, oh, tp, gt = _inputs(B, 9)
    want, _, _ = ofb.loss_and_grads(kind, ow.make_state_dict(kind, seed=SEED_W[kind]), x, oh, tp, gt, ofb.BN_PREFIXES[kind])
    m = _model(kind, dev, ())
    before = _running(m)
    t = tr.ConvModelTrainer(m, lr=1e-3, freeze_bn=True)
    losses = [t.step(x.to(dev), oh.to(dev), tp.to(dev), gt.to(dev)) for _ in range(3)]
    first = {k: float(v) for k, v in losses[0].items()}
    for k in ("loss", "rec_loss", "vel_loss"):
        assert abs(first[k] - want[k]) <= 2e-4 * abs(want[k]), (k, first[k], want[k])
    assert float(losses[-1]["loss"]) < float(losses[0]["loss"])
    assert m.training
    assert all(not m.get_submodule(n).training for n in ofb.BN_PREFIXES[kind])
    got = _running(m)
    assert all(torch.equal(got[k], before[k]) for k in before)
