"""Frozen-encoder fine-tuning of FaceFormer on the GPU: with parameters frozen (requires_grad False) the training step
keeps the forward and its loss bit for bit, computes the trainable gradients it computed before, leaves frozen
parameters without a gradient, and skips the backward launches below the lowest trainable op."""
import os

import numpy as np
import pytest
import torch

from oracle import inputs as oin, ref_train as ort, weights as ow

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PATTERNS = ("feature_encoder", "audio_encoder", "lower_layers", "layernorms")
ENC_WGRAD_SHAPES = {(2304, 768), (768, 768), (3072, 768), (768, 3072), (768, 512), (512, 1536), (512, 1024)}


def _freeze(m, pattern):
    ae = m.audio_encoder
    if pattern == "feature_encoder":
        ae.freeze_feature_encoder()
    elif pattern == "audio_encoder":
        ae.requires_grad_(False)
    elif pattern == "lower_layers":                   # layers 0-5 and everything below them
        for mod in (ae.feature_extractor, ae.feature_projection, ae.encoder.pos_conv_embed, ae.encoder.layer_norm):
            mod.requires_grad_(False)
        for blk in ae.encoder.layers[:6]:
            blk.requires_grad_(False)
    elif pattern == "layernorms":                     # the audio encoder's LayerNorm gamma / beta (and the decoder side)
        ae.requires_grad_(False)
        for n, p in ae.named_parameters():
            if "layer_norm" in n and "conv_layers" not in n:
                p.requires_grad_(True)
    elif pattern is not None:
        raise ValueError(pattern)
    return m


def _inputs():
    z = np.load(os.path.join(G, "faceformer_train.npz"))
    n, seed = int(z["n_samples"]), int(z["seed_in"])
    audio, oh = oin.audio(1, n, seed), oin.one_hot(1, 12, seed)
    tp = oin.batch_templates(1, seed, scale=100.0)
    gt = oin.gt_like((1, n * 60 // 16000, 5023, 3), tp[:, None], seed + 1, scale=100.0)
    return audio, oh, tp, gt


@pytest.fixture(scope="module")
def ff_sd():
    return ow.make_state_dict("faceformer", seed=13)


@pytest.fixture(scope="module")
def oracle(ff_sd):
    return ort.faceformer_loss_and_grads(ff_sd, *_inputs())


def _model(dev, sd, precision, pattern=None):
    from a2f_b200 import modules
    m = modules.Faceformer(15069, 12)
    m.load_state_dict(sd, strict=True)
    return _freeze(m.to(dev).eval().set_precision(precision), pattern)


def _autograd_step(dev, sd, precision, pattern):
    from a2f_b200 import modules, training
    m = _model(dev, sd, precision, pattern)
    audio, oh, tp, gt = (t.to(dev) for t in _inputs())
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    loss = modules.FaceFormerLoss()(m(audio, oh, tp), gt)
    loss["loss"].backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    grads = {k: (p.grad.detach().cpu() if p.grad is not None else None) for k, p in m.named_parameters()}
    trainable = {k for k, p in m.named_parameters() if p.requires_grad} - set(training.no_grad_params(m))
    return loss["loss"].detach().cpu(), grads, peak, trainable


_UNFROZEN = {}


def _unfrozen(dev, sd, precision):
    """Two unfrozen steps: the reference gradients and their run-to-run spread (fp32 atomics / reduce-add order)."""
    if precision not in _UNFROZEN:
        _UNFROZEN[precision] = (_autograd_step(dev, sd, precision, None), _autograd_step(dev, sd, precision, None))
    return _UNFROZEN[precision]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("pattern", PATTERNS)
def test_frozen_step_vs_unfrozen_and_oracle(a2f_lib, dev, ff_sd, oracle, pattern, precision):
    (l0, g0, peak0, _), (l1, g1, _, _) = _unfrozen(dev, ff_sd, precision)
    loss, grads, peak, trainable = _autograd_step(dev, ff_sd, precision, pattern)
    assert torch.equal(l0, l1) and torch.equal(loss, l0), (float(loss), float(l0))       # the forward is unchanged
    assert trainable and len(trainable) < len(grads)
    for k, g in grads.items():
        if k not in trainable:
            assert g is None, k
    # trainable gradients = the unfrozen ones to 1e-5, or to a few times the spread of two unfrozen runs where that is
    # larger: the atomics of the fp32 path alone move tiny-difference gradients (q_proj.bias) by ~1e-4 from run to run
    gmax = max(float(g.norm()) for k, g in g0.items() if g is not None)
    worst = 0.0
    for k in trainable:
        ref, n = 0.5 * (g0[k].double() + g1[k].double()), float(g0[k].norm())
        if n < 1e-6 * gmax:                           # mathematically-zero gradients (k_proj.bias)
            assert float(grads[k].norm()) < 10e-6 * gmax, k
            continue
        err = float((grads[k].double() - ref).norm())
        spread = float((g1[k].double() - g0[k].double()).norm())
        assert err <= max(1e-5 * n, 4.0 * spread + 1e-7 * n), (k, err / n, spread / n)
        worst = max(worst, err / n)
    # ... and the oracle's autograd, restricted to the trainable names, at test_faceformer_train_gpu's tolerances
    tot, want = oracle
    assert abs(float(loss) - tot["loss"]) < 1e-4 * abs(tot["loss"])
    omax = max(float(g.norm()) for g in want.values())
    z = np.load(os.path.join(G, "faceformer_train.npz"))
    noise = {str(n): float(v) for n, v in zip(z["names"], z["bf16_noise"])}
    for k in trainable:
        n = float(want[k].norm())
        if n < 1e-6 * omax:
            continue
        rel = float((grads[k].double() - want[k].double()).norm()) / n
        assert rel < (3e-3 if precision == "fp32" else max(8e-2, 3.0 * noise[k])), (k, rel)
    assert peak < peak0, (peak, peak0)
    print(f"{pattern} {precision}: {len(trainable)} trainable tensors, worst rel. diff to unfrozen {worst:.1e}, "
          f"peak {peak / 2**20:.0f} MiB (unfrozen {peak0 / 2**20:.0f} MiB)")


def _spy(monkeypatch):
    from a2f_b200 import ops
    calls = {}
    for name in ("mha_bwd", "conv0_bwd", "posconv_wgrad", "posconv_dgrad", "weight_norm_bwd", "add_strided3", "gemm_wgrad",
                 "layernorm_bwd", "interp_ln_bwd", "act_bwd"):
        fn = getattr(ops, name)

        def wrap(*a, _fn=fn, _name=name, **kw):
            calls.setdefault(_name, []).append((a, kw))
            return _fn(*a, **kw)
        monkeypatch.setattr(ops, name, wrap)
    return calls


@pytest.mark.parametrize("pattern", PATTERNS)
def test_pruned_backward_launches(a2f_lib, dev, ff_sd, pattern, monkeypatch):
    calls = _spy(monkeypatch)
    _autograd_step(dev, ff_sd, "bf16", pattern)
    n = {k: len(v) for k, v in calls.items()}
    enc_wgrad = [a for a, kw in calls["gemm_wgrad"] if tuple(a[2].shape) in ENC_WGRAD_SHAPES]
    assert "conv0_bwd" not in n and "add_strided3" not in n
    if pattern == "audio_encoder":
        for k in ("mha_bwd", "posconv_wgrad", "posconv_dgrad", "weight_norm_bwd", "layernorm_bwd", "interp_ln_bwd"):
            assert k not in n, k
        assert not enc_wgrad
    elif pattern == "feature_encoder":
        assert n["mha_bwd"] == 12 and n["posconv_dgrad"] == 1
        (_, kw), = calls["interp_ln_bwd"]
        assert kw["want_dx"] is False                 # the boundary: parameter gradients only
    elif pattern == "lower_layers":
        assert n["mha_bwd"] == 6 and "posconv_wgrad" not in n and "posconv_dgrad" not in n and "interp_ln_bwd" not in n
        assert len(enc_wgrad) == 6 * 4                # q|k|v (one fused GEMM), out_proj, intermediate, output
        assert all(kw["want_dx"] for _, kw in calls["layernorm_bwd"])
    elif pattern == "layernorms":
        assert not enc_wgrad and "posconv_wgrad" not in n and "weight_norm_bwd" not in n
        assert n["mha_bwd"] == 12 and n["layernorm_bwd"] == 25
        (_, kw), = calls["interp_ln_bwd"]
        assert kw["want_dx"] is False


def test_unfrozen_backward_launches_everything(a2f_lib, dev, ff_sd, monkeypatch):
    calls = _spy(monkeypatch)
    _autograd_step(dev, ff_sd, "bf16", None)
    n = {k: len(v) for k, v in calls.items()}
    assert n["mha_bwd"] == 12 and n["conv0_bwd"] == 1 and n["add_strided3"] == 6 and n["posconv_wgrad"] == 1
    assert all(kw.get("want_dx", True) for _, kw in calls["layernorm_bwd"] + calls["interp_ln_bwd"])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("C", [512, 768])
def test_layernorm_bwd_parameter_gradients_only(a2f_lib, dev, dtype, C):
    from a2f_b200 import ops
    g = torch.Generator().manual_seed(C)
    rows = 777
    x = (torch.randn(rows, C, generator=g) * 2 + 0.3).to(dtype)
    dy = torch.randn(rows, C, generator=g).to(dtype)
    gamma = torch.randn(C, generator=g) * 0.5 + 1
    xd, dyd, gd = x.to(dev), dy.to(dev), gamma.to(dev)
    full = [torch.zeros(C, device=dev) for _ in range(3)]
    dx = ops.layernorm_bwd(dyd, xd, gd, full[0], full[1], full[2])
    only = [torch.zeros(C, device=dev) for _ in range(2)]
    assert ops.layernorm_bwd(dyd, xd, gd, only[0], only[1], want_dx=False) is None
    beta_only = torch.zeros(C, device=dev)
    ops.layernorm_bwd(dyd, xd, gd, None, beta_only, want_dx=False)
    torch.cuda.synchronize()
    x64 = x.double().requires_grad_(True)
    g64 = gamma.double().requires_grad_(True)
    b64 = torch.zeros(C, dtype=torch.float64, requires_grad=True)
    torch.nn.functional.layer_norm(x64, (C,), g64, b64, 1e-5).backward(dy.double())
    for got, want in ((only[0], g64.grad), (only[1], b64.grad), (beta_only, b64.grad)):
        assert float((got.double().cpu() - want).norm() / want.norm()) < 1e-5
    for a, b in zip(only, full[:2]):
        assert float((a - b).norm() / b.norm()) < 1e-6
    assert float((dx.double().cpu() - x64.grad).norm() / x64.grad.norm()) < (1e-5 if dtype == torch.float32 else 1e-2)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_interp_ln_bwd_parameter_gradients_only(a2f_lib, dev, dtype):
    from a2f_b200 import ops
    g = torch.Generator().manual_seed(5)
    B, S, T, C = 3, 49, 59, 512                       # conv stack at 50 Hz -> 60 fps
    x = (torch.randn(B, S, C, generator=g) + 0.2).to(dtype)
    dy = torch.randn(B, T, C, generator=g).to(dtype)
    gamma = torch.randn(C, generator=g) * 0.5 + 1
    xd, dyd, gd = x.to(dev), dy.to(dev), gamma.to(dev)
    full = [torch.zeros(C, device=dev) for _ in range(2)]
    din = ops.interp_ln_bwd(xd, dyd, gd, full[0], full[1])
    only = [torch.zeros(C, device=dev) for _ in range(2)]
    assert ops.interp_ln_bwd(xd, dyd, gd, only[0], only[1], want_dx=False) is None
    torch.cuda.synchronize()
    # float64 torch: linear interpolation along time (align_corners=True), then LayerNorm
    x64 = x.double().requires_grad_(True)
    g64 = gamma.double().requires_grad_(True)
    b64 = torch.zeros(C, dtype=torch.float64, requires_grad=True)
    v = torch.nn.functional.interpolate(x64.transpose(1, 2), size=T, mode="linear", align_corners=True).transpose(1, 2)
    torch.nn.functional.layer_norm(v, (C,), g64, b64, 1e-5).backward(dy.double())
    for got, ref, want in ((only[0], full[0], g64.grad), (only[1], full[1], b64.grad)):
        assert float((got.double().cpu() - want).norm() / want.norm()) < 1e-5
        assert float((got - ref).norm() / ref.norm()) < 1e-6
    assert float((din.double().cpu() - x64.grad).norm() / x64.grad.norm()) < (1e-5 if dtype == torch.float32 else 1e-2)


def test_trainer_two_steps_frozen_feature_encoder_match_torch_adam(a2f_lib, dev):
    """As test_trainer_gpu's two-step check, with the feature encoder frozen in both: frozen values bit-unchanged,
    .grad None, no Adam moments for them."""
    from a2f_b200 import modules, trainer as tr
    from oracle import ref_models as orm
    n, lr = 6400, 1e-4
    audio, oh = oin.audio(1, n, 61), oin.one_hot(1, 12, 61)
    tp = oin.batch_templates(1, 61, scale=100.0)
    gt = oin.gt_like((1, 24, 5023, 3), tp[:, None], 62, scale=100.0)
    sd = ow.make_state_dict("faceformer", seed=13)
    m = modules.Faceformer(15069, 12)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).eval().set_precision("fp32")
    m.audio_encoder.freeze_feature_encoder()
    frozen = {k for k, p in m.named_parameters() if not p.requires_grad}
    t = tr.FaceformerTrainer(m, lr=lr, fps=60)
    assert t.exp_avg.numel() == t.flat.total and not frozen & {e[0] for e in t.flat.entries}
    got = [float(t.step(audio.to(dev), oh.to(dev), tp.to(dev), gt.to(dev))["loss"]) for _ in range(2)]
    params = {k: (v.detach().clone().requires_grad_(k not in frozen) if v.is_floating_point() and k != "PPE.pe" else v)
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
    print("frozen-feature-encoder trainer losses", got, "oracle", want)
    for a, b in zip(got, want):
        assert abs(a - b) < 1e-4 * abs(b)
    new = {k: p.detach().cpu() for k, p in m.named_parameters()}
    for k, p in m.named_parameters():
        if k in frozen:
            assert p.grad is None and torch.equal(new[k], sd[k]), k
    bad = tot = 0
    for k, p in params.items():
        if k in frozen or not (isinstance(p, torch.Tensor) and p.requires_grad) or k == "audio_encoder.masked_spec_embed":
            continue
        d = (new[k] - p.detach()).abs().reshape(-1)
        bad += int((d > 0.05 * lr).sum())
        tot += d.numel()
    assert bad < 2e-3 * tot


def test_graphed_frozen_step_equals_eager(a2f_lib, dev, ff_sd):
    from a2f_b200 import trainer as tr
    audio, oh, tp, gt = (x.to(dev) for x in _inputs())
    m = _model(dev, ff_sd, "bf16", "lower_layers")
    t = tr.FaceformerTrainer(m, lr=1e-4, fps=60)
    g = t.graphed(audio, oh, tp, gt)
    torch.cuda.synchronize()
    snap = [x.clone() for x in (t.flat.params, t.exp_avg, t.exp_avg_sq, t._step_dev)]
    frozen = {k: p.detach().clone() for k, p in m.named_parameters() if not p.requires_grad}
    l_replay = g(audio, oh, tp, gt)["loss"].clone()
    torch.cuda.synchronize()
    p_replay = t.flat.params.clone()
    for dst, src in zip((t.flat.params, t.exp_avg, t.exp_avg_sq, t._step_dev), snap):
        dst.copy_(src)
    t.flat.bump_versions()
    l_eager = t.step(audio, oh, tp, gt)["loss"].clone()
    torch.cuda.synchronize()
    assert torch.equal(l_replay, l_eager), (float(l_replay), float(l_eager))
    moved = (t.flat.params - snap[0]).abs()
    diff = (t.flat.params - p_replay).abs()
    assert float((diff > 0.05 * 1e-4).float().mean()) < 2e-3 and float(moved.max()) > 0
    for k, p in m.named_parameters():
        if k in frozen:
            assert p.grad is None and torch.equal(p.detach(), frozen[k]), k


def test_requires_grad_flipped_after_forward_does_not_change_the_backward(a2f_lib, dev, ff_sd):
    from a2f_b200 import training
    audio, oh, tp, gt = (x.to(dev) for x in _inputs())
    T = gt.shape[1]
    dout = torch.randn((1, T, 5023, 3), generator=torch.Generator().manual_seed(3)).to(dev)
    res = []
    for flip in (False, True):
        m = _model(dev, ff_sd, "fp32", "feature_encoder")
        with torch.no_grad():
            _, tape = training.forward_train(m, audio, oh.reshape(1, -1), tp.reshape(1, -1), 60)
            if flip:
                m.audio_encoder.feature_extractor.requires_grad_(True)        # frozen at forward time
                m.audio_encoder.encoder.layers[0].final_layer_norm.requires_grad_(False)   # trainable at forward time
            training.backward(m, tape, dout)
        torch.cuda.synchronize()
        res.append({k: (p.grad.cpu() if p.grad is not None else None) for k, p in m.named_parameters()})
    a, b = res
    gmax = max(float(g.norm()) for g in a.values() if g is not None)
    for k in a:
        assert (a[k] is None) == (b[k] is None), k
        if a[k] is not None:                          # equal up to the fp32 atomics' accumulation order
            assert float((a[k] - b[k]).norm()) <= 1e-3 * float(a[k].norm()) + 1e-6 * gmax, k
    assert a["audio_encoder.feature_extractor.conv_layers.3.conv.weight"] is None
    assert a["audio_encoder.encoder.layers.0.final_layer_norm.weight"] is not None


def test_trainer_refuses_a_changed_trainable_set(a2f_lib, dev, ff_sd):
    from a2f_b200 import lib as L, trainer as tr
    audio, oh, tp, gt = (x.to(dev) for x in _inputs())
    m = _model(dev, ff_sd, "bf16", "feature_encoder")
    t = tr.FaceformerTrainer(m, lr=1e-4, fps=60)
    t.step(audio, oh, tp, gt)
    m.audio_encoder.encoder.layers[2].requires_grad_(False)
    with pytest.raises(L.A2FError, match="trainable parameters changed"):
        t.step(audio, oh, tp, gt)
    m.audio_encoder.encoder.layers[2].requires_grad_(True)
    m.audio_encoder.feature_extractor.conv_layers[4].requires_grad_(True)
    with pytest.raises(L.A2FError, match="trainable parameters changed"):
        t.step(audio, oh, tp, gt)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_repack_touches_only_trainable_sources(a2f_lib, dev, ff_sd, precision):
    """After an optimizer step only operands of trainable parameters are re-derived (an operand of a frozen conv weight,
    overwritten here, stays as it is); a frozen weight modified in place (load_state_dict) is re-derived."""
    from a2f_b200 import trainer as tr, training
    audio, oh, tp, gt = (x.to(dev) for x in _inputs())
    m = _model(dev, ff_sd, precision, "feature_encoder")
    t = tr.FaceformerTrainer(m, lr=1e-4, fps=60)
    t.step(audio, oh, tp, gt)
    P, PB = m._packed(), training.packed_backward_weights(m)
    frozen_ops = (P["convs"][2], PB["convs"][2][0])
    keep = [x.clone() for x in frozen_ops]
    for x in frozen_ops:
        x.zero_()
    t.step(audio, oh, tp, gt)
    assert m._packed() is P and training.packed_backward_weights(m) is PB        # re-derived after the update
    torch.cuda.synchronize()
    assert all(not bool(x.any()) for x in frozen_ops)                # frozen sources: not re-derived
    ow_ = m.audio_encoder.encoder.layers[5].feed_forward.output_dense.weight.detach()
    dt = torch.bfloat16 if precision == "bf16" else torch.float32
    assert not torch.equal(ow_.cpu(), ff_sd["audio_encoder.encoder.layers.5.feed_forward.output_dense.weight"])
    assert torch.equal(PB["layers"][5]["f2_t"], ow_.t().to(dt))       # trainable: re-derived from the updated weight
    m.load_state_dict(m.state_dict(), strict=True)                    # in-place copy: every version counter moves
    P2, PB2 = m._packed(), training.packed_backward_weights(m)
    torch.cuda.synchronize()
    assert P2 is P and PB2 is PB
    for x, want in zip(frozen_ops, keep):
        assert torch.equal(x, want)
