"""Train-mode dropout and LayerDrop of the wav2vec2 encoder (modules.Faceformer.encoder_dropout) on the GPU: the masks
against the numpy restatement of the RNG contract (oracle/philox.py), the training step against the oracle's autograd
under the same masks (oracle/ref_dropout.py), CUDA-graph replay, LayerDrop's missing gradients and Adam skipping."""
import os

import numpy as np
import pytest
import torch

from oracle import inputs as oin, philox, ref_dropout as ord_, weights as ow

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
P01 = {"hidden": 0.1, "attention": 0.1, "activation": 0.1, "feat_proj": 0.1, "layerdrop": 0.0}
SEED = 0xC0FFEE1234


@pytest.fixture(scope="module")
def ff_sd():
    return ow.make_state_dict("faceformer", seed=13)


def _inputs(n_samples, seed, B):
    audio, oh = oin.audio(B, n_samples, seed), oin.one_hot(B, 12, seed)
    tp = oin.batch_templates(B, seed, scale=100.0)
    T = n_samples * 60 // 16000
    gt = oin.gt_like((B, T, 5023, 3), tp[:, None], seed + 1, scale=100.0)
    return audio, oh, tp, gt


def _model(dev, sd, precision, p=P01, switch=True, seed=SEED):
    from a2f_b200 import modules
    m = modules.Faceformer(15069, 12)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).train().set_precision(precision)
    m.spec_augment = False
    m.encoder_dropout = switch
    m.dropout_p = dict(p)
    m.dropout_seed = seed
    return m


def _glue_step(m, dev, audio, oh, tp, gt):
    from a2f_b200 import modules
    pred = m(audio.to(dev), oh.to(dev), tp.to(dev))
    loss = modules.FaceFormerLoss()(pred, gt.to(dev))
    loss["loss"].backward()
    torch.cuda.synchronize()
    grads = {k: (p.grad.detach().cpu() if p.grad is not None else None) for k, p in m.named_parameters()}
    return {k: float(v) for k, v in loss.items()}, grads


def _masks(B, T, p=P01, skip=(), offset=0, seed=SEED):
    return philox.encoder_dropout_masks(seed, offset, p, B, T, skip)


def _compare_fp32(grads, want, tol=3e-3):
    """Per-tensor relative L2 error, the bound of test_train_step_fp32_vs_oracle_and_golden."""
    gmax = max(float(g.norm()) for g in want.values() if g is not None)
    worst, worst_k = 0.0, None
    for k, g in want.items():
        if g is None:
            continue
        n = float(g.norm())
        if n < 1e-6 * gmax:
            assert float(grads[k].norm()) < 1e-5 * gmax, k
            continue
        rel = float((grads[k].double() - g.double()).norm()) / n
        if rel > worst:
            worst, worst_k = rel, k
    assert worst < tol, (worst_k, worst)
    return worst, worst_k


# ---------------------------------------------------------------------------------------------------------------- masks
@pytest.mark.parametrize("T", [41, 60, 80, 81, 150, 160, 161, 200, 301])
def test_mask_matches_numpy_philox(a2f_lib, dev, T):
    from a2f_b200 import lib as L, ops, training
    B = 2
    for seed, offset in ((SEED, 0), (0xF0123456789ABCDE, 12345)):         # a key with the top bit set, a later offset
        so = torch.tensor([training._i64(seed), offset], dtype=torch.int64, device=dev)
        sites = [(L.DROP_FEAT_PROJ, 768), (L.DROP_ENC_IN, 768)]
        for l in (0, 11):
            sites += [(8 * l + L.DROP_ATTN_OUT, 768), (8 * l + L.DROP_FFN_ACT, 3072), (8 * l + L.DROP_FFN_OUT, 768)]
        Tp = (T + 7) // 8 * 8
        sites = [(site, (B * T, C)) for site, C in sites] + [(8 * l + L.DROP_ATTN_PROB, (B, 12, T, Tp)) for l in (0, 11)]
        for site, shape in sites:
            got = ops.dropout_mask(0.1, site, so, shape).cpu().numpy().astype(bool)
            want = philox.keep_mask(seed, offset, site, 0.1, shape)
            assert np.array_equal(got, want), (seed, offset, site)
            q = 1 - philox.threshold(0.1) / 65536
            assert abs(got.mean() - q) < 5 * (q * (1 - q) / got.size) ** 0.5


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_dropout_apply_matches_mask(a2f_lib, dev, dtype):
    from a2f_b200 import lib as L, ops
    M, C, p = 2 * 150, 3072, 0.1
    so = torch.tensor([SEED, 3], dtype=torch.int64, device=dev)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(M, C, generator=g).to(dev, dtype)
    r = torch.randn(M, C, generator=g).to(dev, dtype)
    keep = torch.as_tensor(philox.keep_mask(SEED, 3, 8 * 4 + L.DROP_FFN_ACT, p, (M, C))).to(dev)
    sc = float(philox.scale(p))
    want = torch.where(keep, x.float() * sc, torch.zeros((), device=dev))
    y = ops.dropout_apply(x, p, 8 * 4 + L.DROP_FFN_ACT, so)
    assert torch.equal(y, want.to(dtype))                       # zero exactly where dropped, x / (1 - p) elsewhere
    y = ops.dropout_apply(x, p, 8 * 4 + L.DROP_FFN_ACT, so, resid=r)
    assert torch.equal(y, (want + r.float()).to(dtype))
    xc = x.clone()
    ops.dropout_apply(xc, p, 8 * 4 + L.DROP_FFN_ACT, so, out=xc)  # in place
    assert torch.equal(xc, want.to(dtype))
    assert torch.equal(ops.dropout_apply(x, 0.0, 0, so), x)     # p = 0 is a copy


@pytest.mark.parametrize("T", [60, 200, 301])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_attention_dropout_fwd_bwd_vs_float64(a2f_lib, dev, dtype, T):
    """Attention-probability dropout in the training kernels (T = 60: short-clip kernel, 200 / 301: flash kernel; fp32:
    SIMT kernels) against a float64 reference built on the materialised mask: O = (P o Z/(1-p)) V, the LSE of the undropped
    softmax, and dQ / dK / dV."""
    from a2f_b200 import lib as L, ops
    B, p, site = 2, 0.1, 8 * 5 + L.DROP_ATTN_PROB
    Tp = (T + 7) // 8 * 8
    g = torch.Generator().manual_seed(T)
    qkv = (torch.randn((B, T, 2304), generator=g) * 0.5).to(dev, dtype)
    dout = torch.randn((B, T, 768), generator=g).to(dev, dtype)
    so = torch.tensor([SEED, 17], dtype=torch.int64, device=dev)
    keep = ops.dropout_mask(p, site, so, (B, 12, T, Tp))[..., :T].cpu().double()
    qq = qkv.double().cpu().requires_grad_(True)
    q, k, v = [t.view(B, T, 12, 64).transpose(1, 2) for t in qq.split(768, dim=-1)]
    s_ = q @ k.transpose(2, 3) * 0.125
    o = ((torch.softmax(s_, -1) * keep * float(philox.scale(p))) @ v).transpose(1, 2).reshape(B, T, 768)
    o.backward(dout.double().cpu())
    out = torch.empty((B, T, 768), device=dev, dtype=dtype)
    lse = torch.empty((B, 12, T), device=dev)
    out32 = torch.empty((B, T, 768), device=dev) if dtype == torch.bfloat16 else None
    ops.mha_lse(qkv, out, lse, B, T, out_f32=out32, dropout=(p, site, so))
    dqkv = ops.mha_bwd(qkv, out, dout, lse, B, T, out_f32=out32, dropout=(p, site, so))
    torch.cuda.synchronize()
    err = lambda a, b: float((a.double().cpu() - b.double()).abs().max())          # noqa: E731
    fp32 = dtype == torch.float32
    assert err(lse, torch.logsumexp(s_, -1).detach()) < (1e-4 if fp32 else 2e-2)
    assert err(out, o.detach()) < (1e-4 if fp32 else 2e-2)
    if out32 is not None:
        assert err(out32, o.detach()) < 1e-2
    e = err(dqkv, qq.grad)
    print(f"attention dropout {dtype} T={T}: max |d qkv err| {e:.2e}")
    assert e < (1e-4 if fp32 else 8e-2)
    # the same call without dropout differs (the mask is applied at all)
    out0 = torch.empty_like(out)
    ops.mha_lse(qkv, out0, torch.empty_like(lse), B, T, out_f32=None if fp32 else torch.empty_like(out32))
    assert not torch.equal(out0, out)


# ---------------------------------------------------------------------------------------------------------------- step
@pytest.mark.parametrize("B", [1, 2])
def test_train_step_fp32_with_dropout_vs_oracle(a2f_lib, dev, ff_sd, B):
    if B == 1:
        z = np.load(os.path.join(G, "faceformer_train.npz"))
        n, s = int(z["n_samples"]), int(z["seed_in"])
    else:
        n, s = 6400, 43
    audio, oh, tp, gt = _inputs(n, s, B)
    T = n * 60 // 16000
    m = _model(dev, ff_sd, "fp32")
    loss, grads = _glue_step(m, dev, audio, oh, tp, gt)
    assert int(m._drop_state[1]) == 1                                     # one forward = one offset
    tot, want = ord_.faceformer_loss_and_grads(ff_sd, audio, oh, tp, gt, drop=_masks(B, T))
    assert abs(loss["loss"] - tot["loss"]) < 1e-4 * abs(tot["loss"]), (loss, tot)
    worst, k = _compare_fp32(grads, want)
    print(f"fp32 dropout step B={B}: loss {loss['loss']:.6f} (oracle {tot['loss']:.6f}); worst rel grad err {worst:.2e} ({k})")


def test_train_step_bf16_with_dropout_vs_oracle(a2f_lib, dev, ff_sd):
    z = np.load(os.path.join(G, "faceformer_train.npz"))
    n = int(z["n_samples"])
    audio, oh, tp, gt = _inputs(n, int(z["seed_in"]), 1)
    m = _model(dev, ff_sd, "bf16")
    loss, grads = _glue_step(m, dev, audio, oh, tp, gt)
    tot, want = ord_.faceformer_loss_and_grads(ff_sd, audio, oh, tp, gt, drop=_masks(1, n * 60 // 16000))
    assert abs(loss["loss"] - tot["loss"]) < 1e-4 * abs(tot["loss"]), (loss, tot)
    dot = n1 = n2 = 0.0
    for k, g in want.items():
        if g is None:
            continue
        a, b = grads[k].double().reshape(-1), g.double().reshape(-1)
        dot, n1, n2 = dot + float(a @ b), n1 + float(a @ a), n2 + float(b @ b)
    cos = dot / (n1 * n2) ** 0.5
    print(f"bf16 dropout step: loss {loss['loss']:.6f} (oracle {tot['loss']:.6f}); gradient cosine {cos:.4f}")
    assert cos > 0.97, cos


def test_switch_on_with_zero_p_is_switch_off(a2f_lib, dev, ff_sd):
    """p = 0 everywhere with the switch on runs the switch-off kernels: the taped forward is identical bit for bit.  With
    p = 0.1 the loss moves by more than the bf16 step's 1e-4 agreement with the oracle."""
    from a2f_b200 import modules, training
    audio, oh, tp, gt = _inputs(6400, 7, 2)
    outs = {}
    for name, p, switch in (("off", P01, False), ("zero", {k: 0.0 for k in P01}, True), ("on", P01, True)):
        m = _model(dev, ff_sd, "bf16", p=p, switch=switch)
        with torch.no_grad():
            out, tape = training.forward_train(m, audio.to(dev), oh.to(dev), tp.to(dev).reshape(2, -1), 60)
            loss = modules.FaceFormerLoss()(out, gt.to(dev))["loss"]
        outs[name] = (out.cpu(), tape["hs"].cpu(), float(loss))
    assert torch.equal(outs["off"][0], outs["zero"][0]) and torch.equal(outs["off"][1], outs["zero"][1])
    # the backward takes other branches with the switch on (masked bias / weight / data gradients); with p = 0 it must
    # launch exactly the switch-off kernels, and the gradients agree within the run-to-run spread of the fp32 SIMT
    # weight-gradient atomics (3e-3 per tensor, test_train_step_fp32_vs_oracle_and_golden)
    a1, oh1, tp1, gt1 = _inputs(6400, 43, 1)
    runs = []
    for kw in ({"switch": False}, {"p": {k: 0.0 for k in P01}}):
        m = _model(dev, ff_sd, "fp32", **kw)
        n0 = a2f_lib.a2f_launch_count()
        g = _glue_step(m, dev, a1, oh1, tp1, gt1)[1]
        runs.append((int(a2f_lib.a2f_launch_count() - n0), g))
    (na, ga), (nb, gb) = runs
    assert na == nb
    assert all((ga[k] is None) == (gb[k] is None) for k in ga)
    _compare_fp32(gb, ga)
    moved = abs(outs["on"][2] - outs["off"][2]) / abs(outs["off"][2])
    print(f"loss with dropout p=0.1 moved by {moved:.2e} (relative)")
    assert moved > 1e-4


# ---------------------------------------------------------------------------------------------------------------- graph
def test_graphed_step_replays_dropout(a2f_lib, dev, ff_sd):
    """A replay equals the eager step at the same (seed, offset) (loss bit for bit), and every replay advances the offset
    by one: the next replay draws new masks."""
    from a2f_b200 import trainer as tr
    audio, oh, tp, gt = (t.to(dev) for t in _inputs(16000, 9, 2))
    m = _model(dev, ff_sd, "bf16")
    t = tr.FaceformerTrainer(m, lr=1e-4, fps=60)
    g = t.graphed(audio, oh, tp, gt)
    torch.cuda.synchronize()
    snap = [x.clone() for x in (t.flat.params, t.exp_avg, t.exp_avg_sq, t._step_dev, m._drop_state)]
    off0 = int(m._drop_state[1])
    l_replay = g(audio, oh, tp, gt)["loss"].clone()
    torch.cuda.synchronize()
    assert int(m._drop_state[1]) == off0 + 1
    p_replay = t.flat.params.clone()
    for dst, src in zip((t.flat.params, t.exp_avg, t.exp_avg_sq, t._step_dev, m._drop_state), snap):
        dst.copy_(src)
    t.flat.bump_versions()
    l_eager = t.step(audio, oh, tp, gt)["loss"].clone()
    torch.cuda.synchronize()
    assert int(m._drop_state[1]) == off0 + 1
    assert torch.equal(l_replay, l_eager), (float(l_replay), float(l_eager))
    moved = (t.flat.params - snap[0]).abs()
    diff = (t.flat.params - p_replay).abs()
    assert float((diff > 0.05 * 1e-4).float().mean()) < 2e-3 and float(moved.max()) > 0
    g(audio, oh, tp, gt)
    torch.cuda.synchronize()
    assert int(m._drop_state[1]) == off0 + 2


# ---------------------------------------------------------------------------------------------------------------- LayerDrop
SKIP = frozenset({3, 7})


def _force_skip(monkeypatch):
    from a2f_b200 import training
    monkeypatch.setattr(training, "_draw_layerdrop", lambda model, p: SKIP)


def test_layerdrop_step_vs_oracle_and_no_grads(a2f_lib, dev, ff_sd, monkeypatch):
    _force_skip(monkeypatch)
    audio, oh, tp, gt = _inputs(6400, 43, 1)
    p = dict(P01, layerdrop=0.1)
    m = _model(dev, ff_sd, "fp32", p=p)
    loss, grads = _glue_step(m, dev, audio, oh, tp, gt)
    for k, g in grads.items():
        skipped = any(k.startswith(f"audio_encoder.encoder.layers.{l}.") for l in SKIP)
        assert (g is None) == (skipped or k == "audio_encoder.masked_spec_embed"), k
    tot, want = ord_.faceformer_loss_and_grads(ff_sd, audio, oh, tp, gt, drop=_masks(1, 24, p, skip=SKIP))
    assert abs(loss["loss"] - tot["loss"]) < 1e-4 * abs(tot["loss"]), (loss, tot)
    _compare_fp32(grads, want)


def test_layerdrop_trainer_leaves_skipped_layers_untouched(a2f_lib, dev, ff_sd, monkeypatch):
    from a2f_b200 import lib as L, trainer as tr, training
    _force_skip(monkeypatch)
    audio, oh, tp, gt = (t.to(dev) for t in _inputs(6400, 43, 1))
    m = _model(dev, ff_sd, "fp32", p=dict(P01, layerdrop=0.1))
    t = tr.FaceformerTrainer(m, lr=1e-4, fps=60)
    with pytest.raises(L.A2FError, match="LayerDrop"):
        t.graphed(audio, oh, tp, gt)
    t.step(audio, oh, tp, gt)
    torch.cuda.synchronize()
    for name, p, o, n, _ in t.flat.entries:
        if not name.startswith("audio_encoder.encoder.layers."):
            continue
        l = int(name.split(".")[3])
        same = torch.equal(p.detach().cpu(), ff_sd[name])
        if l in SKIP:
            assert same and not t.exp_avg[o:o + n].any() and not t.exp_avg_sq[o:o + n].any(), name
        elif name.endswith("weight") and "layer_norm" not in name:
            assert not same, name
    # the next step without skips: the skipped layers take their first Adam step (step count 1), the others their second
    monkeypatch.setattr(training, "_draw_layerdrop", lambda model, p: frozenset())
    t.step(audio, oh, tp, gt)
    st = t._stage_steps
    assert st[12 - 3] == 1 and st[12 - 7] == 1 and st[12 - 0] == 2 and st[0] == 2


def test_graph_refuses_layerdrop(a2f_lib, dev, ff_sd):
    from a2f_b200 import lib as L, trainer as tr
    audio, oh, tp, gt = (t.to(dev) for t in _inputs(6400, 43, 1))
    m = _model(dev, ff_sd, "bf16", p=dict(P01, layerdrop=0.1))
    with pytest.raises(L.A2FError, match="LayerDrop"):
        tr.FaceformerTrainer(m).graphed(audio, oh, tp, gt)


# ---------------------------------------------------------------------------------------------------------------- replicas
def test_replicas_draw_different_masks_and_the_same_layerdrop(a2f_lib, dev, ff_sd):
    """The data-parallel trainer folds the rank into the Philox key: rank 1 draws other dropout masks than rank 0 from
    the same seed, while the host-side LayerDrop draws (seeded with the seed alone) agree."""
    from a2f_b200 import lib as L, ops, training
    ms = [_model(dev, ff_sd, "bf16", p=dict(P01, layerdrop=0.5)) for _ in range(2)]
    training.set_dropout_rank(ms[1], 1)
    states = [training._dropout_state(m, dev) for m in ms]
    assert int(states[0][0]) == training._i64(SEED) and int(states[1][0]) == training._i64(training.dropout_key(SEED, 1))
    masks = [ops.dropout_mask(0.1, L.DROP_ENC_IN, st, (64, 768)) for st in states]
    assert not torch.equal(masks[0], masks[1])
    want = philox.keep_mask(training.dropout_key(SEED, 1), 0, L.DROP_ENC_IN, 0.1, (64, 768))
    assert np.array_equal(masks[1].cpu().numpy().astype(bool), want)
    for _ in range(4):
        assert training._draw_layerdrop(ms[0], 0.5) == training._draw_layerdrop(ms[1], 0.5)
