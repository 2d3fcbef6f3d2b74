"""Frozen-encoder fine-tuning of FaceFormer, host side (no GPU): HF's freezing API on the drop-in's audio_encoder and
training.grad_plan, the one place that decides which gradients the training backward computes."""
import pytest
import torch

from oracle import weights as ow

FE = "audio_encoder.feature_extractor."
FE_PARAMS = {f"{FE}conv_layers.{i}.conv.weight" for i in range(7)} | {
    f"{FE}conv_layers.0.layer_norm.weight", f"{FE}conv_layers.0.layer_norm.bias"}


def _model():
    from a2f_b200 import modules
    return modules.Faceformer(15069, 12).eval()


def _frozen(m):
    return {n for n, p in m.named_parameters() if not p.requires_grad}


def _layer_ops(li):
    return [f"layers.{li}.{op}" for op in ("qkv", "out_proj", "ln", "f1", "f2", "fln")]


def test_freeze_feature_encoder_freezes_the_nine_feature_extractor_tensors():
    m = _model()
    assert m.audio_encoder.feature_extractor._requires_grad is True
    m.audio_encoder.freeze_feature_encoder()
    assert _frozen(m) == FE_PARAMS
    assert m.audio_encoder.feature_extractor._requires_grad is False
    m2 = _model()
    m2.audio_encoder.feature_extractor._freeze_parameters()
    assert _frozen(m2) == FE_PARAMS
    assert m2.audio_encoder.feature_extractor._requires_grad is False


def test_freezing_matches_hf_wav2vec2():
    """The same tensors HF's Wav2Vec2Model.freeze_feature_encoder() freezes in its own model (base architecture's
    feature encoder: group norm on conv 0, no conv bias), by name."""
    tf = pytest.importorskip("transformers")
    cfg = tf.Wav2Vec2Config(hidden_size=32, num_hidden_layers=1, num_attention_heads=2, intermediate_size=64,
                            num_conv_pos_embeddings=16, num_conv_pos_embedding_groups=2)
    hf = tf.Wav2Vec2Model(cfg)
    hf.freeze_feature_encoder()
    want = {"audio_encoder." + n for n, p in hf.named_parameters() if not p.requires_grad}
    assert hf.feature_extractor._requires_grad is False
    m = _model()
    m.audio_encoder.freeze_feature_encoder()
    assert _frozen(m) == want == FE_PARAMS


def test_state_dict_keys_shapes_dtypes_unchanged():
    sd = ow.make_state_dict("faceformer", seed=13)
    m = _model()
    m.load_state_dict(sd, strict=True)
    m.audio_encoder.freeze_feature_encoder()
    got = m.state_dict()
    assert len(got) == 237
    assert list(got.keys()) == list(sd.keys())
    assert all(got[k].shape == sd[k].shape and got[k].dtype == sd[k].dtype for k in sd)


def _plan(freeze):
    from a2f_b200 import training
    m = _model()
    freeze(m)
    return m, training.grad_plan(m)


def _check(m, plan, first_op):
    from a2f_b200 import training
    names = {n for n, p in m.named_parameters() if p.requires_grad} - set(training.no_grad_params(m))
    assert plan.params == names
    assert plan.ids == frozenset(id(p) for n, p in m.named_parameters() if n in names)
    assert plan.any == bool(names)
    ops_ = list(plan.ops)
    i = ops_.index(first_op) if first_op is not None else len(ops_)
    assert [op for op in ops_ if plan.runs(op)] == ops_[i:]
    assert [op for op in ops_ if plan.dgrad(op)] == ops_[i + 1:]


def test_op_order():
    _, plan = _plan(lambda m: None)
    assert plan.ops[:11] == ("conv0", "conv1", "conv2", "conv3", "conv4", "conv5", "conv6", "interp_ln", "projection",
                             "posconv", "enc_ln")
    assert plan.ops[11:-2] == tuple(op for li in range(12) for op in _layer_ops(li))
    assert plan.ops[-2:] == ("afm", "decoder")
    m = _model().train()                              # SpecAugment runs in train(): its embedding is an op of its own
    from a2f_b200 import training
    p = training.grad_plan(m)
    assert p.ops[8:11] == ("projection", "spec_embed", "posconv")
    assert "audio_encoder.masked_spec_embed" in p.params


def test_plan_nothing_frozen_computes_everything():
    m, plan = _plan(lambda m: None)
    _check(m, plan, "conv0")
    assert len(plan.params) == len(list(m.parameters())) - 1          # masked_spec_embed: no SpecAugment in eval()


def test_plan_feature_encoder_frozen():
    m, plan = _plan(lambda m: m.audio_encoder.freeze_feature_encoder())
    _check(m, plan, "interp_ln")
    assert not plan.params & FE_PARAMS


def test_plan_audio_encoder_frozen():
    m, plan = _plan(lambda m: m.audio_encoder.requires_grad_(False))
    _check(m, plan, "afm")
    assert not any(n.startswith("audio_encoder.") for n in plan.params)
    assert "audio_feature_map.weight" in plan.params and "vertice_map_r.weight" in plan.params


def test_plan_lower_layers_frozen():
    def freeze(m):
        ae = m.audio_encoder
        for mod in (ae.feature_extractor, ae.feature_projection, ae.encoder.pos_conv_embed, ae.encoder.layer_norm):
            mod.requires_grad_(False)
        for blk in ae.encoder.layers[:6]:
            blk.requires_grad_(False)
    m, plan = _plan(freeze)
    _check(m, plan, "layers.6.qkv")
    assert not any(n.startswith("audio_encoder.encoder.layers.5.") for n in plan.params)


def test_plan_layernorms_only():
    """Only the encoder's LayerNorm gamma / beta and the decoder side train: the boundary is the feature-projection
    LayerNorm, whose parameter gradients are computed but not its input gradient."""
    def freeze(m):
        m.audio_encoder.requires_grad_(False)
        for n, p in m.audio_encoder.named_parameters():
            if "layer_norm" in n and "conv_layers" not in n:
                p.requires_grad_(True)
    m, plan = _plan(freeze)
    _check(m, plan, "interp_ln")
    assert "audio_encoder.encoder.layers.3.final_layer_norm.bias" in plan.params
    assert "audio_encoder.encoder.layers.3.feed_forward.output_dense.bias" not in plan.params


def test_plan_top_final_layernorm_only():
    def freeze(m):
        m.requires_grad_(False)
        m.audio_encoder.encoder.layers[11].final_layer_norm.weight.requires_grad_(True)
    m, plan = _plan(freeze)
    _check(m, plan, "layers.11.fln")
    assert plan.params == {"audio_encoder.encoder.layers.11.final_layer_norm.weight"}


def test_plan_decoder_only_and_nothing():
    m, plan = _plan(lambda m: [p.requires_grad_(False) for n, p in m.named_parameters()
                               if n.startswith(("audio_encoder.", "audio_feature_map."))])
    _check(m, plan, "decoder")
    m, plan = _plan(lambda m: m.requires_grad_(False))
    _check(m, plan, None)
    assert not plan.any


def test_plan_decoder_frozen_encoder_trainable():
    def freeze(m):
        for n, p in m.named_parameters():
            if not n.startswith("audio_encoder."):
                p.requires_grad_(False)
    m, plan = _plan(freeze)
    _check(m, plan, "conv0")
    assert "vertice_map_r.weight" not in plan.params


def test_plan_single_projection_and_single_layernorm_parameter():
    """q but not k / v; one LayerNorm beta: per parameter, the op's position decides the data gradients."""
    def freeze(m):
        m.requires_grad_(False)
        m.audio_encoder.encoder.layers[4].attention.q_proj.weight.requires_grad_(True)
        m.audio_encoder.encoder.layers[9].layer_norm.bias.requires_grad_(True)
    m, plan = _plan(freeze)
    _check(m, plan, "layers.4.qkv")
    assert plan.params == {"audio_encoder.encoder.layers.4.attention.q_proj.weight",
                           "audio_encoder.encoder.layers.9.layer_norm.bias"}


def test_plan_is_a_snapshot():
    from a2f_b200 import training
    m = _model()
    m.audio_encoder.freeze_feature_encoder()
    plan = training.grad_plan(m)
    m.audio_encoder.requires_grad_(True)
    assert not plan.params & FE_PARAMS and plan.ops[plan.first] == "interp_ln"
