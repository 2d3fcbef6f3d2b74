"""CPU checks of the encoder-dropout RNG contract (include/a2f.h) as restated in oracle/philox.py, and of the dropout-aware
oracle (oracle/ref_dropout.py) against the eval-mode oracle."""
import numpy as np
import pytest
import torch

from oracle import inputs as oin, philox, ref_dropout as ord_, ref_train as ort, weights as ow


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox_known_answers(ctr, key, want):
    """Random123's known-answer vectors for Philox4x32-10."""
    got = philox.philox4x32_10(ctr, key)
    assert " ".join("%08x" % int(w) for w in got) == want


def test_element_to_halfword_mapping():
    """Element e uses call g = e // 8 (counter (g lo, g hi, site, offset), key = seed) and half-word e % 8, low half of
    word (e % 8) // 2 first."""
    seed, offset, site = 0x0123456789ABCDEF, 7, 8 * 5 + philox.FFN_ACT
    u = philox.uniforms16(seed, offset, site, 40)
    for e in (0, 1, 6, 7, 8, 13, 39):
        w = philox.philox4x32_10((e // 8, 0, site, offset), (seed & 0xFFFFFFFF, seed >> 32))
        h = e % 8
        assert int(u[e]) == (int(w[h // 2]) >> (16 * (h % 2))) & 0xFFFF


def test_threshold_and_keep_fraction():
    assert philox.threshold(0.0) == 0 and philox.threshold(0.1) == 6554 and philox.threshold(0.5) == 32768
    assert philox.scale(0.1) == np.float32(1.0) / np.float32(0.9)
    k = philox.keep_mask(3, 0, philox.ENC_IN, 0.1, (600, 768))
    n = k.size
    q = 1 - philox.threshold(0.1) / 65536
    assert abs(k.mean() - q) < 5 * (q * (1 - q) / n) ** 0.5
    assert philox.keep_mask(3, 0, philox.ENC_IN, 0.0, (4, 8)).all()


def test_masks_depend_on_seed_offset_site_only():
    a = philox.encoder_dropout_masks(11, 0, {"hidden": .1, "activation": .1, "feat_proj": .1}, 2, 9)
    b = philox.encoder_dropout_masks(11, 1, {"hidden": .1, "activation": .1, "feat_proj": .1}, 2, 9)
    assert (a["enc_in"] != b["enc_in"]).any()                          # a new offset draws new masks
    assert (a["layers"][0]["attn_out"] != a["layers"][0]["ffn_out"]).any()   # sites are independent
    # an utterance's masks are rows b*T .. b*T+T-1 of the batch masks
    u1 = philox.utterance(a, 1)
    assert np.array_equal(u1["layers"][4]["ffn_act"], a["layers"][4]["ffn_act"][9:18])
    s = philox.encoder_dropout_masks(11, 0, {"hidden": .1}, 2, 9, skip={3})
    assert s["layers"][3] is None and np.array_equal(s["layers"][2]["attn_out"], a["layers"][2]["attn_out"])


@pytest.fixture(scope="module")
def small_step():
    sd = ow.make_state_dict("faceformer", seed=13)
    audio, oh = oin.audio(2, 4000, 5), oin.one_hot(2, 12, 5)
    tp = oin.batch_templates(2, 5, scale=100.0)
    gt = oin.gt_like((2, 15, 5023, 3), tp[:, None], 6, scale=100.0)
    return sd, audio, oh, tp, gt


def test_dropout_oracle_without_dropout_is_the_eval_oracle(small_step):
    """drop=None and all p = 0 reproduce oracle/ref_train.py bit for bit."""
    sd, audio, oh, tp, gt = small_step
    tot, want = ort.faceformer_loss_and_grads(sd, audio, oh, tp, gt)
    zero = philox.encoder_dropout_masks(5, 0, {"hidden": 0.0, "activation": 0.0, "feat_proj": 0.0}, 2, 15)
    for drop in (None, zero):
        t2, g2 = ord_.faceformer_loss_and_grads(sd, audio, oh, tp, gt, drop=drop)
        assert t2 == tot
        for k, g in want.items():                   # ref_train reports an unused parameter's gradient as zeros
            assert torch.equal(g2[k], g) if g2[k] is not None else not g.any(), k


def test_dropout_oracle_layerdrop_gives_no_gradient(small_step):
    sd, audio, oh, tp, gt = small_step
    drop = philox.encoder_dropout_masks(5, 0, {"hidden": .1, "activation": .1, "feat_proj": .1}, 2, 15, skip={2})
    tot, g = ord_.faceformer_loss_and_grads(sd, audio, oh, tp, gt, drop=drop)
    assert np.isfinite(tot["loss"])
    assert g["audio_encoder.encoder.layers.2.attention.q_proj.weight"] is None
    assert g["audio_encoder.encoder.layers.1.attention.q_proj.weight"] is not None
