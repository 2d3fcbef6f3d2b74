"""TEST INFRASTRUCTURE -- numpy restatement of the encoder-dropout RNG contract of include/a2f.h ("Encoder dropout").

Philox4x32-10 (Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC'11; the Random123
constants), vectorised over counters.  A keep mask is a function of (seed, offset, site, element index) only, so the
masks the CUDA kernels apply can be regenerated here bit for bit.
"""
from __future__ import annotations

from typing import Dict, Iterable, Optional

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK32 = np.uint64(0xFFFFFFFF)

# site ids (include/a2f.h A2F_DROP_*): 8 * layer + kind, and the two sites in front of the layers
ATTN_PROB, ATTN_OUT, FFN_ACT, FFN_OUT = 0, 1, 2, 3
FEAT_PROJ, ENC_IN = 96, 97
N_LAYERS = 12
N_HEADS = 12


def philox4x32_10(ctr, key):
    """ctr: 4 arrays (or ints) of uint32 counter words, key: 2 of key words -> 4 uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) for x in ctr]
    k0, k1 = (np.uint64(int(x)) for x in key)
    for r in range(10):
        if r:
            k0, k1 = (k0 + W0) & _MASK32, (k1 + W1) & _MASK32
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK32]
    return [x.astype(np.uint32) for x in c]


def threshold(p: float) -> int:
    """Keep iff the 16-bit uniform is >= round(p * 65536) (computed in fp32 like the kernels, round half to even)."""
    t = float(np.rint(np.float32(p) * np.float32(65536.0)))
    return int(min(max(t, 0.0), 65536.0))


def scale(p: float) -> np.float32:
    return np.float32(1.0) / (np.float32(1.0) - np.float32(p))


def uniforms16(seed: int, offset: int, site: int, n: int) -> np.ndarray:
    """The 16-bit values of elements 0..n-1 of one site (uint32 array of length n)."""
    seed &= (1 << 64) - 1
    g = np.arange((n + 7) // 8, dtype=np.uint64)
    words = philox4x32_10((g & _MASK32, g >> np.uint64(32), np.full_like(g, site), np.full_like(g, offset & 0xFFFFFFFF)),
                          (seed & 0xFFFFFFFF, seed >> 32))
    w = np.stack(words, axis=1)                                          # [groups, 4]
    u = np.stack([w & np.uint32(0xFFFF), w >> np.uint32(16)], axis=2)     # [groups, 4, 2]: low half first
    return u.reshape(-1)[:n]


def keep_mask(seed: int, offset: int, site: int, p: float, shape) -> np.ndarray:
    """bool keep mask of one site over its logical tensor `shape` (row-major linear index)."""
    n = int(np.prod(shape))
    if p == 0:
        return np.ones(shape, dtype=bool)
    return (uniforms16(seed, offset, site, n) >= threshold(p)).reshape(shape)


def encoder_dropout_masks(seed: int, offset: int, p: Dict[str, float], B: int, T: int,
                          skip: Iterable[int] = ()) -> Dict:
    """Every mask of one training forward of the wav2vec2 encoder over the whole batch ([B*T, C] row-major; utterance b
    owns rows b*T .. b*T+T-1; the attention probabilities are [B, 12, T, Tp], Tp = ceil(T/8)*8, keys >= T unused).
    p: the drop probabilities by key ("hidden", "attention", "activation", "feat_proj"); skip: layers removed by
    LayerDrop (they draw nothing).  Returns {"p": p, "T": T, "feat_proj", "enc_in", "layers": [per layer
    {"attn_prob", "attn_out", "ffn_act", "ffn_out"} or None]}."""
    M = B * T
    Tp = (T + 7) // 8 * 8
    skip = set(skip)
    ph, pa, pf, pt = p.get("hidden", 0.0), p.get("activation", 0.0), p.get("feat_proj", 0.0), p.get("attention", 0.0)
    out = {"p": dict(p), "T": T,
           "feat_proj": keep_mask(seed, offset, FEAT_PROJ, pf, (M, 768)),
           "enc_in": keep_mask(seed, offset, ENC_IN, ph, (M, 768)), "layers": []}
    for l in range(N_LAYERS):
        if l in skip:
            out["layers"].append(None)
            continue
        out["layers"].append({"attn_prob": keep_mask(seed, offset, 8 * l + ATTN_PROB, pt, (B, N_HEADS, T, Tp)),
                              "attn_out": keep_mask(seed, offset, 8 * l + ATTN_OUT, ph, (M, 768)),
                              "ffn_act": keep_mask(seed, offset, 8 * l + FFN_ACT, pa, (M, 3072)),
                              "ffn_out": keep_mask(seed, offset, 8 * l + FFN_OUT, ph, (M, 768))})
    return out


def utterance(drop: Optional[Dict], b: int) -> Optional[Dict]:
    """The masks of utterance b (global batch index) out of encoder_dropout_masks(): rows b*T .. b*T+T-1 of each."""
    if drop is None:
        return None
    T = drop["T"]
    sl = lambda m: m[b * T:(b + 1) * T]                                            # noqa: E731
    sl_attn = lambda m: m[b:b + 1, :, :, :T]                                         # noqa: E731
    return {"p": drop["p"], "T": T, "feat_proj": sl(drop["feat_proj"]), "enc_in": sl(drop["enc_in"]),
            "layers": [None if d is None else {k: (sl_attn(v) if k == "attn_prob" else sl(v)) for k, v in d.items()}
                       for d in drop["layers"]]}
