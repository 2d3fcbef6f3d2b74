"""GPU parity of a2f_gemm / a2f_posconv (SIMT fp32 and tcgen05 back ends) against fp64 CPU matmuls of the same
(bf16-rounded where applicable) operands."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _ref(a, w, bias=None, act=0, resid=None, tmpl=None, rows_per_tmpl=1):
    y = a.double().cpu() @ w.double().cpu().T
    if bias is not None:
        y = y + bias.double().cpu()
    if act == 1:
        y = torch.relu(y)
    elif act == 2:
        y = F.gelu(y)
    elif act == 3:
        y = torch.tanh(y)
    if resid is not None:
        y = y + resid.double().cpu()
    if tmpl is not None:
        idx = torch.arange(y.shape[0]) // rows_per_tmpl
        y = y + tmpl.double().cpu()[idx]
    return y


def _rand(shape, dev, seed, dtype=torch.float32, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (scale * torch.randn(shape, generator=g)).to(dev).to(dtype)


@pytest.mark.parametrize("M,N,K", [(64, 64, 16), (130, 70, 50), (257, 333, 129), (9, 15069, 50)])
def test_simt_fp32_plain(a2f_lib, dev, M, N, K):
    from a2f_b200 import ops, lib as L
    a, w, b = _rand((M, K), dev, 1), _rand((N, K), dev, 2), _rand((N,), dev, 3)
    out = torch.empty((M, N), device=dev)
    ops.gemm(a, w, out, bias=b, act=L.ACT_TANH, backend=L.SIMT_F32)
    want = _ref(a, w, b, 3)
    assert float((out.cpu().double() - want).abs().max()) < 2e-5


def test_simt_fp32_epilogue_resid_tmpl(a2f_lib, dev):
    from a2f_b200 import ops, lib as L
    M, N, K = 40, 301, 64
    a, w, b = _rand((M, K), dev, 4), _rand((N, K), dev, 5), _rand((N,), dev, 6)
    r, t = _rand((M, N), dev, 7), _rand((4, N), dev, 8)
    out = torch.empty((M, N), device=dev)
    ops.gemm(a, w, out, bias=b, act=L.ACT_GELU, resid=r, tmpl=t, rows_per_tmpl=10, backend=L.SIMT_F32)
    want = _ref(a, w, b, 2, r, t, 10)
    assert float((out.cpu().double() - want).abs().max()) < 2e-5


TC_CASES = [
    # M, N, K, act, use_resid, out_bf16, use_tmpl
    (128, 256, 64, 0, False, False, False),
    (256, 512, 256, 0, False, True, False),
    (300, 768, 512, 2, True, True, False),
    (1000, 100, 72, 1, False, False, False),
    (77, 40, 128, 3, True, False, False),
    (513, 2304, 768, 0, False, True, False),
    (200, 333, 64, 0, False, False, True),
    (384, 768, 3072, 0, True, False, False),
]


@pytest.mark.parametrize("M,N,K,act,use_resid,out_bf16,use_tmpl", TC_CASES)
def test_tcgen05_plain(a2f_lib, dev, M, N, K, act, use_resid, out_bf16, use_tmpl):
    from a2f_b200 import ops, lib as L
    a = _rand((M, K), dev, 11, torch.bfloat16)
    w = _rand((N, K), dev, 12, torch.bfloat16, scale=K ** -0.5)
    b = _rand((N,), dev, 13)
    r = _rand((M, N), dev, 14, torch.bfloat16) if use_resid else None
    t = _rand((7, N), dev, 15) if use_tmpl else None
    rpt = (M + 6) // 7
    out = torch.empty((M, N), device=dev, dtype=torch.bfloat16 if out_bf16 else torch.float32)
    ops.gemm(a, w, out, bias=b, act=act, resid=r, tmpl=t, rows_per_tmpl=rpt, backend=L.TCGEN05)
    torch.cuda.synchronize()
    want = _ref(a, w, b, act, r, t, rpt)
    err = float((out.cpu().double() - want).abs().max())
    tol = 3e-2 if out_bf16 else 2e-4
    assert err < tol, (err, tol)


@pytest.mark.parametrize("bn", [64, 128, 256])
def test_tcgen05_forced_tile_widths(a2f_lib, dev, bn):
    from a2f_b200 import ops, lib as L
    M, N, K = 390, 520, 192
    a = _rand((M, K), dev, 21, torch.bfloat16)
    w = _rand((N, K), dev, 22, torch.bfloat16, scale=K ** -0.5)
    out = torch.empty((M, N), device=dev)
    try:
        L.check(a2f_lib.a2f_debug_set_umma_field(4, bn))
        ops.gemm(a, w, out, backend=L.TCGEN05)
        torch.cuda.synchronize()
    finally:
        a2f_lib.a2f_debug_set_umma_field(4, 0)
    assert float((out.cpu().double() - _ref(a, w)).abs().max()) < 2e-4


@pytest.mark.parametrize("taps,L_in,B", [(3, 41, 2), (3, 40, 3), (2, 38, 2), (3, 515, 2)])
def test_conv1d_implicit_gemm(a2f_lib, dev, taps, L_in, B):
    """Conv1d(512->512, k taps, stride 2, no bias)+GELU over channels-last activations == F.conv1d on NCL."""
    from a2f_b200 import ops, lib as L
    C = 512
    L_out = (L_in - taps) // 2 + 1
    L_pad = L_in + (L_in % 2)         # batch stride kept a multiple of the row stride (see DESIGN.md)
    x = _rand((B, L_pad, C), dev, 31)
    x[:, L_in:] = 0
    w = _rand((C, C, taps), dev, 32, scale=(C * taps) ** -0.5)
    want = F.gelu(F.conv1d(x[:, :L_in].transpose(1, 2).double().cpu(), w.double().cpu(), stride=2)).transpose(1, 2)
    for backend, dt, tol in ((L.SIMT_F32, torch.float32, 2e-5), (L.TCGEN05, torch.bfloat16, 3e-2)):
        wp = torch.empty((C, taps * C), device=dev, dtype=dt)
        L.check(a2f_lib.a2f_pack_conv1d_weight(w.data_ptr(), wp.data_ptr(), 1 if dt == torch.bfloat16 else 0, C, C, taps,
                                                torch.cuda.current_stream().cuda_stream))
        xa = x.to(dt)
        out = torch.empty((B * L_out, C), device=dev, dtype=dt)
        ops.gemm(xa, wp, out, act=L.ACT_GELU, backend=backend, M=B * L_out, K=taps * C, a_row_stride=2 * C,
                 a_batch_stride=L_pad * C, rows_per_batch=L_out)
        torch.cuda.synchronize()
        ref = want if dt == torch.float32 else F.gelu(
            F.conv1d(xa[:, :L_in].transpose(1, 2).double().cpu(), wp.double().cpu().view(C, taps, C).permute(0, 2, 1),
                     stride=2)).transpose(1, 2)
        err = float((out.view(B, L_out, C).cpu().double() - ref).abs().max())
        assert err < tol, (backend, err)


@pytest.mark.parametrize("B,T", [(1, 60), (2, 150), (1, 300), (3, 129), (1, 777)])
def test_posconv(a2f_lib, dev, B, T):
    """h + gelu(weight-normed grouped conv k=128 pad 64 groups 16, last step dropped) vs torch."""
    from a2f_b200 import lib as L
    st = torch.cuda.current_stream().cuda_stream
    h = _rand((B, T, 768), dev, 41)
    g = (0.5 + torch.rand(1, 1, 128, generator=torch.Generator().manual_seed(42))).to(dev)
    v = _rand((768, 48, 128), dev, 43, scale=(48 * 128) ** -0.5)
    bias = _rand((768,), dev, 44, scale=0.05)
    wfull = torch._weight_norm(v.cpu(), g.cpu(), 2)
    norm = torch.empty(128, device=dev)
    # kpad 8 = chunked layout [16][128 taps][6][48 out][8 in] of posconv_tc.cu; kpad 64 = legacy gemm_tc mode 2 (debug field 9)
    for backend, dt, kpad, tol in ((L.SIMT_F32, torch.float32, 48, 3e-5), (L.TCGEN05, torch.bfloat16, 8, 5e-2),
                                   (L.TCGEN05, torch.bfloat16, 64, 5e-2)):
        a2f_lib.a2f_debug_set_umma_field(9, 1 if kpad == 64 else 0)
        wp = torch.empty((16, 128, 6, 48, 8) if kpad == 8 else (16, 48, 128, kpad), device=dev, dtype=dt)
        L.check(a2f_lib.a2f_pack_posconv_weight(g.data_ptr(), v.data_ptr(), wp.data_ptr(), 1 if dt == torch.bfloat16 else 0,
                                                 kpad, norm.data_ptr(), st))
        ha = h.to(dt).contiguous()
        out = torch.empty((B, T, 768), device=dev, dtype=dt)
        L.check(a2f_lib.a2f_posconv(ha.data_ptr(), 1 if dt == torch.bfloat16 else 0, wp.data_ptr(), bias.data_ptr(),
                                     out.data_ptr(), 1 if dt == torch.bfloat16 else 0, B, T, backend, st), "a2f_posconv")
        torch.cuda.synchronize()
        hh = ha.double().cpu()
        a2f_lib.a2f_debug_set_umma_field(9, 0)
        if kpad == 8:              # reference on the bf16-rounded packed weights: [g][tap][chunk][n][8] -> [g*48+n][c][tap]
            wq = wp.double().cpu().permute(0, 3, 2, 4, 1).reshape(768, 48, 128)
        elif dt == torch.bfloat16:
            wq = wp[..., :48].double().cpu().permute(0, 1, 3, 2).reshape(768, 48, 128)
        else:
            wq = wfull.double()
        pos = F.conv1d(hh.transpose(1, 2), wq, bias.double().cpu(), padding=64, groups=16)[:, :, :-1]
        want = hh + F.gelu(pos).transpose(1, 2)
        err = float((out.cpu().double() - want).abs().max())
        assert err < tol, (backend, err)


# Wide scalar epilogue of the 256-column fp32 tile (gemm_tc.cu, WIDE): 32 rows x 128 columns per epilogue warp, rolling
# template window that runs ahead into the CTA's next tile.  Cases: more tiles than SMs (the window crosses tiles), ragged
# last row tile (quarters with 28 and 0 live rows), ragged last column tile (221 / 89 live columns: partial and empty
# chunks), one template row per output row / shared by 150 rows (changes inside a tile) / none, with and without bias.
WIDE_CASES = [
    # M, N, K, rows_per_tmpl (0 = no template), use_bias
    (700, 15069, 192, 1, True),
    (700, 15069, 192, 150, True),
    (700, 15069, 64, 0, False),
    (1, 15069, 64, 1, True),
    (33, 601, 64, 1, False),
    (2500, 2137, 128, 7, True),
]


@pytest.mark.parametrize("M,N,K,rpt,use_bias", WIDE_CASES)
def test_tcgen05_wide_scalar_epilogue(a2f_lib, dev, M, N, K, rpt, use_bias):
    from a2f_b200 import ops, lib as L
    a = _rand((M, K), dev, 31, torch.bfloat16)
    w = _rand((N, K), dev, 32, torch.bfloat16, scale=K ** -0.5)
    b = _rand((N,), dev, 33) if use_bias else None
    t = _rand(((M + rpt - 1) // rpt, N), dev, 34) if rpt else None
    out = torch.full((M + 1, N), 7.0, device=dev)            # one guard row behind the output
    try:
        L.check(a2f_lib.a2f_debug_set_umma_field(4, 256))
        ops.gemm(a, w, out[:M], bias=b, tmpl=t, rows_per_tmpl=max(rpt, 1), backend=L.TCGEN05)
        torch.cuda.synchronize()
    finally:
        a2f_lib.a2f_debug_set_umma_field(4, 0)
    want = _ref(a, w, b, 0, None, t, max(rpt, 1))
    err = float((out[:M].cpu().double() - want).abs().max())
    assert err < 2e-4, err
    assert bool((out[M] == 7.0).all()), "the epilogue wrote past the last row"


@pytest.mark.parametrize("M,N,K", [(4800, 768, 768), (4800, 768, 3072), (300, 768, 768), (1, 768, 128), (1000, 512, 256),
                                   (129, 256, 64), (40000, 768, 192)])
def test_gemm_ln_fused_epilogue(a2f_lib, dev, M, N, K):
    """a2f_gemm_ln: LayerNorm(A W^T + bias + resid) in the GEMM epilogue (cluster of N/256 CTA pairs, row statistics over
    distributed shared memory) vs torch fp32 on the same bf16 operands.  Shapes: the two encoder GEMMs at the bench batch,
    a ragged last row block, a single row, 2- and 1-pair clusters, and more row blocks than resident clusters (persistent
    loop, parity double-buffering of the stats slots)."""
    from a2f_b200 import ops
    g = torch.Generator().manual_seed(M + N + K)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16()
    w = (torch.randn(N, K, generator=g) * (1.0 / K ** 0.5)).bfloat16()
    bias = 0.1 * torch.randn(N, generator=g)
    resid = torch.randn(M, N, generator=g).bfloat16()
    gamma, beta = torch.rand(N, generator=g) + 0.5, 0.1 * torch.randn(N, generator=g)
    want = torch.nn.functional.layer_norm(a.float() @ w.float().t() + bias + resid.float(), (N,), gamma, beta, 1e-5)
    out = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
    ops.gemm_ln(a.to(dev), w.to(dev), bias.to(dev), resid.to(dev), gamma.to(dev), beta.to(dev), out)
    torch.cuda.synchronize()
    err = (out.float().cpu() - want).abs()
    tol = 2.0 ** -8 * (want.abs() + 1.0)          # bf16 rounding of the output (2^-9 relative) + fp32 reduction-order noise
    assert bool((err <= tol).all()), (float(err.max()), int((err > tol).sum()))
    # run to run deterministic (no atomics on the path); the training variant also stores the pre-LayerNorm sum
    out2 = torch.empty_like(out)
    pre = torch.empty_like(out)
    ops.gemm_ln(a.to(dev), w.to(dev), bias.to(dev), resid.to(dev), gamma.to(dev), beta.to(dev), out2, pre_out=pre)
    assert torch.equal(out, out2)
    x = a.float() @ w.float().t() + bias + resid.float()
    assert bool(((pre.float().cpu() - x).abs() <= 2.0 ** -8 * (x.abs() + 1.0)).all())


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,F", [(4800, 768, 3072), (257, 768, 3072), (1, 768, 3072), (9000, 768, 3072), (12000, 768, 3072),
                                   (700, 512, 1024), (300, 256, 1024), (300, 256, 256)])
def test_ffn_one_kernel_equals_two(a2f_lib, dev, M, N, F):
    """a2f_encoder_block with only its feed-forward phases (no att, no wq: W1 + GELU + W2 + residual + LayerNorm in one
    kernel; the intermediate goes TMA store -> L2 -> TMA load between CTAs of a cluster, ordered by cluster-scope mbarriers)
    must give the SAME bits as a2f_gemm(GELU) followed by a2f_gemm_ln, and match torch fp32.  Shapes: the bench batch,
    ragged / single-row blocks, more row blocks than resident clusters (the per-round barriers wrap their parity), 2- and
    1-pair clusters, 1 to 4 phase-1 tiles per pair."""
    from a2f_b200 import ops, lib as L
    g = torch.Generator().manual_seed(M + N + F)
    x = torch.randn(M, N, generator=g).bfloat16().to(dev)
    w1 = (torch.randn(F, N, generator=g) * N ** -0.5).bfloat16().to(dev)
    w2 = (torch.randn(N, F, generator=g) * F ** -0.5).bfloat16().to(dev)
    b1, b2 = (0.1 * torch.randn(F, generator=g)).to(dev), (0.1 * torch.randn(N, generator=g)).to(dev)
    gamma, beta = (torch.rand(N, generator=g) + 0.5).to(dev), (0.1 * torch.randn(N, generator=g)).to(dev)
    f_ref = torch.empty((M, F), dtype=torch.bfloat16, device=dev)
    want = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
    ops.gemm(x, w1, f_ref, bias=b1, act=L.ACT_GELU, backend=L.TCGEN05)
    ops.gemm_ln(f_ref, w2, b2, x, gamma, beta, want)
    for rep in range(3):                                # repeated: a stale scratch from the previous run must not be read
        scratch = torch.full((M, F), float("nan"), dtype=torch.bfloat16, device=dev) if rep == 0 else scratch
        out = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
        ops.encoder_block(x, w1, b1, w2, b2, gamma, beta, scratch, out)
        torch.cuda.synchronize()
        assert torch.equal(scratch, f_ref), rep
        assert torch.equal(out, want), (rep, float((out.float() - want.float()).abs().max()))
        scratch.add_(1.0)                               # poison: the next run has to overwrite every element it reads
    xf = x.float()
    ref = torch.nn.functional.layer_norm(
        xf + torch.nn.functional.gelu(xf @ w1.float().t() + b1, approximate="tanh").bfloat16().float() @ w2.float().t() + b2,
        (N,), gamma, beta, 1e-5)
    err = (out.float() - ref).abs()
    tol = 2.0 ** -7 * (ref.abs() + 1.0)
    assert bool((err <= tol).all()), float(err.max())


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,F,NQ,p0,p3", [(4800, 768, 3072, 2304, True, True), (4800, 768, 3072, 2304, True, False),
                                            (4800, 768, 3072, 2304, False, True), (130, 768, 3072, 2304, True, True),
                                            (12000, 768, 3072, 2304, True, True), (9000, 768, 1536, 768, True, True),
                                            (700, 512, 1024, 1536, True, True), (300, 256, 1024, 512, True, True)])
def test_encoder_block_one_kernel_equals_four(a2f_lib, dev, M, N, F, NQ, p0, p3):
    """a2f_encoder_block (attention out-projection + LayerNorm, FFN, LayerNorm, next layer's q|k|v projection in one kernel,
    phase outputs handed over inside the cluster through L2) must give the SAME bits as the four separate launches.
    Shapes: the bench batch with and without the optional phases, a ragged block, more row blocks than resident clusters
    (every hand-over barrier wraps its parity), 2- and 1-pair clusters, fewer tiles per pair in phases 1 / 3."""
    from a2f_b200 import ops, lib as L
    g = torch.Generator().manual_seed(M + N + F + NQ)
    rnd = lambda *sh, s=1.0: (torch.randn(*sh, generator=g) * s)
    att, h_in = rnd(M, N).bfloat16().to(dev), rnd(M, N).bfloat16().to(dev)
    wo, w1 = rnd(N, N, s=N ** -0.5).bfloat16().to(dev), rnd(F, N, s=N ** -0.5).bfloat16().to(dev)
    w2, wq = rnd(N, F, s=F ** -0.5).bfloat16().to(dev), rnd(NQ, N, s=N ** -0.5).bfloat16().to(dev)
    bo, b1, b2, bq = (0.1 * rnd(N)).to(dev), (0.1 * rnd(F)).to(dev), (0.1 * rnd(N)).to(dev), (0.1 * rnd(NQ)).to(dev)
    g1, be1 = (torch.rand(N, generator=g) + 0.5).to(dev), (0.1 * rnd(N)).to(dev)
    g2, be2 = (torch.rand(N, generator=g) + 0.5).to(dev), (0.1 * rnd(N)).to(dev)
    bf = lambda *sh: torch.empty(sh, dtype=torch.bfloat16, device=dev)
    # reference: four launches
    h1_ref, f_ref, ho_ref, q_ref = bf(M, N), bf(M, F), bf(M, N), bf(M, NQ)
    if p0:
        ops.gemm_ln(att, wo, bo, h_in, g1, be1, h1_ref)
    else:
        h1_ref.copy_(h_in)
    ops.gemm(h1_ref, w1, f_ref, bias=b1, act=L.ACT_GELU, backend=L.TCGEN05)
    ops.gemm_ln(f_ref, w2, b2, h1_ref, g2, be2, ho_ref)
    ops.gemm(ho_ref, wq, q_ref, bias=bq, backend=L.TCGEN05)
    nan = float("nan")
    for rep in range(3):
        h1 = torch.full((M, N), nan, dtype=torch.bfloat16, device=dev) if p0 else h1_ref.clone()
        f, ho, q = torch.full((M, F), nan, dtype=torch.bfloat16, device=dev), bf(M, N), bf(M, NQ)
        kw = {}
        if p0:
            kw.update(att=att, wo=wo, bo=bo, h_in=h_in, ln1_g=g1, ln1_b=be1)
        if p3:
            kw.update(wq=wq, bq=bq, qkv=q)
        ops.encoder_block(h1, w1, b1, w2, b2, g2, be2, f, ho, **kw)
        torch.cuda.synchronize()
        assert torch.equal(h1, h1_ref), ("h1", rep)
        assert torch.equal(f, f_ref), ("f", rep)
        assert torch.equal(ho, ho_ref), ("h_out", rep, float((ho.float() - ho_ref.float()).abs().max()))
        if p3:
            assert torch.equal(q, q_ref), ("qkv", rep)


@pytest.mark.parametrize("M,N,K,act,use_resid", [(4800, 3072, 768, 2, False), (4800, 2304, 768, 0, False), (9600, 768, 256, 0, True),
                                                  (2400, 3072, 128, 0, False), (40000, 512, 192, 2, False)])
def test_tcgen05_pair_kernel_tail_split(a2f_lib, dev, M, N, K, act, use_resid):
    """Wave quantisation of the CTA-pair kernel: tiles of a partly filled last wave are cut into 2 or 4 column slices
    (FFN1: 228 tiles on 74 pairs, QKV: 171).  The sliced schedule must give the SAME bits as the unsliced one (same MMA
    order per output element) and match the fp64 reference."""
    from a2f_b200 import ops, lib as L
    a = _rand((M, K), dev, 31, torch.bfloat16)
    w = _rand((N, K), dev, 32, torch.bfloat16, scale=K ** -0.5)
    b = _rand((N,), dev, 33)
    r = _rand((M, N), dev, 34, torch.bfloat16) if use_resid else None
    outs = []
    for split in (1, 0):
        out = torch.empty((M, N), device=dev, dtype=torch.bfloat16)
        try:
            L.check(a2f_lib.a2f_debug_set_umma_field(11, split))
            ops.gemm(a, w, out, bias=b, act=act, resid=r, backend=L.TCGEN05)
            torch.cuda.synchronize()
        finally:
            a2f_lib.a2f_debug_set_umma_field(11, 1)
        outs.append(out)
    assert torch.equal(outs[0], outs[1])
    want = _ref(a, w, b, act, r)
    assert bool(((outs[0].cpu().double() - want).abs() <= 2.0 ** -8 * (want.abs() + 1.0)).all())


@pytest.mark.parametrize("M,N,K,batches", [(2400, 3072, 768, 1), (4800, 3072, 768, 1), (300, 512, 256, 1), (1998, 512, 1536, 2)])
def test_tcgen05_pair_kernel_two_outputs(a2f_lib, dev, M, N, K, batches):
    """a2f_gemm_args::C2: one launch writes the pre-activation z = A W^T + b (kept for the activation backward) AND gelu(z)
    (the operand of the next GEMM).  Must equal the two-launch sequence GEMM + a2f_act_fwd bit for bit."""
    from a2f_b200 import ops, lib as L
    a = _rand((M, K), dev, 41, torch.bfloat16)
    w = _rand((N, K), dev, 42, torch.bfloat16, scale=K ** -0.5)
    b = _rand((N,), dev, 43)
    rpb = M // batches
    kw = dict(M=M, rows_per_batch=rpb, a_batch_stride=rpb * K, c_batch_stride=rpb * N)
    z1 = torch.empty((M, N), device=dev, dtype=torch.bfloat16)
    ops.gemm(a, w, z1, bias=b, backend=L.TCGEN05, **kw)
    y1 = ops.act_fwd(z1, L.ACT_GELU)
    z2, y2 = torch.empty_like(z1), torch.empty_like(z1)
    ops.gemm(a, w, z2, bias=b, act=L.ACT_GELU, out2=y2, backend=L.TCGEN05, **kw)
    torch.cuda.synchronize()
    assert torch.equal(z1, z2)
    # act_fwd applies GELU to the bf16-ROUNDED z, the fused epilogue to the fp32 z: the two bf16 results can sit two ulps apart
    err = (y1.float() - y2.float()).abs()
    assert bool((err <= 2.0 ** -6 * (y1.float().abs() + 0.05)).all()), float(err.max())
    want = _ref(a, w, b, 2)
    # vs fp64 erf-GELU: bf16 rounding of the output + the tanh-form GELU of the bf16 path (|tanh form - erf form| <= 4.7e-4)
    assert bool(((y2.cpu().double() - want).abs() <= 2.0 ** -7 * want.abs() + 2e-3).all())
