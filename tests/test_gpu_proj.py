"""GPU parity of the concat + dense projection variants (tcgen05 path) against the CPU oracle and against the
reference's own golden outputs.

Bars: the projection kernels alone (bf16 operands, fp32 accumulation in tensor memory, one rounding of the result)
are held to the bf16 bar, normalised max-abs <= 2^-8, against an fp32 matmul of the same bf16 operands.  The whole
variant chains three bf16 roundings exactly where the reference does ([tok|bytes] operand, F.linear output, norm
output -- runs/7:317-319,233-234 run in bf16), so against the fp32-math oracle the stated bar is 2^-6 on outputs and
dense gradients."""
import os

import numpy as np
import pytest
import torch

from oracle import mot_oracle as O

pytestmark = pytest.mark.gpu

TOL_KERNEL = 2.0 ** -8
TOL_CHAIN = 2.0 ** -6
TOL_TF32_CHAIN = 2.0 ** -8   # fp32 tables, TF32 products (10 mantissa bits) through projection + norm, fwd and bwd


def dev():
    return torch.device("cuda:0")


def nerr(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("n,K,Do", [(1, 64, 8), (37, 160, 40), (128, 64, 256), (300, 1024, 1024), (777, 1920, 1000),
                                    (4096, 2048, 1024),
                                    (40000, 512, 1024)])   # 1252 output tiles: several tiles per persistent CTA
def test_linear_kernels_match_fp32_matmul(n, K, Do):
    from mot_b200 import ops
    d = dev()
    g = torch.Generator(device=d).manual_seed(n * 7 + K)
    x = torch.randn(n, K, generator=g, device=d).bfloat16()
    w = (torch.randn(Do, K, generator=g, device=d) / K ** 0.5).bfloat16()
    dy = torch.randn(n, Do, generator=g, device=d).bfloat16()
    bias = torch.randn(Do, generator=g, device=d)
    y = torch.empty(n, Do, dtype=torch.bfloat16, device=d)
    ops.linear_forward_out(x, w, y)
    assert nerr(y, x.float() @ w.float().t()) <= TOL_KERNEL
    y32 = torch.empty(n, Do, dtype=torch.float32, device=d)
    ops.linear_forward_out(x, w, y32, bias)
    assert nerr(y32, x.float() @ w.float().t() + bias) <= 1e-5
    dx = torch.empty(n, K, dtype=torch.bfloat16, device=d)
    ops.linear_bwd_input_out(dy, w, dx)
    assert nerr(dx, dy.float() @ w.float()) <= TOL_KERNEL
    dw32 = torch.empty(Do, K, dtype=torch.float32, device=d)
    dw16 = torch.empty(Do, K, dtype=torch.bfloat16, device=d)
    ops.linear_bwd_weight_out(dy, x, dw32, dw16)
    ref = dy.float().t() @ x.float()
    assert nerr(dw32, ref) <= 1e-4      # fp32 split-K reduction order differs from torch's
    assert nerr(dw16, ref) <= TOL_KERNEL


def test_linear_refuses_fp16_operands_and_misaligned_dims():
    from mot_b200 import ops, _lib as L
    d = dev()
    x = torch.randn(8, 64, device=d).half()
    with pytest.raises(NotImplementedError):
        ops.linear_forward_out(x, x, torch.empty(8, 8, device=d))
    xb = torch.randn(8, 60, device=d).bfloat16()
    with pytest.raises(RuntimeError):
        ops.linear_forward_out(xb, xb, torch.empty(8, 8, dtype=torch.bfloat16, device=d))
    assert L.lib().mot_linear_fwd(None, None, None, None, 0, 64, 64, L.BF16, 0, None) == L.OK   # empty batch


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("n,D", [(5, 40), (300, 768), (1000, 1024)])
def test_rmsnorm_rows(n, D, dtype):
    from mot_b200 import ops
    d = dev()
    g = torch.Generator(device=d).manual_seed(n + D)
    y = torch.randn(n, D, generator=g, device=d).to(dtype)
    go = torch.randn(n, D, generator=g, device=d).to(dtype)
    out, dy = torch.empty_like(y), torch.empty_like(y)
    ops.rmsnorm_forward_out(y, out)
    ops.rmsnorm_backward_out(y, go, dy)
    yr = y.detach().float().cpu().requires_grad_(True)
    ref = O.rms_norm(yr)
    ref.backward(go.float().cpu())
    tol = 1e-5 if dtype == torch.float32 else TOL_KERNEL
    assert nerr(out, ref) <= tol and nerr(dy, yr.grad) <= tol


CASES = {
    # name: (oracle variant, MixSpec kwargs, (V, Vb, bpt, Dt, bd, Do), slot_major)
    "V1_runs7": ("V1", dict(combine="concat", tok_norm=True, byte_norm=True, out_norm=True), (300, 458, 16, 64, 16, 128), False),
    "V1_spt_256_48": ("V1", dict(combine="concat", tok_norm=True, byte_norm=True, out_norm=True), (500, 458, 16, 256, 48, 1024), False),
    "V2_runs72": ("V2", dict(combine="concat", out_norm=True, slot_major=True), (300, 458, 16, 128, 8, 256), True),
    "V2_tok896": ("V2", dict(combine="concat", out_norm=True, slot_major=True), (200, 458, 16, 896, 64, 1024), True),
}


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("N,w_fp32", [(37, False), (700, True)])
def test_projection_variants_vs_oracle(name, N, w_fp32):
    import mot_b200
    variant, kw, (V, Vb, bpt, Dt, bd, Do), slot_major = CASES[name]
    K = Dt + bpt * bd
    g = torch.Generator().manual_seed(N + K)
    toks = torch.randint(0, V, (N,), generator=g, dtype=torch.int32)
    ids = torch.randint(0, Vb, (N, bpt), generator=g, dtype=torch.int32)
    ids_given = ids.t().contiguous() if slot_major else ids.reshape(1, -1)
    E_tok = torch.randn(V, Dt, generator=g).bfloat16()
    E_byte = torch.randn(Vb, bd, generator=g).bfloat16()
    W = (torch.rand(Do, K, generator=g) * 2 - 1) * (3 ** 0.5) * 0.5 * K ** -0.5   # CastedLinear init
    W = W if w_fp32 else W.bfloat16()
    gout = torch.randn(N, Do, generator=g).bfloat16()
    # the kernels see the weight rounded to bf16 (W.type_as(x), spt/train_gpt.py:186): so does the oracle
    want_out, want = O.mot_embed_fwd_bwd(O.VARIANTS[variant][0], toks, ids_given, E_tok, E_byte, gout, bpt=bpt,
                                         slot_major=slot_major, W=W.bfloat16())
    d = dev()
    Et, Eb = E_tok.to(d).requires_grad_(True), E_byte.to(d).requires_grad_(True)
    Wd = W.to(d).requires_grad_(True)
    out = mot_b200.mot_embed_proj(toks.to(d), ids_given.to(d), Et, Eb, Wd, mot_b200.MixSpec(**kw), bpt=bpt)
    out.backward(gout.to(d))
    torch.cuda.synchronize()
    assert out.dtype == torch.bfloat16 and tuple(out.shape) == (N, Do)
    assert Wd.grad.dtype == W.dtype
    errs = {"out": nerr(out, want_out), "gE_tok": nerr(Et.grad, want["E_tok"]), "gE_byte": nerr(Eb.grad, want["E_byte"]),
            "gW": nerr(Wd.grad, want["W"])}
    assert all(e <= TOL_CHAIN for e in errs.values()), errs
    untouched = torch.ones(V, dtype=torch.bool)
    untouched[toks.long()] = False
    assert float(Et.grad[untouched.to(d)].abs().max()) == 0.0


def test_reference_golden_projection_through_cuda(golden_dir):
    """The reference's own bf16 runs of mixin_bytes (runs/7, runs/72) and of FlexibleEmbedding + ByteMixinConcat
    (scaled-pre-train), generated by tests/golden/make_golden.py, reproduced by the CUDA path."""
    import mot_b200
    d = dev()
    g = np.load(os.path.join(golden_dir, "runs_float_bf16.npz"))
    for tag, variant in [("V1_run7_bf16", "V1"), ("V2_run72_bf16", "V2")]:
        m = mot_b200.MoTProjEmbedding(80, 458, 32, 8, 40, 16, variant=variant).to(d)
        with torch.no_grad():
            m.embed_tokens.weight.copy_(torch.from_numpy(g[f"{tag}_E_tok"]))
            m.embed_bytes.weight.copy_(torch.from_numpy(g[f"{tag}_E_byte"]))
            m.byte_mixin_weight.copy_(torch.from_numpy(g[f"{tag}_W"]))
        m = m.bfloat16()
        out = m(torch.from_numpy(g[f"{tag}_tokens"]).to(d), torch.from_numpy(g[f"{tag}_byte_inputs"]).to(d))
        out.backward(torch.from_numpy(g[f"{tag}_gout"]).to(d).bfloat16().reshape(out.shape))
        assert nerr(out, torch.from_numpy(g[f"{tag}_out"]).reshape(out.shape)) <= TOL_CHAIN
        assert nerr(m.embed_tokens.weight.grad, torch.from_numpy(g[f"{tag}_gE_tok"])) <= TOL_CHAIN
        assert nerr(m.embed_bytes.weight.grad, torch.from_numpy(g[f"{tag}_gE_byte"])) <= TOL_CHAIN
        assert nerr(m.byte_mixin_weight.grad, torch.from_numpy(g[f"{tag}_gW"])) <= TOL_CHAIN
    s = np.load(os.path.join(golden_dir, "spt_float.npz"))
    tag = "concat_bf16"
    Dt, bd = s[f"{tag}_E_tok"].shape[1], s[f"{tag}_E_byte"].shape[1]
    Do, K = s[f"{tag}_W"].shape
    bpt = (K - Dt) // bd
    m = mot_b200.SptByteMixEmbedding(s[f"{tag}_E_tok"].shape[0], 458, Dt, bd, Do, bpt, pull_in=True).to(d)
    with torch.no_grad():
        m.embed.embed_tokens.weight.copy_(torch.from_numpy(s[f"{tag}_E_tok"]))
        m.embed.embed_bytes.weight.copy_(torch.from_numpy(s[f"{tag}_E_byte"]))
        m.byte_mixin.mixin.mixin.weight.copy_(torch.from_numpy(s[f"{tag}_W"]))
    m.embed.bfloat16()     # tables bf16, projection weight stays an fp32 master (spt/train_gpt.py:1124-1126)
    out = m(torch.from_numpy(s[f"{tag}_tokens"]).to(d), torch.from_numpy(s[f"{tag}_bytes_padded"]).to(d),
            torch.from_numpy(s[f"{tag}_bytes_pulled"]).to(d))
    out.backward(torch.from_numpy(s[f"{tag}_gout"]).to(d).bfloat16())
    assert m.byte_mixin.mixin.mixin.weight.grad.dtype == torch.float32
    assert nerr(out, torch.from_numpy(s[f"{tag}_out"])) <= TOL_CHAIN
    assert nerr(m.embed.embed_tokens.weight.grad, torch.from_numpy(s[f"{tag}_gE_tok"])) <= TOL_CHAIN
    assert nerr(m.embed.embed_bytes.weight.grad, torch.from_numpy(s[f"{tag}_gE_byte"])) <= TOL_CHAIN
    assert nerr(m.byte_mixin.mixin.mixin.weight.grad, torch.from_numpy(s[f"{tag}_gW"])) <= TOL_CHAIN


@pytest.mark.parametrize("dtype,bpt,bd,N", [
    (torch.float32, 16, 48, 301), (torch.float32, 18, 56, 77), (torch.float32, 20, 64, 130), (torch.float32, 4, 8, 33),
    (torch.float32, 32, 32, 65), (torch.bfloat16, 8, 128, 40),
    (torch.bfloat16, 16, 48, 4097), (torch.bfloat16, 18, 32, 513), (torch.bfloat16, 16, 64, 1),
])
def test_byte_pair_kernels_match_oracle(dtype, bpt, bd, N):
    """mot_byte_pair_fwd / _bwd (spt/train_gpt.py:371-379: norm(embed_bytes(padded) + embed_bytes(pulled))) written into
    / read from the byte columns of wider rows, against the oracle's byte_ids2 path; int64 ids like spt."""
    from mot_b200 import ops
    d = dev()
    g = torch.Generator().manual_seed(bpt * 100 + bd)
    Vb, Dt = 458, 64
    K = Dt + bpt * bd
    ia = torch.randint(0, Vb, (N, bpt), generator=g)
    ib = torch.randint(0, Vb, (N, bpt), generator=g)
    ib[::3] = ia[::3]                      # equal ids in both tensors (pad/pad): both REDs hit the same row
    E = torch.randn(Vb, bd, generator=g).to(dtype)
    gout = torch.randn(N, bpt * bd, generator=g).to(dtype)
    spec = O.MixSpec(combine="bytes_only", byte_norm=True, out_norm=False)
    want_out, want = O.mot_embed_fwd_bwd(spec, torch.zeros(N, dtype=torch.int64), ia, None, E, gout, bpt=bpt, byte_ids2=ib)
    A = torch.full((N, K), 7.0, dtype=dtype, device=d)
    ops.byte_pair_forward_out(ia.to(d), ib.to(d), bpt, E.to(d), A, Dt)
    tol = 1e-5 if dtype == torch.float32 else TOL_KERNEL
    assert nerr(A[:, Dt:], want_out) <= tol
    assert float((A[:, :Dt] - 7.0).abs().max()) == 0.0            # the token columns are not touched
    dA = torch.zeros(N, K, dtype=dtype, device=d)
    dA[:, Dt:] = gout.to(d)
    gE = torch.full((Vb, bd), float("nan"), dtype=dtype, device=d)
    ops.byte_pair_backward_out(ia.to(d), ib.to(d), bpt, E.to(d), dA, Dt, gE)
    assert nerr(gE, want["E_byte"]) <= tol, f"{nerr(gE, want['E_byte']):.3e}"
    ops.byte_pair_backward_out(ia.to(d).int(), ib.to(d).int(), bpt, E.to(d), dA, Dt, gE)   # int32 ids, fresh workspace
    assert nerr(gE, want["E_byte"]) <= tol


def test_spt_add_padded_and_pulled_matches_reference_golden_and_oracle(golden_dir):
    """`--add-padded-and-pulled` (spt/train_gpt.py:371-379,949-951) end to end through SptByteMixEmbedding: the
    reference's own fp32 output / gradients (TF32 tensor cores here), then bf16 at the spt default dims vs the oracle."""
    import mot_b200
    d = dev()
    s = np.load(os.path.join(golden_dir, "spt_float.npz"))
    tag = "concat_addpp_f32"
    Dt, bd = s[f"{tag}_E_tok"].shape[1], s[f"{tag}_E_byte"].shape[1]
    Do, K = s[f"{tag}_W"].shape
    bpt = (K - Dt) // bd
    m = mot_b200.SptByteMixEmbedding(s[f"{tag}_E_tok"].shape[0], 458, Dt, bd, Do, bpt, pull_in=True,
                                     add_padded_and_pulled=True).to(d)
    with torch.no_grad():
        m.embed.embed_tokens.weight.copy_(torch.from_numpy(s[f"{tag}_E_tok"]))
        m.embed.embed_bytes.weight.copy_(torch.from_numpy(s[f"{tag}_E_byte"]))
        m.byte_mixin.mixin.mixin.weight.copy_(torch.from_numpy(s[f"{tag}_W"]))
    out = m(torch.from_numpy(s[f"{tag}_tokens"]).to(d), torch.from_numpy(s[f"{tag}_bytes_padded"]).to(d),
            torch.from_numpy(s[f"{tag}_bytes_pulled"]).to(d))
    out.backward(torch.from_numpy(s[f"{tag}_gout"]).to(d))
    assert nerr(out, torch.from_numpy(s[f"{tag}_out"])) <= TOL_TF32_CHAIN
    assert nerr(m.embed.embed_tokens.weight.grad, torch.from_numpy(s[f"{tag}_gE_tok"])) <= TOL_TF32_CHAIN
    assert nerr(m.embed.embed_bytes.weight.grad, torch.from_numpy(s[f"{tag}_gE_byte"])) <= TOL_TF32_CHAIN
    assert nerr(m.byte_mixin.mixin.mixin.weight.grad, torch.from_numpy(s[f"{tag}_gW"])) <= TOL_TF32_CHAIN

    g = torch.Generator().manual_seed(17)
    V, Vb, Dt, bd, Do, bpt, B, S = 700, 458, 256, 48, 1024, 16, 2, 300
    m = mot_b200.SptByteMixEmbedding(V, Vb, Dt, bd, Do, bpt, pull_in=True, add_padded_and_pulled=True).to(d)
    m.embed.bfloat16()
    toks = torch.randint(0, V, (B, S), generator=g, dtype=torch.int32)
    pad = torch.randint(0, Vb, (B, S * bpt), generator=g)
    pul = torch.randint(0, Vb, (B, S * bpt), generator=g)
    gout = torch.randn(B, S, Do, generator=g).bfloat16()
    out = m(toks.to(d), pad.to(d), pul.to(d))
    out.backward(gout.to(d))
    Et, Eb, W = (t.detach().cpu() for t in (m.embed.embed_tokens.weight, m.embed.embed_bytes.weight, m.byte_mixin.mixin.mixin.weight))
    want_out, want = O.mot_embed_fwd_bwd(O.VARIANTS["V1"][0], toks, pad, Et, Eb, gout, bpt=bpt, W=W.bfloat16(), byte_ids2=pul)
    assert nerr(out.view(-1, Do), want_out) <= TOL_CHAIN
    assert nerr(m.embed.embed_tokens.weight.grad, want["E_tok"]) <= TOL_CHAIN
    assert nerr(m.embed.embed_bytes.weight.grad, want["E_byte"]) <= TOL_CHAIN
    assert nerr(m.byte_mixin.mixin.mixin.weight.grad, want["W"]) <= TOL_CHAIN


def test_byte_fc_variant_matches_reference_golden_and_oracle(golden_dir):
    """V3f (runs/71051:226-229,312-314): norm(tok + F.linear(cat(bytes), byte_fc)) through MoTByteFcEmbedding: the
    reference's own bf16 / fp32 outputs and gradients at toy size, then the shipped 1024 = 16 x 64 shape vs the oracle."""
    import mot_b200
    d = dev()
    for tag, dtype, tol in (("V3f_run71051_bf16", torch.bfloat16, TOL_CHAIN), ("V3f_run71051_f32", torch.float32, TOL_TF32_CHAIN)):
        g = np.load(os.path.join(golden_dir, f"runs_float_{tag.rsplit('_', 1)[1]}.npz"))
        V, Dm = g[f"{tag}_E_tok"].shape
        bd = g[f"{tag}_E_byte"].shape[1]
        m = mot_b200.MoTByteFcEmbedding(V, 458, Dm, bd, Dm // bd).to(d)
        assert sorted(n for n, _ in m.named_parameters()) == ["byte_fc", "embed_bytes.weight", "embed_tokens.weight"]
        m = m.to(dtype)
        with torch.no_grad():
            m.embed_tokens.weight.copy_(torch.from_numpy(g[f"{tag}_E_tok"]))
            m.embed_bytes.weight.copy_(torch.from_numpy(g[f"{tag}_E_byte"]))
            m.byte_fc.copy_(torch.from_numpy(g[f"{tag}_W"]))
        out = m(torch.from_numpy(g[f"{tag}_tokens"]).to(d), torch.from_numpy(g[f"{tag}_byte_inputs"]).to(d))
        out.backward(torch.from_numpy(g[f"{tag}_gout"]).to(d).to(dtype).reshape(out.shape))
        assert nerr(out, torch.from_numpy(g[f"{tag}_out"]).reshape(out.shape)) <= tol
        assert nerr(m.embed_tokens.weight.grad, torch.from_numpy(g[f"{tag}_gE_tok"])) <= tol
        assert nerr(m.embed_bytes.weight.grad, torch.from_numpy(g[f"{tag}_gE_byte"])) <= tol
        assert nerr(m.byte_fc.grad, torch.from_numpy(g[f"{tag}_gW"])) <= tol

    gen = torch.Generator().manual_seed(23)
    V, Vb, bpt, bd, N = 3000, 458, 16, 64, 2500
    Dm = bpt * bd
    m = mot_b200.MoTByteFcEmbedding(V, Vb, Dm, bd, bpt).to(d).bfloat16()
    toks = (torch.rand(N, generator=gen) ** 3 * V).long().clamp_(0, V - 1).int()      # hot rows straddle stream chunks
    ids = torch.randint(0, Vb, (bpt, N), generator=gen, dtype=torch.int32)
    gout = torch.randn(1, N, Dm, generator=gen).bfloat16()
    out = m(toks.to(d), ids.to(d))
    out.backward(gout.to(d))
    Et, Eb, W = (t.detach().cpu() for t in (m.embed_tokens.weight, m.embed_bytes.weight, m.byte_fc))
    want_out, want = O.mot_embed_fwd_bwd(O.VARIANTS["V3f"][0], toks, ids, Et, Eb, gout, bpt=bpt, slot_major=True, W=W)
    assert nerr(out[0], want_out) <= TOL_CHAIN
    assert nerr(m.embed_tokens.weight.grad, want["E_tok"]) <= TOL_CHAIN
    assert nerr(m.embed_bytes.weight.grad, want["E_byte"]) <= TOL_CHAIN
    assert nerr(m.byte_fc.grad, want["W"]) <= TOL_CHAIN


def test_spt_module_refuses_unsupported_options():
    import mot_b200
    for kw in (dict(byte_mixin_method="cross_attn"), dict(use_byte_self_attn=True)):
        with pytest.raises(NotImplementedError):
            mot_b200.SptByteMixEmbedding(100, 458, 64, 16, 128, 16, **kw)


# ------------------------------------------------------------------ fp32 operands on the TF32 tensor-core path (V8)
TOL_TF32 = 2.0 ** -9   # tf32 keeps 10 mantissa bits; mathblations itself runs F.linear in TF32 (main.py:522)


@pytest.mark.parametrize("n,K,Do", [(33, 64, 32), (128, 1280, 256), (11264, 1280, 256), (1000, 328, 72)])
def test_linear_kernels_tf32_match_fp32_matmul(n, K, Do):
    from mot_b200 import ops
    d = dev()
    g = torch.Generator(device=d).manual_seed(n + K)
    x = torch.randn(n, K, generator=g, device=d)
    w = torch.randn(Do, K, generator=g, device=d) / K ** 0.5
    dy = torch.randn(n, Do, generator=g, device=d)
    bias = torch.randn(Do, generator=g, device=d)
    y = torch.empty(n, Do, device=d)
    ops.linear_forward_out(x, w, y, bias)
    assert nerr(y, x.double() @ w.double().t() + bias.double()) <= TOL_TF32
    dx = torch.empty(n, K, device=d)
    ops.linear_bwd_input_out(dy, w, dx)
    assert nerr(dx, dy.double() @ w.double()) <= TOL_TF32
    dw = torch.empty(Do, K, device=d)
    ops.linear_bwd_weight_out(dy, x, dw)
    assert nerr(dw, dy.double().t() @ x.double()) <= TOL_TF32
    with pytest.raises(NotImplementedError):   # mixed operand dtypes are refused, not converted behind the caller's back
        ops.linear_forward_out(x, w.bfloat16(), y)


def test_mathblations_digit_mixin_matches_reference_golden(golden_dir):
    """DigitMixinConcat (mathblations/model.py:256-268,323-327) on the reference's own inputs / outputs, and the digit
    expansion of GenerateEquations.tokens_to_digits bit-exact."""
    import mot_b200
    g = np.load(os.path.join(golden_dir, "mathblations.npz"))
    d = dev()
    dpt, op, eq, pad, _ = (int(v) for v in g["digits_meta"])
    got = mot_b200.tokens_to_digits(torch.from_numpy(g["digits_tokens"]).to(d), dpt, op, eq, pad)
    assert np.array_equal(got.cpu().numpy(), g["digits_out"])
    toks = torch.tensor([0, 7, 10, 99, 105, 9999, op, eq, pad], dtype=torch.int32, device=d)
    want = O.tokens_to_digits(toks.cpu().tolist(), 4, op, eq, pad)
    assert np.array_equal(mot_b200.tokens_to_digits(toks, 4, op, eq, pad, out_dtype=torch.int32).cpu().numpy(), want)

    V, Dt = g["mix_wte"].shape
    Dd = g["mix_dte"].shape[1]
    dpt_m = g["mix_digits"].shape[1] // g["mix_idx"].shape[1]
    m = mot_b200.DigitMixinEmbedding(V, Dt, Dd, dpt_m).to(d)
    with torch.no_grad():
        m.wte.weight.copy_(torch.from_numpy(g["mix_wte"]))
        m.dte.weight.copy_(torch.from_numpy(g["mix_dte"]))
        m.digit_mixin.fc.weight.copy_(torch.from_numpy(g["mix_fc_w"]))
        m.digit_mixin.fc.bias.copy_(torch.from_numpy(g["mix_fc_b"]))
    assert sorted(m.state_dict()) == ["digit_mixin.fc.bias", "digit_mixin.fc.weight", "dte.weight", "wte.weight"]
    out = m(torch.from_numpy(g["mix_idx"]).to(d), torch.from_numpy(g["mix_digits"]).to(d))
    out.backward(torch.from_numpy(g["mix_gout"]).to(d))
    assert out.dtype == torch.float32
    assert nerr(out, torch.from_numpy(g["mix_out"])) <= TOL_TF32
    assert nerr(m.wte.weight.grad, torch.from_numpy(g["mix_gwte"])) <= TOL_TF32
    assert nerr(m.dte.weight.grad, torch.from_numpy(g["mix_gdte"])) <= TOL_TF32
    assert nerr(m.digit_mixin.fc.weight.grad, torch.from_numpy(g["mix_gfc_w"])) <= TOL_TF32
    assert nerr(m.digit_mixin.fc.bias.grad, torch.from_numpy(g["mix_gfc_b"])) <= 1e-5


def test_mathblations_config2_vs_oracle():
    """BASELINE config 2: B=1024, S=11, dpt 4, vocab 10003, 256/256 -> K = 1280, fp32 (SURVEY 8d cfg 2)."""
    import mot_b200
    d = dev()
    g = torch.Generator().manual_seed(2)
    B, S, dpt, V, Dt, Dd = 1024, 11, 4, 10003, 256, 256
    idx = torch.randint(0, 10000, (B, S), generator=g)
    idx[torch.rand(B, S, generator=g) < 0.2] = 10000          # operator tokens
    digits = torch.from_numpy(O.tokens_to_digits(idx.reshape(-1).tolist(), dpt, 10000, 10001, 10002)).view(B, S * dpt)
    m = mot_b200.DigitMixinEmbedding(V, Dt, Dd, dpt)
    gout = torch.randn(B * S, Dt, generator=g)
    spec = O.VARIANTS["V8"][0]
    want_out, want = O.mot_embed_fwd_bwd(spec, idx.reshape(-1).int(), digits.reshape(1, -1), m.wte.weight.detach(), m.dte.weight.detach(),
                                         gout, bpt=dpt, W=m.digit_mixin.fc.weight.detach(), bias=m.digit_mixin.fc.bias.detach())
    m = m.to(d)
    out = m(idx.to(d), digits.to(d))
    out.backward(gout.to(d).view_as(out))
    assert nerr(out.view(B * S, Dt), want_out) <= TOL_TF32
    assert nerr(m.wte.weight.grad, want["E_tok"]) <= TOL_TF32
    assert nerr(m.dte.weight.grad, want["E_byte"]) <= TOL_TF32
    assert nerr(m.digit_mixin.fc.weight.grad, want["W"]) <= TOL_TF32
    assert nerr(m.digit_mixin.fc.bias.grad, want["bias"]) <= 1e-4
