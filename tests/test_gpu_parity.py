"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle.

Bars (SURVEY.md 8c): integer outputs bit-exact; fp32 tables: normalised max-abs
error <= 1e-5 against the fp32 oracle; bf16 tables: against the fp32-math oracle
evaluated on the same bf16 parameters, outputs and dense grads within one bf16
ulp of the largest element (normalised max-abs <= 2^-8 = 3.9e-3)."""
import os

import numpy as np
import pytest
import torch

from oracle import mot_oracle as O

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-5, torch.bfloat16: 2.0 ** -8}


def dev():
    return torch.device("cuda:0")


def nerr(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def golden_table(golden_dir):
    tab = np.load(os.path.join(golden_dir, "ttb_8_left_pad.npz"))["table"]
    full = np.full((50257, 8), O.PAD_BYTE, dtype=np.int16)
    full[:50256] = tab
    full[50256] = O.EOT_BYTE
    return full


# ------------------------------------------------------------------ integer half
@pytest.mark.parametrize("bpt", [8, 16, 4])
@pytest.mark.parametrize("container", ["i16", "f32", "bf16"])
def test_ttb_expand_bit_exact(golden_dir, bpt, container):
    import mot_b200
    tab = O.ttb_repad(golden_table(golden_dir), bpt, "left")
    g = torch.Generator().manual_seed(7)
    toks = torch.randint(0, 50257, (4, 257), generator=g, dtype=torch.int32)
    toks[0, :3] = torch.tensor([50256, 0, 50255])
    if container == "i16":
        t = torch.from_numpy(tab).to(dev())
        want_tab = tab
    elif container == "f32":
        t = torch.from_numpy(tab.astype(np.float32)).to(dev())
        want_tab = tab
    else:  # the runs' bf16 table quirk (runs/7:441)
        t = torch.from_numpy(tab.astype(np.float32)).to(dev()).bfloat16()
        want_tab = O.bf16_round_ids(tab)
    want = O.tokens_to_bytes(toks.numpy(), want_tab)
    got = mot_b200.ttb_expand(toks.to(dev()), t)
    assert got.dtype == torch.int64 and tuple(got.shape) == want.shape
    assert np.array_equal(got.cpu().numpy(), want)
    got32 = mot_b200.ttb_expand(toks.to(dev())[0], t, out_dtype=torch.int32)  # 1-D tokens -> [1, T*bpt]
    assert got32.dtype == torch.int32 and tuple(got32.shape) == (1, 257 * bpt)
    assert np.array_equal(got32.cpu().numpy(), O.tokens_to_bytes(toks.numpy()[0], want_tab))


def test_ttb_expand_matches_reference_golden(golden_dir):
    import mot_b200
    g = np.load(os.path.join(golden_dir, "integer_path.npz"))
    t = torch.from_numpy(golden_table(golden_dir)).to(dev())
    for case in "abcd":
        toks = torch.from_numpy(g[f"{case}_tokens"]).to(dev())
        assert np.array_equal(mot_b200.ttb_expand(toks, t).cpu().numpy(), g[f"{case}_bytes_left"])
    q = torch.from_numpy(golden_table(golden_dir).astype(np.float32)).to(dev()).bfloat16()
    assert np.array_equal(mot_b200.ttb_expand(torch.from_numpy(g["e_tokens"]).to(dev()), q).cpu().numpy(),
                          g["e_bytes_left_bf16quirk"])


def test_ttb_expand_empty_and_errors(golden_dir):
    import mot_b200
    t = torch.from_numpy(golden_table(golden_dir)).to(dev())
    out = mot_b200.ttb_expand(torch.zeros((2, 0), dtype=torch.int32, device=dev()), t)
    assert tuple(out.shape) == (2, 0)
    with pytest.raises(RuntimeError):
        mot_b200.ttb_expand(torch.zeros(4, dtype=torch.int32), t)  # CPU tensor: no fallback
    with pytest.raises(NotImplementedError):
        mot_b200.ttb_expand(torch.zeros(4, dtype=torch.int32, device=dev()), t.double())


# ------------------------------------------------------------------ float half
CASES = {
    # name: (oracle variant, mot spec kwargs, dims (V, Vb, bpt, Dt, bd), slot_major, lambdas)
    "V0_tok_only": ("V0", dict(combine="tok_only"), (300, 458, 16, 256, 16), False, False),
    "V3_sum_scramble": ("V3", dict(combine="add", slot_major=True), (500, 458, 16, 768, 48), True, False),
    "V3_sum_bpt8x128": ("V3", dict(combine="add", slot_major=True), (300, 458, 8, 1024, 128), True, False),
    "V3_sum_bpt32x32": ("V3", dict(combine="add", slot_major=True), (300, 458, 32, 1024, 32), True, False),
    "V3b": ("V3b", dict(combine="add", tok_norm=True, byte_norm=True, out_norm=False, slot_major=True), (400, 458, 16, 1024, 64), True, False),
    "V3c_lambdas": ("V3c", dict(combine="add", tok_norm=True, byte_norm=True, out_norm=False, slot_major=True), (400, 458, 16, 512, 32), True, True),
    "V3d_lambdas": ("V3d", dict(combine="add", tok_norm=True, byte_norm=True, out_norm=True, slot_major=True), (400, 458, 16, 1024, 64), True, True),
    "V4_concat": ("V4", dict(combine="concat"), (300, 458, 16, 512, 32), False, False),
    "V5_bytes_only": ("V5", dict(combine="bytes_only"), (1, 458, 16, 0, 64), False, False),
    "V7_mean": ("V7", dict(combine="mean", out_norm=False), (200, 132, 8, 256, 256), False, True),
    "V1_A_operand": (None, dict(combine="concat", tok_norm=True, byte_norm=True, out_norm=False), (300, 458, 16, 256, 48), False, False),
    "V8_A_operand": (None, dict(combine="concat", out_norm=False, bytes_first=True), (1003, 14, 4, 256, 256), False, False),
}


def run_case(name, dtype, N, seed=0, ids_dtype=torch.int32, zipf=False):
    import mot_b200
    variant, kw, (V, Vb, bpt, Dt, bd), slot_major, use_lam = CASES[name]
    spec_o = O.VARIANTS[variant][0] if variant else O.MixSpec(
        combine=kw["combine"], tok_norm=kw.get("tok_norm", False), byte_norm=kw.get("byte_norm", False),
        out_norm=kw.get("out_norm", True), bytes_first=kw.get("bytes_first", False))
    g = torch.Generator().manual_seed(seed)
    if zipf:  # heavy duplicates -> hot rows split over several work items
        toks = (torch.rand(N, generator=g) ** 4 * V).long().clamp_(0, V - 1).int()
    else:
        toks = torch.randint(0, V, (N,), generator=g, dtype=torch.int32)
    ids = torch.randint(0, Vb, (N, bpt), generator=g).to(ids_dtype)
    ids_given = ids.t().contiguous() if slot_major else ids   # [bpt, N] like runs/71:479
    E_tok = torch.randn(V, max(Dt, 8), generator=g).to(dtype) if Dt else None
    E_byte = torch.randn(Vb, bd, generator=g).to(dtype) if kw["combine"] != "tok_only" else None
    lam = torch.tensor([0.7, 0.4]) if use_lam else None
    Do = {"add": Dt, "tok_only": Dt, "mean": Dt, "concat": Dt + bpt * bd, "bytes_only": bpt * bd}[kw["combine"]]
    gout = torch.randn(N, Do, generator=g).to(dtype)

    okw = dict(bpt=bpt, slot_major=slot_major)
    if use_lam:
        okw["lam_tok"], okw["lam_byte"] = lam[0], lam[1]
    want_out, want = O.mot_embed_fwd_bwd(spec_o, toks, ids_given if E_byte is not None else None, E_tok, E_byte, gout, **okw)

    d = dev()
    Et = E_tok.to(d).requires_grad_(True) if E_tok is not None else None
    Eb = E_byte.to(d).requires_grad_(True) if E_byte is not None else None
    lam_d = lam.to(d).requires_grad_(True) if use_lam else None
    spec = mot_b200.MixSpec(**kw)
    out = mot_b200.mot_embed(toks.to(d) if E_tok is not None else None, ids_given.to(d) if E_byte is not None else None,
                             Et, Eb, spec, bpt=bpt, lam=lam_d)
    out.backward(gout.to(d))
    torch.cuda.synchronize()
    tol = TOL[dtype]
    assert out.dtype == dtype and tuple(out.shape) == (N, Do)
    assert nerr(out, want_out) <= tol, f"out {nerr(out, want_out):.3e}"
    if Et is not None:
        assert nerr(Et.grad, want["E_tok"]) <= tol, f"gE_tok {nerr(Et.grad, want['E_tok']):.3e}"
        # rows never gathered are exactly zero (dense-grad contract)
        untouched = torch.ones(V, dtype=torch.bool)
        untouched[toks.long()] = False
        assert float(Et.grad[untouched.to(d)].abs().max() if untouched.any() else 0.0) == 0.0
    if Eb is not None:
        assert nerr(Eb.grad, want["E_byte"]) <= tol, f"gE_byte {nerr(Eb.grad, want['E_byte']):.3e}"
    if use_lam:
        got = lam_d.grad.cpu().double()
        ref = torch.stack([want["lam_tok"], want["lam_byte"]]).double()
        # scalar sums of N*D products: fp32 accumulation order differs from torch's
        assert float((got - ref).abs().max() / ref.abs().max()) <= (1e-4 if dtype == torch.float32 else tol)


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_variants_small(name, dtype):
    run_case(name, dtype, N=37)


@pytest.mark.parametrize("name", ["V3_sum_scramble", "V3d_lambdas", "V4_concat", "V1_A_operand", "V7_mean"])
def test_variants_hot_rows_and_int64_ids(name):
    """~3000 positions over a few hundred rows with a skewed distribution: rows with more than L
    occurrences take the partial-sum + finalize path; ids as int64 like scaled-pre-train."""
    run_case(name, torch.bfloat16, N=3001, seed=3, ids_dtype=torch.int64, zipf=True)
    run_case(name, torch.float32, N=1500, seed=4, ids_dtype=torch.int64, zipf=True)


def test_ids_from_ttb_token_major_and_scramble(golden_dir):
    """forward(token_ids) -> embeddings: byte ids derived from the ttb table inside the kernel,
    token-major and with the `.view(bpt,-1)` index map of runs/71:479."""
    import mot_b200
    tab = O.ttb_repad(golden_table(golden_dir), 16, "left")
    d = dev()
    g = torch.Generator().manual_seed(11)
    N, V, Dt, bd, bpt = 512, 50257, 768, 48, 16
    toks = torch.randint(0, V, (N,), generator=g, dtype=torch.int32)
    E_tok = torch.randn(V, Dt, generator=g).bfloat16()
    E_byte = torch.randn(458, bd, generator=g).bfloat16()
    gout = torch.randn(N, Dt, generator=g).bfloat16()
    flat = O.tokens_to_bytes(toks.numpy(), tab)  # [1, N*bpt] token-major
    for scramble in (False, True):
        ids_o = torch.from_numpy(O.scramble_view(flat, bpt).copy() if scramble else flat.copy())
        want_out, want = O.mot_embed_fwd_bwd(O.VARIANTS["V3"][0], toks, ids_o, E_tok, E_byte, gout, bpt=bpt, slot_major=scramble)
        for ttb_t in (torch.from_numpy(tab).to(d), torch.from_numpy(tab.astype(np.float32)).to(d)):
            Et, Eb = E_tok.to(d).requires_grad_(True), E_byte.to(d).requires_grad_(True)
            spec = mot_b200.MixSpec(combine="add", ttb_scramble=scramble)
            out = mot_b200.mot_embed(toks.to(d), None, Et, Eb, spec, bpt=bpt, ttb=ttb_t, seq_len=N)
            out.backward(gout.to(d))
            assert nerr(out, want_out) <= TOL[torch.bfloat16]
            assert nerr(Et.grad, want["E_tok"]) <= TOL[torch.bfloat16]
            assert nerr(Eb.grad, want["E_byte"]) <= TOL[torch.bfloat16]


def test_reference_golden_runs_through_cuda(golden_dir):
    """The reference's own outputs (tests/golden/runs_float_f32.npz, fp32 runs) reproduced by the CUDA path."""
    import mot_b200
    g = np.load(os.path.join(golden_dir, "runs_float_f32.npz"))
    d = dev()
    for tag, kw, slot_major in [
        ("V3_run71", dict(combine="add"), True),
        ("V3b_run73", dict(combine="add", tok_norm=True, byte_norm=True, out_norm=False), True),
        ("V4_run711", dict(combine="concat"), False),
    ]:
        k = f"{tag}_f32"
        Et = torch.from_numpy(g[f"{k}_E_tok"]).to(d).requires_grad_(True)
        Eb = torch.from_numpy(g[f"{k}_E_byte"]).to(d).requires_grad_(True)
        spec = mot_b200.MixSpec(slot_major=slot_major, **kw)
        out = mot_b200.mot_embed(torch.from_numpy(g[f"{k}_tokens"]).to(d), torch.from_numpy(g[f"{k}_byte_inputs"]).to(d),
                                 Et, Eb, spec, bpt=16)
        out.backward(torch.from_numpy(g[f"{k}_gout"]).to(d).reshape(out.shape))
        assert nerr(out, torch.from_numpy(g[f"{k}_out"]).reshape(out.shape)) <= 1e-5
        assert nerr(Et.grad, torch.from_numpy(g[f"{k}_gE_tok"])) <= 1e-5
        assert nerr(Eb.grad, torch.from_numpy(g[f"{k}_gE_byte"])) <= 1e-5


def test_full_size_properties():
    """BASELINE size (N = 49152, V = 50257, 768 = 16 x 48, bf16): size-independent properties.
    (1) out rows have unit rms (out_norm); (2) sum of the dense token grad over rows equals the sum over
    positions of d z (linearity of the scatter-add), checked through a plain torch reduction of the
    oracle formula on the GPU in fp32; (3) untouched rows are exactly zero; (4) byte-grad total matches."""
    import mot_b200
    d = dev()
    g = torch.Generator(device="cuda").manual_seed(5)
    N, V, Dt, bd, bpt = 49152, 50257, 768, 48, 16
    toks = torch.randint(0, V, (N,), generator=g, device=d, dtype=torch.int32)
    ids = torch.randint(0, 458, (bpt, N), generator=g, device=d, dtype=torch.int32)
    Et = (torch.randn(V, Dt, generator=g, device=d)).bfloat16().requires_grad_(True)
    Eb = (torch.randn(458, bd, generator=g, device=d)).bfloat16().requires_grad_(True)
    gout = torch.randn(N, Dt, generator=g, device=d).bfloat16()
    out = mot_b200.mot_embed(toks, ids, Et, Eb, mot_b200.MixSpec(combine="add", slot_major=True), bpt=bpt)
    out.backward(gout)
    rms = out.float().pow(2).mean(-1).sqrt()
    assert float((rms - 1).abs().max()) < 1e-2
    # fp32 restatement on the GPU (torch ops, test-only) of d z
    z = Et.detach().float()[toks.long()] + Eb.detach().float()[ids.long().t()].reshape(N, -1)
    r = torch.rsqrt(z.pow(2).mean(-1, keepdim=True) + mot_b200.FP32_EPS)
    gf = gout.float()
    dz = r * gf - z * (r ** 3) * (gf * z).mean(-1, keepdim=True)
    col_sum = dz.sum(0)
    got = Et.grad.float().sum(0)
    assert float((got - col_sum).abs().max() / col_sum.abs().max()) < 2e-2  # 50k bf16-rounded rows summed
    untouched = torch.ones(V, dtype=torch.bool, device=d)
    untouched[toks.long()] = False
    assert float(Et.grad[untouched].abs().max()) == 0.0
    want_b = torch.zeros(458, bd, device=d).index_add_(0, ids.long().t().reshape(-1), dz.reshape(N * bpt, bd))
    assert nerr(Eb.grad, want_b) <= 2.0 ** -8


@pytest.mark.parametrize("dtype,Dt,bd,bpt,N,V,zipf", [
    (torch.float32, 512, 64, 8, 333, 200, False),
    (torch.float32, 768, 48, 16, 5000, 1500, True),       # hot rows straddle stream chunks -> slot + finalize path
    (torch.float32, 1024, 32, 32, 2049, 50257, False),    # mostly single-occurrence rows, many empty rows
    (torch.bfloat16, 768, 48, 16, 70001, 20000, True),    # R = 64: two batches per stream chunk, ragged tail
    (torch.bfloat16, 1024, 64, 16, 4097, 1100, False),
    (torch.bfloat16, 512, 64, 8, 1, 10, False),
])
def test_saved_output_backward_vs_recompute_and_oracle(dtype, Dt, bd, bpt, N, V, zipf):
    """mot_embed_bwd_ex (reads grad_out + the kept forward result, mot_embed_bwd_sum.cuh) against mot_embed_bwd
    (rebuilds the mixed row) and against the oracle, through the C ABI on caller-allocated tensors."""
    import mot_b200
    from mot_b200 import ops
    d = dev()
    g = torch.Generator().manual_seed(11)
    toks = ((torch.rand(N, generator=g) ** 4 * V).long().clamp_(0, V - 1).int() if zipf
            else torch.randint(0, V, (N,), generator=g, dtype=torch.int32))
    ids = torch.randint(0, 458, (bpt, N), generator=g, dtype=torch.int32)       # slot-major like runs/71:479
    E_tok = torch.randn(V, Dt, generator=g).to(dtype)
    E_byte = torch.randn(458, bd, generator=g).to(dtype)
    gout = torch.randn(N, Dt, generator=g).to(dtype)
    want_out, want = O.mot_embed_fwd_bwd(O.VARIANTS["V3"][0], toks, ids, E_tok, E_byte, gout, bpt=bpt, slot_major=True)
    spec = mot_b200.MixSpec(combine="add", slot_major=True)
    tk, idd, Et, Eb, go = toks.to(d), ids.to(d), E_tok.to(d), E_byte.to(d), gout.to(d)
    desc = ops.make_desc(spec, N, Et, Eb, bpt, ids=idd, ttb=None, has_lam=False)
    assert ops.embed_bwd_uses_saved(desc)                   # these shapes take the saved-output kernel
    big = ops.make_desc(spec, 8 * V, Et, Eb, bpt, ids=idd, ttb=None, has_lam=False)
    assert not ops.embed_bwd_uses_saved(big)                # > 4 positions per vocabulary row: recompute kernel
    out = torch.empty(N, Dt, dtype=dtype, device=d)
    rstd = torch.full((N,), float("nan"), dtype=torch.float32, device=d)
    ops.embed_forward_out(desc, tk, idd, None, Et, Eb, None, out, rstd=rstd)
    z = E_tok.double()[toks.long()] + E_byte.double()[ids.long().t()].reshape(N, -1)
    want_rstd = torch.rsqrt(z.pow(2).mean(-1) + mot_b200.FP32_EPS)
    assert nerr(rstd, want_rstd) <= 1e-5
    ws = torch.empty(ops.embed_workspace_bytes(desc), dtype=torch.uint8, device=d)
    res = {}
    for name, kw in (("saved", dict(out_saved=out, rstd=rstd)), ("recompute", {})):
        for rep in range(2):   # twice on the same workspace: the first call leaves it clean for the second
            # dense gradients inside guard rows: a write outside [0, V) x [0, Dt) would clear a NaN sentinel
            gt_buf = torch.full((V + 2, Dt), float("nan"), dtype=dtype, device=d)
            gb_buf = torch.full((458 + 2, bd), float("nan"), dtype=dtype, device=d)
            gt, gb = gt_buf[1:-1], gb_buf[1:-1]
            ops.embed_backward_out(desc, tk, idd, None, Et, Eb, None, go, gt, gb, None, ws, plan_ready=False,
                                   ws_clean=(rep == 1 or name == "recompute"), **kw)
            torch.cuda.synchronize()
            for buf in (gt_buf, gb_buf):
                assert bool(torch.isnan(buf[0]).all()) and bool(torch.isnan(buf[-1]).all()), f"{name}: write outside the table"
                assert not bool(torch.isnan(buf[1:-1]).any()), f"{name}: a row was not written"
        res[name] = (gt, gb)
    tol = TOL[dtype]
    assert nerr(out, want_out) <= tol
    for name, (gt, gb) in res.items():
        assert nerr(gt, want["E_tok"]) <= tol, f"{name} gE_tok {nerr(gt, want['E_tok']):.3e}"
        assert nerr(gb, want["E_byte"]) <= tol, f"{name} gE_byte {nerr(gb, want['E_byte']):.3e}"
    untouched = torch.ones(V, dtype=torch.bool)
    untouched[toks.long()] = False
    if untouched.any():
        assert float(res["saved"][0][untouched.to(d)].abs().max()) == 0.0


@pytest.mark.parametrize("variant", ["V3d", "V3b", "V3c", "V4", "V1A", "V3_256k", "V3_zipf", "V3d_zipf"])
def test_full_size_static_flag_kernels_vs_torch_restatement(variant):
    """The compile-time-flag backward kernels at the shipped sizes (65536 tokens, V = 50257, 1024 columns, bf16), where
    the CPU oracle is too slow: the same formulas restated with torch fp32 ops on the GPU (test-only) through autograd."""
    import mot_b200
    import torch.nn.functional as F
    d = dev()
    g = torch.Generator(device="cuda").manual_seed(9)
    N, V, bpt = 65536, 50257, 16
    Dt, bd = (512, 32) if variant in ("V4", "V1A") else (1024, 64)
    if variant == "V3_256k":      # more than 4 positions per vocabulary row: the recompute kernel, stream chunks of 5 batches
        N, Dt, bd = 262144, 768, 48
    toks = torch.randint(0, V, (N,), generator=g, device=d, dtype=torch.int32)
    if variant.endswith("_zipf"):   # hot rows spread over hundreds of stream chunks: fp32 slot + finalize path at scale
        toks = (torch.rand(N, generator=g, device=d) ** 6 * V).long().clamp_(0, V - 1).int()
        variant = variant[:-5]
    slot_major = variant not in ("V4", "V1A")
    ids = torch.randint(0, 458, (bpt, N) if slot_major else (1, N * bpt), generator=g, device=d, dtype=torch.int32)
    Et = torch.randn(V, Dt, generator=g, device=d).bfloat16().requires_grad_(True)
    Eb = torch.randn(458, bd, generator=g, device=d).bfloat16().requires_grad_(True)
    lam = torch.tensor([0.7, 0.4], device=d, requires_grad=True) if variant in ("V3d", "V3c") else None
    Do = Dt + bpt * bd if variant in ("V4", "V1A") else Dt
    gout = torch.randn(N, Do, generator=g, device=d).bfloat16()
    # V1A: the [norm(tok) | norm(bytes)] operand of the projection variants (runs/7:317-318), split into a tok-only and a
    # bytes-only launch
    spec = mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True, out_norm=False) if variant == "V1A" \
        else mot_b200.MixSpec(**mot_b200.RUN_VARIANTS["V3" if variant == "V3_256k" else variant])
    out = mot_b200.mot_embed(toks, ids, Et, Eb, spec, bpt=bpt, lam=lam)
    out.backward(gout)
    # restatement (runs/71041:311-313, runs/73:313-315, runs/711:314-316)
    Etf, Ebf = Et.detach().float().requires_grad_(True), Eb.detach().float().requires_grad_(True)
    lamf = lam.detach().clone().requires_grad_(True) if lam is not None else None
    nrm = lambda x: F.rms_norm(x, (x.size(-1),), eps=mot_b200.FP32_EPS)  # noqa: E731
    t = Etf[toks.long()]
    idm = ids.long().t() if slot_major else ids.long().view(N, bpt)
    b = Ebf[idm]                                   # [N, bpt, bd]
    if variant == "V4":
        ref = nrm(torch.cat([t, b.reshape(N, -1)], dim=-1))
    elif variant == "V1A":
        ref = torch.cat([nrm(t), nrm(b).reshape(N, -1)], dim=-1)
    else:
        tn, bn = nrm(t), nrm(b).reshape(N, -1)
        if variant == "V3d":
            ref = nrm(tn * lamf[0] + bn * lamf[1])
        elif variant == "V3c":
            ref = tn * lamf[0] + bn * lamf[1]
        elif variant in ("V3_256k", "V3"):
            ref = nrm(t + b.reshape(N, -1))
        else:
            ref = tn + bn
    ref.backward(gout.float())
    assert nerr(out, ref) <= 2.0 ** -8
    assert nerr(Et.grad, Etf.grad) <= 2.0 ** -8, f"gE_tok {nerr(Et.grad, Etf.grad):.3e}"
    assert nerr(Eb.grad, Ebf.grad) <= 2.0 ** -8, f"gE_byte {nerr(Eb.grad, Ebf.grad):.3e}"
    if lam is not None:
        assert float((lam.grad - lamf.grad).abs().max() / lamf.grad.abs().max()) <= 2.0 ** -8


def test_unsupported_and_bad_arguments():
    import mot_b200
    d = dev()
    Et = torch.randn(10, 64, device=d).bfloat16()
    Eb = torch.randn(458, 4, device=d).bfloat16()
    toks = torch.zeros(4, dtype=torch.int32, device=d)
    ids = torch.zeros(4, 16, dtype=torch.int32, device=d)
    with pytest.raises(RuntimeError):  # byte_dim not a multiple of 8
        mot_b200.mot_embed(toks, ids, Et, Eb, mot_b200.MixSpec(combine="add"), bpt=16)
    with pytest.raises(NotImplementedError):
        mot_b200.mot_embed(toks, ids, Et.half(), Eb.half(), mot_b200.MixSpec(combine="add"), bpt=16)
    with pytest.raises(RuntimeError):
        mot_b200.mot_embed(toks.cpu(), ids.cpu(), Et.cpu(), Eb.cpu(), mot_b200.MixSpec(combine="add"), bpt=16)
    # empty batch
    Eb8 = torch.randn(458, 8, device=d).bfloat16()
    Et128 = torch.randn(10, 128, device=d).bfloat16().requires_grad_(True)
    out = mot_b200.mot_embed(toks[:0], ids[:0], Et128, Eb8, mot_b200.MixSpec(combine="add"), bpt=16)
    assert tuple(out.shape) == (0, 128)


def test_module_backward_writes_into_grad_bucket():
    """Data-parallel path: with a GradBucket attached the backward kernels write the dense gradients straight into
    the flat bucket (param.grad is a view of it) and the values equal the un-bucketed run."""
    import mot_b200
    d = dev()
    torch.manual_seed(3)
    m = mot_b200.MoTEmbedding(1000, 458, 256, 16, 16, variant="V3").to(d).bfloat16()
    toks = torch.randint(0, 1000, (300,), device=d, dtype=torch.int32)
    ids = torch.randint(0, 458, (16, 300), device=d, dtype=torch.int32)
    gout = torch.randn(1, 300, 256, device=d).bfloat16()
    m(toks, ids).backward(gout)
    want_tok, want_byte = m.embed_tokens.weight.grad.clone(), m.embed_bytes.weight.grad.clone()
    for p in m.parameters():
        p.grad = None
    bucket = m.attach_grad_bucket()
    m(toks, ids).backward(gout)
    assert m.embed_tokens.weight.grad.data_ptr() == bucket.flat.data_ptr()
    assert m.embed_bytes.weight.grad.data_ptr() == bucket.view_of(m.embed_bytes.weight).data_ptr()
    # fp32 summation order of duplicates / atomics differs run to run: same bar as against the oracle
    assert nerr(m.embed_tokens.weight.grad, want_tok) <= 2.0 ** -8
    assert nerr(m.embed_bytes.weight.grad, want_byte) <= 2.0 ** -8
    assert bucket.all_reduce_avg() is None   # single process: no collective
