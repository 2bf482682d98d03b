"""Pin the CPU oracle against the reference's golden vectors (tests/golden/,
generated from the reference itself by tests/golden/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import mot_oracle as O


def load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


# ------------------------------------------------------------------ integer half
def test_byte_to_int_is_bijection(golden_dir):
    b2i = json.load(open(os.path.join(golden_dir, "byte_to_int.json")))
    assert len(b2i) == O.BYTE_VOCAB
    assert sorted(b2i.values()) == list(range(458))
    assert b2i["pad"] == O.PAD_BYTE and b2i["endoftext"] == O.EOT_BYTE


def test_create_ttb_reproduces_checked_in_table(golden_dir):
    """Strings reconstructed from the table, pushed through the restated
    create_ttb, give the table back bit-exactly (SURVEY 8c annex)."""
    tab = load(golden_dir, "ttb_8_left_pad.npz")["table"]
    assert tab.shape == (50256, 8) and tab.min() >= 0 and tab.max() == 456
    pads = (tab == 456).sum(1)
    hist = np.bincount(pads, minlength=8).tolist()
    assert hist == [15956, 5913, 6410, 7294, 7162, 4983, 1850, 688]
    b2i = json.load(open(os.path.join(golden_dir, "byte_to_int.json")))
    i2b = {v: k for k, v in b2i.items()}
    strings = ["".join(i2b[int(c)] for c in row[row != 456]) for row in tab]
    ttb = O.create_ttb(lambda i: strings[i], b2i, 50256, bpt=8, pad_position="left")
    again = O.ttb_dict_to_array(ttb, 50257, 8)
    assert np.array_equal(again[:50256], tab)
    assert np.all(again[50256] == O.EOT_BYTE)
    # right padding / shorter bpt follow create_ttb.py:24-28
    right = O.create_ttb(lambda i: strings[i], b2i, 50256, bpt=8, pad_position="right")
    r = O.ttb_dict_to_array(right, 50257, 8)
    assert np.array_equal(O.ttb_repad(again, 8, "right"), r)
    t4 = O.ttb_dict_to_array(O.create_ttb(lambda i: strings[i], b2i, 50256, bpt=4), 50257, 4)
    assert np.array_equal(O.ttb_repad(again, 4, "left"), t4)
    t16 = O.ttb_dict_to_array(O.create_ttb(lambda i: strings[i], b2i, 50256, bpt=16), 50257, 16)
    assert np.array_equal(O.ttb_repad(again, 16, "left"), t16)
    with pytest.raises(ValueError):
        O.create_ttb(lambda i: "a", b2i, 1, bpt=4, pad_position="middle")
    eot = O.create_ttb(lambda i: "<|endoftext|>", b2i, 1, bpt=4)
    assert eot[0] == [457] * 4


def _table(golden_dir):
    tab = load(golden_dir, "ttb_8_left_pad.npz")["table"]
    full = np.full((50257, 8), O.PAD_BYTE, dtype=np.int16)
    full[:50256] = tab
    full[50256] = O.EOT_BYTE
    return full


@pytest.mark.parametrize("case", ["a", "b", "c", "d"])
def test_tokens_to_bytes_and_pull_match_reference(golden_dir, case):
    g = load(golden_dir, "integer_path.npz")
    tab = _table(golden_dir)
    toks = g[f"{case}_tokens"]
    left = O.tokens_to_bytes(toks, tab)
    assert left.dtype == np.int64
    assert np.array_equal(left, g[f"{case}_bytes_left"])
    assert np.array_equal(O.pull_from_left(left, 8), g[f"{case}_pull_from_left"])
    right = O.tokens_to_bytes(toks, O.ttb_repad(tab, 8, "right"))
    assert np.array_equal(right, g[f"{case}_bytes_right"])
    assert np.array_equal(O.pull_from_right(right, 8), g[f"{case}_pull_from_right"])


def test_tokens_to_bytes_1d_and_bf16_quirk(golden_dir):
    g = load(golden_dir, "integer_path.npz")
    tab = _table(golden_dir)
    out = O.tokens_to_bytes(g["e_tokens"], tab)
    assert out.shape == (1, 40 * 8)
    assert np.array_equal(out, g["e_bytes_left"])
    quirk = O.bf16_round_ids(tab)
    assert np.array_equal(O.tokens_to_bytes(g["e_tokens"], quirk), g["e_bytes_left_bf16quirk"])
    m = O.bf16_round_ids(np.arange(458))
    assert np.array_equal(m, g["bf16_id_map"])
    assert (m != np.arange(458)).sum() == 101 and m[457] == 456 and m[455] == 456 and m[257] == 256


def test_pull_edge_cases():
    empty = np.zeros((2, 0), dtype=np.int64)
    assert O.pull_from_left(empty, 4).shape == (2, 0)
    # all-pad token contributes nothing and receives the pool
    x = np.array([[456, 456, 7, 8, 456, 456, 456, 456, 457, 457, 457, 457, 456, 456, 456, 9]])
    assert O.pull_from_left(x, 4).tolist() == [[456, 456, 7, 8, 456, 456, 7, 8, 457, 457, 457, 457, 456, 456, 456, 9]]
    y = np.array([[7, 8, 456, 456, 9, 456, 456, 456, 457, 457, 457, 457, 1, 2, 3, 4]])
    assert O.pull_from_right(y, 4).tolist() == [[7, 8, 9, 456, 9, 456, 456, 456, 457, 457, 457, 457, 1, 2, 3, 4]]
    with pytest.raises(AssertionError):
        O.pull_from_left(np.zeros((1, 5), dtype=np.int64), 4)


def test_scramble_view_formula():
    flat = np.arange(32).reshape(1, 32)
    v = O.scramble_view(flat, 4)
    assert v.shape == (4, 8)
    for i in range(4):
        for s in range(8):
            assert v[i, s] == i * 8 + s


def test_tokens_to_digits(golden_dir):
    g = load(golden_dir, "mathblations.npz")
    dpt, op, eq, pad, vocab = g["digits_meta"].tolist()
    out = O.tokens_to_digits(g["digits_tokens"], dpt, op, eq, pad)
    assert np.array_equal(out, g["digits_out"])
    assert O.tokens_to_digits([4245], 4, 10000, 10001, 10002).tolist() == [4, 2, 4, 5]
    assert O.tokens_to_digits([10000], 4, 10000, 10001, 10002).tolist() == [13, 13, 13, 10]


# ------------------------------------------------------------------ float half
def T(a):
    return torch.from_numpy(np.asarray(a))


def close(a, b, tol):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = max(np.abs(b).max(), 1e-30)
    err = np.abs(a - b).max() / scale
    assert err <= tol, f"normalised max-abs err {err:.3e} > {tol:.1e}"


RUN_CASES = {
    # tag: (variant, slot_major, weight key)
    "V1_run7": ("V1", False, "W"),
    "V2_run72": ("V2", True, "W"),
    "V3_run71": ("V3", True, None),
    "V3b_run73": ("V3b", True, None),
    "V3c_run74": ("V3c", True, None),
    "V3d_run71041": ("V3d", True, None),
    "V3f_run71051": ("V3f", True, "W"),
    "V4_run711": ("V4", False, None),
}


@pytest.mark.parametrize("tag", sorted(RUN_CASES))
@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_runs_variants_match_reference(golden_dir, tag, dt):
    """fp32: oracle == reference to fp32 round-off.  bf16: the reference rounds
    every intermediate to bf16 (eager), the oracle does fp32 math on the same
    bf16 parameters -> agreement to a few bf16 ulps of the largest element."""
    g = load(golden_dir, f"runs_float_{dt}.npz")
    variant, slot_major, wkey = RUN_CASES[tag]
    spec, _ = O.VARIANTS[variant]
    k = f"{tag}_{dt}"
    kw = dict(bpt=16, slot_major=slot_major)
    if wkey:
        kw["W"] = T(g[f"{k}_W"])
    if f"{k}_scalars" in g.files:
        sc = T(g[f"{k}_scalars"])
        kw["lam_tok"], kw["lam_byte"] = sc[-1], sc[-2]
    out, grads = O.mot_embed_fwd_bwd(spec, T(g[f"{k}_tokens"]), T(g[f"{k}_byte_inputs"]),
                                     T(g[f"{k}_E_tok"]), T(g[f"{k}_E_byte"]), T(g[f"{k}_gout"]), **kw)
    tol = 2e-6 if dt == "f32" else 3e-2
    close(out, g[f"{k}_out"].reshape(out.shape), tol)
    close(grads["E_tok"], g[f"{k}_gE_tok"], tol)
    close(grads["E_byte"], g[f"{k}_gE_byte"], tol)
    if wkey:
        close(grads["W"], g[f"{k}_gW"], tol)
    if f"{k}_scalars" in g.files:
        gs = g[f"{k}_gscalars"]
        # the eager-bf16 reference sums N*D bf16-rounded products for these two scalars
        close(torch.stack([grads["lam_byte"], grads["lam_tok"]]), gs[-2:], tol if dt == "f32" else 8e-2)


@pytest.mark.parametrize("tag", ["concat_f32", "concat_bf16", "concat_padded_f32", "concat_addpp_f32", "noop_f32"])
def test_spt_modules_match_reference(golden_dir, tag):
    g = load(golden_dir, "spt_float.npz")
    toks = T(g[f"{tag}_tokens"])
    kw = dict(bpt=4, slot_major=False)
    if tag.startswith("noop"):
        spec, _ = O.VARIANTS["V0"]
        ids = None
        E_byte = None
    else:
        spec, _ = O.VARIANTS["V1"]
        E_byte = T(g[f"{tag}_E_byte"])
        kw["W"] = T(g[f"{tag}_W"])
        if "padded" in tag:      # pull_in=False -> _forward_bytes_padded (train_gpt.py:350-358)
            ids = T(g[f"{tag}_bytes_padded"])
        elif "addpp" in tag:     # train_gpt.py:371-379
            ids = T(g[f"{tag}_bytes_padded"])
            kw["byte_ids2"] = T(g[f"{tag}_bytes_pulled"])
        else:                    # train_gpt.py:361-369
            ids = T(g[f"{tag}_bytes_pulled"])
    out, grads = O.mot_embed_fwd_bwd(spec, toks, ids, T(g[f"{tag}_E_tok"]), E_byte, T(g[f"{tag}_gout"]), **kw)
    tol = 3e-2 if "bf16" in tag else 2e-6
    close(out, g[f"{tag}_out"].reshape(out.shape), tol)
    close(grads["E_tok"], g[f"{tag}_gE_tok"], tol)
    if not tag.startswith("noop"):
        close(grads["E_byte"], g[f"{tag}_gE_byte"], tol)
        close(grads["W"], g[f"{tag}_gW"], tol)


def test_mathblations_digit_mixin_matches_reference(golden_dir):
    g = load(golden_dir, "mathblations.npz")
    spec, _ = O.VARIANTS["V8"]
    out, grads = O.mot_embed_fwd_bwd(spec, T(g["mix_idx"]), T(g["mix_digits"]), T(g["mix_wte"]), T(g["mix_dte"]),
                                     T(g["mix_gout"]), bpt=2, slot_major=False,
                                     W=T(g["mix_fc_w"]), bias=T(g["mix_fc_b"]))
    close(out, g["mix_out"].reshape(out.shape), 2e-6)
    close(grads["E_tok"], g["mix_gwte"], 2e-6)
    close(grads["E_byte"], g["mix_gdte"], 2e-6)
    close(grads["W"], g["mix_gfc_w"], 2e-6)
    close(grads["bias"], g["mix_gfc_b"], 2e-6)


def test_mean_pool_variant_formula():
    """inference/inference.py:267: lambda_tok*toks + lambda_char*chars.mean(dim=-2)."""
    torch.manual_seed(0)
    E_tok, E_byte = torch.randn(10, 16), torch.randn(132, 16)
    toks = torch.randint(0, 10, (5,))
    chars = torch.randint(0, 132, (5, 8))
    spec, _ = O.VARIANTS["V7"]
    lt, lb = torch.tensor(0.7), torch.tensor(0.2)
    out = O.mot_embed_forward(spec, toks, chars, E_tok, E_byte, bpt=8, lam_tok=lt, lam_byte=lb)
    ref = lt * E_tok[toks] + lb * E_byte[chars].mean(dim=-2)
    assert torch.allclose(out, ref, atol=1e-6)
