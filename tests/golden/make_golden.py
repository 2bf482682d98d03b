"""Generate the golden fixtures in this directory FROM THE REFERENCE ITSELF.

Runs only in the build container, where the reference checkout is mounted at
/root/reference (read-only).  It imports / AST-extracts the reference's own
functions and modules, runs them eagerly on CPU on seeded inputs and stores
inputs + outputs as small .npz files.  The GPU box has no /root/reference, so
tests only ever read the committed .npz files.

    TORCHDYNAMO_DISABLE=1 python tests/golden/make_golden.py

Nothing from the reference's sources is copied: only numeric inputs/outputs.
"""
from __future__ import annotations

import ast
import zlib
import dataclasses
import json
import os
import sys
from typing import Literal

os.environ.setdefault("TORCHDYNAMO_DISABLE", "1")

import numpy as np
import torch
import torch.nn.functional as F
from torch import Tensor, nn

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))


def extract(path: str, names: list[str], ns: dict) -> dict:
    """exec the named top-level ClassDef/FunctionDef nodes of `path` in `ns`."""
    src = open(path).read()
    tree = ast.parse(src)
    want = set(names)
    body = []
    for node in tree.body:
        if isinstance(node, (ast.ClassDef, ast.FunctionDef)) and node.name in want:
            # drop decorators such as @torch.compile: eager CPU execution
            if isinstance(node, ast.FunctionDef):
                node.decorator_list = [d for d in node.decorator_list
                                       if "compile" not in ast.unparse(d)]
            body.append(node)
    mod = ast.Module(body=body, type_ignores=[])
    exec(compile(mod, path, "exec"), ns)
    missing = want - {n.name for n in body}
    assert not missing, f"{path}: missing {missing}"
    return ns


def np_(t):
    if isinstance(t, torch.Tensor):
        t = t.detach()
        if t.dtype == torch.bfloat16:
            return t.float().numpy()
        return t.numpy()
    return np.asarray(t)


# --------------------------------------------------------------------------
# 1. the checked-in integer golden: ttb_8_left_pad.json, byte_to_int.json
# --------------------------------------------------------------------------
def golden_tables():
    ttb = json.load(open(f"{REF}/modded-nanogpt/embeddings/ttb_8_left_pad.json"))
    keys = sorted(int(k) for k in ttb)
    assert keys == list(range(50256))
    tab = np.asarray([ttb[str(k)] for k in keys], dtype=np.int16)
    np.savez_compressed(f"{HERE}/ttb_8_left_pad.npz", table=tab)
    b2i = json.load(open(f"{REF}/modded-nanogpt/embeddings/byte_to_int.json"))
    i2b = json.load(open(f"{REF}/modded-nanogpt/embeddings/int_to_byte.json"))
    assert {v: k for k, v in b2i.items()} == {int(k): v for k, v in i2b.items()}
    with open(f"{HERE}/byte_to_int.json", "w") as f:
        json.dump(b2i, f)
    print("tables:", tab.shape)


# --------------------------------------------------------------------------
# 2. integer path run through the reference's data_creation.py
# --------------------------------------------------------------------------
def golden_integer_path():
    sys.path.insert(0, f"{REF}/scaled-pre-train")
    cwd = os.getcwd()
    os.chdir(f"{REF}/modded-nanogpt")  # embeddings/ttb_8_left_pad.json resolves (data_creation.py:44)
    import data_creation as dc
    torch.manual_seed(1234)
    emb = dc.make_embedding("ttb_8_left_pad.json", 50257)
    os.chdir(cwd)
    # the reference leaves row 50256 at its N(0,1) init; give it the row the pull
    # functions need (create_ttb.py:20-22) -- documented in oracle.ttb_dict_to_array
    emb.weight.data[50256] = 457.0
    out = {}
    g = torch.Generator().manual_seed(12345)
    for name, (B, T, p_eot) in {"a": (2, 6, 0.0), "b": (4, 33, 0.2), "c": (3, 64, 0.5), "d": (1, 128, 0.05)}.items():
        toks = torch.randint(0, 50256, (B, T), generator=g, dtype=torch.int32)
        eot = torch.rand(B, T, generator=g) < p_eot
        toks = torch.where(eot, torch.tensor(50256, dtype=torch.int32), toks)
        if name == "c":  # EOT at first and last position
            toks[0, 0] = 50256
            toks[1, -1] = 50256
        left = dc.tokens_to_bytes(toks, emb)
        pfl = dc.pull_from_left(left, 8, 456, 457)
        out[f"{name}_tokens"] = np_(toks)
        out[f"{name}_bytes_left"] = np_(left)
        out[f"{name}_pull_from_left"] = np_(pfl)
        # right-padded table: derive rows the way create_ttb would (exact for all
        # rows with >= 1 pad; for full rows left == right)
        w = emb.weight.data.clone().long()
        wr = torch.full_like(w, 456)
        for v in range(w.shape[0]):
            row = w[v]
            ch = row[row != 456]
            wr[v, : len(ch)] = ch
        emb_r = nn.Embedding(50257, 8)
        emb_r.weight.data = wr.float()
        right = dc.tokens_to_bytes(toks, emb_r)
        pfr = dc.pull_from_right(right, 8, 456, 457)
        out[f"{name}_bytes_right"] = np_(right)
        out[f"{name}_pull_from_right"] = np_(pfr)
    # 1-D tokens -> [1, T*bpt] (data_creation.py:66-67)
    t1 = torch.randint(0, 50256, (40,), generator=g, dtype=torch.int32)
    out["e_tokens"] = np_(t1)
    out["e_bytes_left"] = np_(dc.tokens_to_bytes(t1, emb))
    # the bf16 table quirk of the runs (runs/7:441,446)
    emb16 = nn.Embedding(50257, 8)
    emb16.weight.data = emb.weight.data.clone()
    emb16 = emb16.bfloat16()
    out["e_bytes_left_bf16quirk"] = np_(dc.tokens_to_bytes(t1, emb16))
    out["bf16_id_map"] = torch.arange(458.0).bfloat16().long().numpy()
    np.savez_compressed(f"{HERE}/integer_path.npz", **out)
    print("integer path:", {k: v.shape for k, v in out.items()})
    return dc


# --------------------------------------------------------------------------
# 3. scaled-pre-train float path (FlexibleEmbedding + ByteMixinConcat)
# --------------------------------------------------------------------------
def golden_spt():
    import einops
    ns = dict(torch=torch, nn=nn, F=F, einops=einops, Tensor=Tensor, Literal=Literal,
              dataclass=dataclasses.dataclass)
    extract(f"{REF}/scaled-pre-train/train_gpt.py",
            ["ByteHyperparameters", "ModelDims", "norm", "CastedLinear", "FlexibleEmbedding",
             "ByteMixinNoop", "ByteMixinConcat", "ByteMixin"], ns)
    # ByteMixinConcat references ByteSelfAttn only when use_byte_self_attn=True
    ns["ByteSelfAttn"] = None
    ns["ByteMixinCrossAttn"] = None
    out = {}
    V, Vb = 96, 458
    for tag, (Dt, bd, Do, bpt, pull_in, add_pp, dtype) in {
        "concat_f32": (32, 8, 48, 4, True, False, torch.float32),
        "concat_bf16": (64, 16, 64, 4, True, False, torch.bfloat16),
        "concat_padded_f32": (32, 8, 48, 4, False, False, torch.float32),
        "concat_addpp_f32": (32, 8, 48, 4, True, True, torch.float32),
        "noop_f32": (32, 8, 32, 4, True, False, torch.float32),
    }.items():
        torch.manual_seed(zlib.crc32(tag.encode()) % 1000 + 7)
        method = "noop" if tag.startswith("noop") else "concat"
        bp = ns["ByteHyperparameters"](bytes_per_token=bpt, vocab_size=Vb, byte_mixin_method=method,
                                       pull_in=pull_in, add_padded_and_pulled=add_pp)
        dims = ns["ModelDims"](model_dim=Do, byte_dim=bd, token_dim=Dt)
        emb = ns["FlexibleEmbedding"](dims, V, bp)
        mix = ns["ByteMixin"](dims, 16, bp)
        if dtype == torch.bfloat16:  # train_gpt.py:1124-1126: embeddings to bf16, linear stays fp32
            for m in emb.modules():
                if isinstance(m, nn.Embedding):
                    m.bfloat16()
        B, S = 2, 12
        toks = torch.randint(0, V, (B, S), dtype=torch.int32)
        bytes_padded = torch.randint(0, Vb, (B, S * bpt), dtype=torch.int64)
        bytes_pulled = torch.randint(0, Vb, (B, S * bpt), dtype=torch.int64)
        xt, xb = emb(toks, bytes_padded, bytes_pulled)
        x = mix(xt, xb)
        gout = torch.randn_like(x.float()).to(x.dtype)
        x.backward(gout)
        out[f"{tag}_tokens"] = np_(toks)
        out[f"{tag}_bytes_padded"] = np_(bytes_padded)
        out[f"{tag}_bytes_pulled"] = np_(bytes_pulled)
        out[f"{tag}_E_tok"] = np_(emb.embed_tokens.weight)
        out[f"{tag}_gE_tok"] = np_(emb.embed_tokens.weight.grad)
        if method != "noop":
            out[f"{tag}_E_byte"] = np_(emb.embed_bytes.weight)
            out[f"{tag}_gE_byte"] = np_(emb.embed_bytes.weight.grad)
            out[f"{tag}_W"] = np_(mix.mixin.mixin.weight)
            out[f"{tag}_gW"] = np_(mix.mixin.mixin.weight.grad)
        out[f"{tag}_out"] = np_(x)
        out[f"{tag}_gout"] = np_(gout)
    np.savez_compressed(f"{HERE}/spt_float.npz", **out)
    print("spt float:", len(out), "arrays")


# --------------------------------------------------------------------------
# 4. modded-nanogpt runs: mixin_bytes of each variant + the three forward lines
# --------------------------------------------------------------------------
RUNS = {
    # tag: (file, has_weight, forward-lines restated below, slot_major ids)
    "V1_run7": ("7_mot-in_toks-valemb.py", "W"),
    "V2_run72": ("72_mot-in_toks-valemb.py", "W"),
    "V3_run71": ("71_mot-in_toks-valemb.py", None),
    "V3b_run73": ("73_mot-in_toks-valemb.py", None),
    "V3c_run74": ("74_mot-in_toks-valemb.py", None),
    "V3d_run71041": ("71041_mot-in_toks-valemb.py", None),
    "V3f_run71051": ("71051_mot-in_toks-valemb.py", "FC"),
    "V4_run711": ("711_mot-in_toks-valemb.py", None),
}


def golden_runs():
    out = {}
    T, bpt, bd, V, Vb = 24, 16, 8, 80, 458
    for tag, (fname, wkind) in RUNS.items():
        ns = dict(torch=torch, nn=nn, F=F, Tensor=Tensor)
        extract(f"{REF}/modded-nanogpt/runs/{fname}", ["norm", "mixin_bytes"], ns)
        norm, mixin_bytes = ns["norm"], ns["mixin_bytes"]
        for dt_tag, dtype in (("f32", torch.float32), ("bf16", torch.bfloat16)):
            torch.manual_seed(zlib.crc32(tag.encode()) % 997 + (0 if dt_tag == "f32" else 1))
            Dt = bpt * bd if tag.startswith(("V3",)) else 32
            Do = {"V1_run7": 40, "V2_run72": 40}.get(tag, Dt if tag.startswith("V3") else Dt + bpt * bd)
            embed_tokens = nn.Embedding(V, Dt).to(dtype)
            embed_bytes = nn.Embedding(Vb, bd).to(dtype)
            W = None
            if wkind == "W":
                W = nn.Parameter((torch.randn(Do, Dt + bpt * bd) * (Dt + bpt * bd) ** -0.5).to(dtype))
            elif wkind == "FC":
                W = nn.Parameter((torch.randn(Do, Do) * Do ** -0.5).to(dtype))
            scalars = nn.Parameter(torch.tensor([0.3, 0.7]))  # [-2]=byte lambda, [-1]=token lambda
            token_inputs = torch.randint(0, V, (T,), dtype=torch.int32)
            flat = torch.randint(0, Vb, (1, T * bpt), dtype=torch.int32)
            # the forward lines of GPT.forward, restated per run (cited in oracle.VARIANTS)
            if tag == "V1_run7":      # runs/7:317-319, ids [1, T*bpt]
                byte_inputs = flat
                x_toks = norm(embed_tokens(token_inputs)[None])
                x_bytes = norm(embed_bytes(byte_inputs).squeeze()[None])
                x = mixin_bytes(x_toks, x_bytes, W)
            elif tag == "V2_run72":   # runs/72:313-315, ids .view(16,-1) (:480)
                byte_inputs = flat.view(bpt, -1).contiguous()
                x_toks = embed_tokens(token_inputs)[None]
                x_bytes = embed_bytes(byte_inputs).squeeze()
                x = mixin_bytes(x_toks, x_bytes, W)
            elif tag == "V3_run71":   # runs/71:312-314, ids .view(16,-1) (:479)
                byte_inputs = flat.view(bpt, -1).contiguous()
                x_toks = embed_tokens(token_inputs)[None]
                x_bytes = embed_bytes(byte_inputs).squeeze()
                x = mixin_bytes(x_toks, x_bytes)
            elif tag == "V3b_run73":  # runs/73:313-315
                byte_inputs = flat.view(bpt, -1).contiguous()
                x_toks = norm(embed_tokens(token_inputs)[None])
                x_bytes = norm(embed_bytes(byte_inputs).squeeze())
                x = mixin_bytes(x_toks, x_bytes)
            elif tag in ("V3c_run74", "V3d_run71041"):  # runs/74:314-316, runs/71041:311-313
                byte_inputs = flat.view(bpt, -1).contiguous()
                x_toks = norm(embed_tokens(token_inputs)[None]) * scalars[-1]
                x_bytes = norm(embed_bytes(byte_inputs).squeeze()) * scalars[-2]
                x = mixin_bytes(x_toks, x_bytes)
            elif tag == "V3f_run71051":  # runs/71051:312-314
                byte_inputs = flat.view(bpt, -1).contiguous()
                x_toks = embed_tokens(token_inputs)[None]
                x_bytes = embed_bytes(byte_inputs).squeeze()
                x = mixin_bytes(x_toks, x_bytes, W)
            elif tag == "V4_run711":  # runs/711:314-316, ids [1, T*bpt] (:481)
                byte_inputs = flat
                x_toks = embed_tokens(token_inputs)[None]
                x_bytes = embed_bytes(byte_inputs).squeeze()[None]
                x = mixin_bytes(x_toks, x_bytes)
            gout = torch.randn(x.shape).to(x.dtype)
            x.backward(gout)
            k = f"{tag}_{dt_tag}"
            out[f"{k}_tokens"] = np_(token_inputs)
            out[f"{k}_byte_inputs"] = np_(byte_inputs)
            out[f"{k}_E_tok"] = np_(embed_tokens.weight)
            out[f"{k}_E_byte"] = np_(embed_bytes.weight)
            out[f"{k}_gE_tok"] = np_(embed_tokens.weight.grad)
            out[f"{k}_gE_byte"] = np_(embed_bytes.weight.grad)
            if W is not None:
                out[f"{k}_W"] = np_(W)
                out[f"{k}_gW"] = np_(W.grad)
            if scalars.grad is not None:
                out[f"{k}_scalars"] = np_(scalars)
                out[f"{k}_gscalars"] = np_(scalars.grad)
            out[f"{k}_out"] = np_(x)
            out[f"{k}_gout"] = np_(gout)
    for dt in ("f32", "bf16"):     # one file per dtype keeps each fixture under 1 MB
        np.savez_compressed(f"{HERE}/runs_float_{dt}.npz", **{k: v for k, v in out.items() if k.split("_")[2] == dt})
    print("runs float:", len(out), "arrays")


# --------------------------------------------------------------------------
# 5. mathblations: tokens_to_digits + DigitMixinConcat
# --------------------------------------------------------------------------
def golden_mathblations():
    sys.path.insert(0, f"{REF}/mathblations")
    import data as mdata
    import model as mmodel
    out = {}
    gen = mdata.GenerateEquations(max_digits_per_token=4, max_tokens_per_num=3, op="+", mod=None)
    toks = torch.tensor([0, 7, 42, 999, 4245, 9999, gen.op_token, gen.eq_token, gen.pad_token, 1000, 10])
    out["digits_tokens"] = np_(toks)
    out["digits_out"] = np_(gen.tokens_to_digits(toks))
    out["digits_meta"] = np.asarray([gen.max_digits_per_token, gen.op_token, gen.eq_token, gen.pad_token, gen.vocab_size])
    torch.manual_seed(5)
    gen = mdata.GenerateEquations(max_digits_per_token=2, max_tokens_per_num=3, op="+", mod=None)  # small vocab (103)
    cfg = mmodel.GPTConfig(vocab_size=gen.vocab_size, n_layer=1, n_head=2, n_embd_tok=32, n_embd_digit=16, T=12, length_factor=2,
                           digit_mixin_method="concat")
    net = mmodel.GPT(cfg)
    B, S = 3, 11
    idx = torch.randint(0, gen.vocab_size, (B, S))
    digits = torch.stack([gen.tokens_to_digits(row) for row in idx])
    we = net.wte(idx)
    de = net.dte(digits)
    x = net.digit_mixin(we, de)
    gout = torch.randn_like(x)
    x.backward(gout)
    out["mix_idx"] = np_(idx)
    out["mix_digits"] = np_(digits)
    out["mix_wte"] = np_(net.wte.weight)
    out["mix_dte"] = np_(net.dte.weight)
    out["mix_fc_w"] = np_(net.digit_mixin.fc.weight)
    out["mix_fc_b"] = np_(net.digit_mixin.fc.bias)
    out["mix_out"] = np_(x)
    out["mix_gout"] = np_(gout)
    out["mix_gwte"] = np_(net.wte.weight.grad)
    out["mix_gdte"] = np_(net.dte.weight.grad)
    out["mix_gfc_w"] = np_(net.digit_mixin.fc.weight.grad)
    out["mix_gfc_b"] = np_(net.digit_mixin.fc.bias.grad)
    np.savez_compressed(f"{HERE}/mathblations.npz", **out)
    print("mathblations:", len(out), "arrays")


if __name__ == "__main__":
    assert os.path.isdir(REF), "make_golden.py runs only where /root/reference is mounted"
    golden_tables()
    golden_integer_path()
    golden_spt()
    golden_runs()
    golden_mathblations()
