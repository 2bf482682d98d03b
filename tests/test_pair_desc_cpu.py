"""Return codes of the byte pair's descriptor entry points (mot_byte_pair_fwd/bwd), checked without a GPU.  For every
input the former scalar entry points could express (explicit ids, and the padded and pulled ids derived from the ttb
table, left, right and right with its lookahead) the descriptor form returns the code they returned, except for three
inputs that now follow the rules the fused kernels apply to every descriptor:
  (a) derived ids with pad_id or eot_id outside int16: MOT_ERR_BAD_ARG (was accepted);
  (b) row_stride 0 with col_offset 0: dense rows of out_dim elements (was MOT_ERR_BAD_ARG);
  (c) a row stride above INT32_MAX: MOT_ERR_BAD_ARG (was accepted).
The expected codes below were produced by the former entry points.  The calls pass dummy, non-null, 256-aligned device
addresses: without a device an accepted call stops at the device query (MOT_ERR_NO_DEVICE) before it launches or
dereferences anything, so the file runs only where torch finds no CUDA device."""
import ctypes as C

import pytest
import torch

from mot_b200 import _lib as L

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="passes dummy device addresses: CPU-only machines")

SOURCES = ("i32", "i64", "left", "right", "next")   # explicit int32 / int64 ids; derived: left, right, right + lookahead
NS = (0, 64)
BDS = tuple(range(8, 521, 8)) + (44,)
BASE = dict(dtype=L.BF16, bpt=16, bd=48, Vb=458, col=256, ld=None, eps=1e-7, seq_len=16, tok_vocab=100,
            ttb_dtype=L.TTB_I16, pad=456, eot=457, null=None, shift=None)
PTR = dict(tok=0x100000, ids_a=0x200000, ids_b=0x300000, ttb=0x400000, E_byte=0x500000, out=0x600000, gE=0x700000,
           ws=0x800000)
PULL = {"left": L.F_TTB_PULL_LEFT, "right": L.F_TTB_PULL_RIGHT, "next": L.F_TTB_PULL_RIGHT | L.F_TTB_NEXT_TOK}

# one field (or one pointer) changed from BASE; every variant runs for each source and each n
VARIANTS = (
    {}, {"dtype": L.F32}, {"dtype": 7}, {"dtype": 7, "bd": 44}, {"dtype": L.F32, "bpt": 4, "bd": 512},
    {"Vb": 0}, {"Vb": -1}, {"n": -1}, {"n": 1 << 31},
    {"ld": 256 + 16 * 48 + 8}, {"ld": 256 + 16 * 48 - 8}, {"ld": 256 + 16 * 48 + 4}, {"ld": 0},
    {"col": 4}, {"col": -8}, {"col": 8}, {"col": 0, "ld": 16 * 48}, {"col": 0, "ld": 0}, {"col": 0, "ld": 1 << 31},
    {"seq_len": 64}, {"seq_len": 48}, {"seq_len": 0}, {"seq_len": -16},
    {"tok_vocab": 1}, {"tok_vocab": 0}, {"tok_vocab": -1},
    {"ttb_dtype": L.TTB_F32}, {"ttb_dtype": L.TTB_BF16}, {"ttb_dtype": 3}, {"ttb_dtype": -1},
    {"pad": 32767}, {"pad": 32768}, {"eot": -32768}, {"eot": -32769},
    {"null": "tok"}, {"null": "ids_a"}, {"null": "ids_b"}, {"null": "ttb"}, {"null": "E_byte"}, {"null": "out"},
    {"shift": ("E_byte", 8)}, {"shift": ("out", 8)}, {"shift": ("ids_a", 4)}, {"shift": ("tok", 4)},
)


def case(src, n_tokens, **over):
    c = dict(BASE, src=src, n=n_tokens)
    c.update(over)
    if c["ld"] is None:
        c["ld"] = c["col"] + c["bpt"] * c["bd"]
    return c


def pointers(c):
    """Device addresses of the call: the unused id source NULL, as the descriptor form asks."""
    p = dict(PTR)
    for k in (("tok", "ttb") if c["src"] in ("i32", "i64") else ("ids_a", "ids_b")):
        p[k] = None
    if c["null"]:
        p[c["null"]] = None
    if c["shift"] and p[c["shift"][0]]:
        p[c["shift"][0]] += c["shift"][1]
    return p


def changed(c):
    """The new code of the three inputs (a)-(c) of the module docstring, else None."""
    derived = c["src"] not in ("i32", "i64")
    if derived and (c["pad"] != C.c_int16(c["pad"]).value or c["eot"] != C.c_int16(c["eot"]).value):
        return L.ERR_BAD_ARG
    if c["ld"] == 0 and c["col"] == 0:
        return old_dense(c)
    if c["ld"] > 0x7FFFFFFF:
        return L.ERR_BAD_ARG
    return None


def old_dense(c):
    """Code of the same call with the dense stride spelt out (ld = bpt*bd)."""
    return CODES[variant_key(dict(c, ld=c["bpt"] * c["bd"]))]


def desc(c):
    derived = c["src"] not in ("i32", "i64")
    flags = L.F_BYTE_NORM | (L.F_IDS_FROM_TTB | PULL[c["src"]] if derived else 0)
    flags |= L.F_IDS_I64 if c["src"] == "i64" else 0
    return L.MotDesc(abi_version=L.ABI_VERSION, dtype=c["dtype"], n_tokens=c["n"], seq_len=c["seq_len"] if derived else 0,
                     tok_vocab=c["tok_vocab"] if derived else 0, byte_vocab=c["Vb"], bpt=c["bpt"], tok_dim=0,
                     byte_dim=c["bd"], out_dim=c["bpt"] * c["bd"], combine=L.BYTES_ONLY, flags=flags,
                     ttb_dtype=c["ttb_dtype"] if derived else 0, eps=c["eps"], row_stride=c["ld"], col_offset=c["col"],
                     pad_id=c["pad"] if derived else 0, eot_id=c["eot"] if derived else 0)


def new_fwd(c):
    p = pointers(c)
    return L.lib().mot_byte_pair_fwd(desc(c), p["tok"], p["ids_a"], p["ids_b"], p["ttb"], p["E_byte"], p["out"], None)


def new_bwd(c):
    p = pointers(c)
    return L.lib().mot_byte_pair_bwd(desc(c), p["tok"], p["ids_a"], p["ids_b"], p["ttb"], p["E_byte"], p["out"], p["gE"],
                                     p["ws"], 1 << 30, None)


def refused_before_memset(c, code):
    """The backward clears gE_byte (n == 0) or its workspace before the pair kernels' own capacity check: it is called
    only where the descriptor checks refuse the call.  At n == 0 every refusal is one of those."""
    return code in (L.ERR_BAD_ARG, L.ERR_MISALIGNED) or (code == L.ERR_UNSUPPORTED and c["n"] == 0)


def variant_key(c):
    over = tuple(sorted((k, v) for k, v in c.items() if k not in ("src", "n") and BASE.get(k, object()) != v
                        and not (k == "ld" and v == c["col"] + c["bpt"] * c["bd"])))
    return c["src"], c["n"], over


# ---- codes of the former entry points ---------------------------------------------------------------------------
# SHAPES[n][bpt - 1][i]: the code for byte_dim BDS[i] with the BASE layout, the same for every source and dtype 0 / 1
SHAPES = {
    0: (
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "000000000000000000000000000000000000000000000000000000000000000003",
        "111111111111111111111111111111111111111111111111111111111111111111",
    ),
    64: (
        "666666666666666222222222222222222222222222222222222222222222222223",
        "666666666666666222222222222222222222222222222222222222222222222223",
        "666666666666666666666666666666666666666666666666666666666666666623",
        "666666666666666666666666666666666666666666666666666666666666666623",
        "666666666666666666666666666666662222222222222222222222222222222223",
        "666666666666666666666666666666662222222222222222222222222222222223",
        "666666666666666666666666666666662222222222222222222222222222222223",
        "666666666666666666666666666666662222222222222222222222222222222223",
        "666666666666666622222222222222222222222222222222222222222222222223",
        "666666666666666622222222222222222222222222222222222222222222222223",
        "666666666666666622222222222222222222222222222222222222222222222223",
        "666666666666666622222222222222222222222222222222222222222222222223",
        "666666666666666622222222222222222222222222222222222222222222222223",
        "666666666666666622222222222222222222222222222222222222222222222223",
        "666666666666666622222222222222222222222222222222222222222222222223",
        "666666666666666622222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "666666662222222222222222222222222222222222222222222222222222222223",
        "111111111111111111111111111111111111111111111111111111111111111111",
    ),
}
# VARIANT_CODES[i]: codes of VARIANTS[i] for (source, n) in SOURCES x NS order
VARIANT_CODES = (
    "0606060606",   # {}
    "0606060606",   # {'dtype': 1}
    "2222222222",   # {'dtype': 7}
    "2222222222",   # {'dtype': 7, 'bd': 44}
    "0606060606",   # {'dtype': 1, 'bpt': 4, 'bd': 512}
    "1111111111",   # {'Vb': 0}
    "1111111111",   # {'Vb': -1}
    "1111111111",   # {'n': -1}
    "1111111111",   # {'n': 2147483648}
    "0606060606",   # {'ld': 1032}
    "1111111111",   # {'ld': 1016}
    "3333333333",   # {'ld': 1028}
    "1111111111",   # {'ld': 0}
    "3333333333",   # {'col': 4}
    "1111111111",   # {'col': -8}
    "0606060606",   # {'col': 8}
    "0606060606",   # {'col': 0, 'ld': 768}
    "1111111111",   # {'col': 0, 'ld': 0}
    "0606060606",   # {'col': 0, 'ld': 2147483648}
    "0606060606",   # {'seq_len': 64}
    "0606010101",   # {'seq_len': 48}
    "0606111111",   # {'seq_len': 0}
    "0606111111",   # {'seq_len': -16}
    "0606060606",   # {'tok_vocab': 1}
    "0606111111",   # {'tok_vocab': 0}
    "0606111111",   # {'tok_vocab': -1}
    "0606060606",   # {'ttb_dtype': 1}
    "0606060606",   # {'ttb_dtype': 2}
    "0606222222",   # {'ttb_dtype': 3}
    "0606222222",   # {'ttb_dtype': -1}
    "0606060606",   # {'pad': 32767}
    "0606060606",   # {'pad': 32768}
    "0606060606",   # {'eot': -32768}
    "0606060606",   # {'eot': -32769}
    "0606010101",   # {'null': 'tok'}
    "0101060606",   # {'null': 'ids_a'}
    "0101060606",   # {'null': 'ids_b'}
    "0606010101",   # {'null': 'ttb'}
    "0101010101",   # {'null': 'E_byte'}
    "0101010101",   # {'null': 'out'}
    "0303030303",   # {'shift': ('E_byte', 8)}
    "0303030303",   # {'shift': ('out', 8)}
    "0606060606",   # {'shift': ('ids_a', 4)}
    "0606060606",   # {'shift': ('tok', 4)}
)


def _expected_variants():
    out = {}
    for v, codes in zip(VARIANTS, VARIANT_CODES):
        for (src, n), code in zip([(s, n) for s in SOURCES for n in NS], codes):
            out[variant_key(case(src, n, **v))] = int(code)
    return out


CODES = _expected_variants()


def test_expected_codes_cover_the_grid():
    assert len(VARIANT_CODES) == len(VARIANTS) and all(len(s) == len(SOURCES) * len(NS) for s in VARIANT_CODES)
    assert sorted(SHAPES) == list(NS)
    assert all(len(SHAPES[n]) == 33 and all(len(r) == len(BDS) for r in SHAPES[n]) for n in NS)


@pytest.mark.parametrize("src", SOURCES)
@pytest.mark.parametrize("dtype", [L.BF16, L.F32])
@pytest.mark.parametrize("n", NS)
def test_shape_grid_keeps_the_codes(src, dtype, n):
    got, want = [], []
    for bpt in range(1, 34):
        for i, bd in enumerate(BDS):
            c = case(src, n, dtype=dtype, bpt=bpt, bd=bd)
            code = int(SHAPES[n][bpt - 1][i])
            got.append((bpt, bd, new_fwd(c)))
            want.append((bpt, bd, code))
            if refused_before_memset(c, code):
                got.append((bpt, bd, "bwd", new_bwd(c)))
                want.append((bpt, bd, "bwd", code))
    assert got == want
    # the pair keeps byte_dim up to 64 * G: the fused kernels' 256 cap under MOT_F_BYTE_NORM does not reach it
    assert int(SHAPES[64][3][BDS.index(512)]) == L.ERR_NO_DEVICE


@pytest.mark.parametrize("src", SOURCES)
@pytest.mark.parametrize("n", NS)
def test_one_field_at_a_time_keeps_the_codes(src, n):
    got, want = [], []
    for v in VARIANTS:
        c = case(src, n, **v)
        old = CODES[variant_key(c)]
        new = changed(c)
        code = old if new is None else new
        got.append((v, new_fwd(c)))
        want.append((v, code))
        if new is None and refused_before_memset(c, code):
            got.append((v, "bwd", new_bwd(c)))
            want.append((v, "bwd", code))
    assert got == want


def test_the_three_changed_verdicts():
    """(a)-(c) of the module docstring, one input each: the former code, then the new one."""
    for c, old, new in ((case("left", 64, pad=32768), L.ERR_NO_DEVICE, L.ERR_BAD_ARG),
                        (case("i64", 64, col=0, ld=0), L.ERR_BAD_ARG, L.ERR_NO_DEVICE),
                        (case("i32", 0, col=0, ld=1 << 31), L.OK, L.ERR_BAD_ARG)):
        assert (CODES[variant_key(c)], new_fwd(c)) == (old, new)
