"""Backward workspaces (sort plan + self-cleaning accumulators) under CUDA graphs.

A captured step is replayed with a different batch each time; eager calls and replays of a module of the same geometry
are interleaved; two modules of one geometry are graphed separately and run in one step; a second backward runs through
the same autograd graph (retain_graph); one capture holds more same-shaped workspaces than the eager pool keeps.  Every
gradient is checked against a float64 restatement of the operation on the same bf16 parameters (torch ops and autograd
on the GPU), on both dispatch paths (autograd.Function and torch.ops.mot_b200).  A gradient computed from another
batch's token plan is wrong by O(1), far above the bars: normalised max-abs 2^-8 for the sum and the gathers, 2^-6 for
the projection and byte-FC chains; rows no position gathered must be exactly zero.

Should a graph and an eager call (or two graphs) ever share a workspace again, these tests fail through wrong numbers
and not through a fault: every batch that could meet another's workspace has the same n_tokens and vocabulary, so a
plan of the wrong batch still indexes in bounds, and an eager forward and a replay are separated by a device synchronise
(two plans running at once on one histogram could produce offsets past the end of the stream).  Nothing here replays
after an eager forward was dropped without its backward.
"""
import gc

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

EPS = float(torch.finfo(torch.float32).eps)   # F.rms_norm's default eps, as the kernels use it
TOL_SUM = 2.0 ** -8                           # MoT-sum and token gathers
TOL_CHAIN = 2.0 ** -6                         # projection and byte-FC chains (bf16 product rounded before its norm)
BPT, VB, PAD = 16, 458, 456                   # bytes per token, byte vocabulary, the ttb tables' pad byte
BATCHES = ("uniform", "zipf", "one_token", "all_pad")


def dev():
    return torch.device("cuda:0")


@pytest.fixture(params=["autograd", "custom_ops"])
def dispatch(request):
    """Both dispatch paths: the autograd.Functions (eager default) and the torch.library operators."""
    import mot_b200
    from mot_b200 import _library
    prev = _library._FORCE
    mot_b200.set_custom_ops(request.param == "custom_ops")
    try:
        yield request.param
    finally:
        mot_b200.set_custom_ops(prev)


# ------------------------------------------------------------------------------------------- module families
class _Family:
    """One module family: how to build it, its inputs, and its float64 forward on the module's parameters."""
    tol = TOL_SUM
    ids_shape = None

    def __init__(self, V, N):
        self.V, self.N = V, N

    def args(self, tok, ids):
        return (tok, ids)

    def batch(self, kind, gen):
        """(tok, ids, gouts) of one batch: uniform tokens; Zipf tokens (rand^6: hot rows straddle the stream chunks);
        one token at every position (one row spanning every chunk); uniform tokens with every byte id the pad id."""
        d, N, V = dev(), self.N, self.V
        if kind == "zipf":
            tok = (torch.rand(N, generator=gen, device=d) ** 6 * V).long().clamp_(0, V - 1).int()
        elif kind == "one_token":
            tok = torch.randint(0, V, (1,), generator=gen, device=d, dtype=torch.int32).expand(N).contiguous()
        else:
            tok = torch.randint(0, V, (N,), generator=gen, device=d, dtype=torch.int32)
        ids = None
        if self.ids_shape is not None:
            ids = (torch.full(self.ids_shape, PAD, device=d, dtype=torch.int32) if kind == "all_pad"
                   else torch.randint(0, VB, self.ids_shape, generator=gen, device=d, dtype=torch.int32))
        gouts = [torch.randn(s, generator=gen, device=d).bfloat16() for s in self.out_shapes]
        return tok, ids, gouts


class _Sum(_Family):
    """MoTEmbedding V3 (runs/71): rms_norm(E_tok[tok] + cat_k E_byte[ids[k]]), ids [bpt, N]."""

    def __init__(self, V, N, Dt=512, bd=32, saved=True):
        super().__init__(V, N)
        self.Dt, self.bd, self.saved = Dt, bd, saved
        self.ids_shape = (BPT, N)
        self.out_shapes = [(1, N, Dt)]

    def build(self, seed):
        import mot_b200
        torch.manual_seed(seed)
        return mot_b200.MoTEmbedding(self.V, VB, self.Dt, self.bd, BPT, variant="V3").to(dev()).bfloat16()

    def check_kernel(self, m, tok, ids):
        """The family runs the backward kernel it is named after (saved-output for N <= 4V, else recompute)."""
        import mot_b200
        from mot_b200 import ops
        desc = ops.make_desc(mot_b200.MixSpec(combine="add", slot_major=True), self.N, m.embed_tokens.weight,
                             m.embed_bytes.weight, BPT, ids=ids, ttb=None, has_lam=False)
        assert ops.embed_bwd_uses_saved(desc) == self.saved

    def ref_forward(self, params, tok, ids):
        Et, Eb = params["embed_tokens.weight"], params["embed_bytes.weight"]
        z = _rows(Et, tok) + _rows(Eb, ids.t()).reshape(self.N, -1)
        return [F.rms_norm(z, (self.Dt,), eps=EPS)[None]]


class _Value(_Family):
    """TokenValueEmbeddings: three plain gathers E_i[tok]; the float64 gradient is index_add_ of the upstream rows."""

    def __init__(self, V, N, D=256):
        super().__init__(V, N)
        self.D = D
        self.out_shapes = [(N, D)] * 3

    def build(self, seed):
        import mot_b200
        torch.manual_seed(seed)
        return mot_b200.TokenValueEmbeddings(self.V, self.D).to(dev()).bfloat16()

    def args(self, tok, ids):
        return (tok,)

    def ref_grads(self, params, tok, ids, gouts):
        _rows(params["value_embeds.0.weight"], tok)                       # bounds check of the ids only
        return {f"value_embeds.{i}.weight": torch.zeros_like(params[f"value_embeds.{i}.weight"]).index_add_(
                    0, tok.long(), g.double()) for i, g in enumerate(gouts)}


def _v1_chain(Et, Eb, W, tok, ids_tm, N):
    """V1 (runs/7:226-234): rms_norm(F.linear(cat[rms_norm(E_tok[tok]) | rms_norm(E_byte[ids]) per byte], W)); ids
    token-major [N, bpt]."""
    t = F.rms_norm(_rows(Et, tok), (Et.shape[1],), eps=EPS)
    b = F.rms_norm(_rows(Eb, ids_tm), (Eb.shape[1],), eps=EPS).reshape(N, -1)
    y = F.linear(torch.cat([t, b], dim=-1), W)
    return F.rms_norm(y, (W.shape[0],), eps=EPS)


class _Proj(_Family):
    """MoTProjEmbedding V1, ids [1, N*bpt] token-major."""
    tol = TOL_CHAIN

    def __init__(self, V, N, Dt=128, bd=16, Do=256):
        super().__init__(V, N)
        self.Dt, self.bd, self.Do = Dt, bd, Do
        self.ids_shape = (1, N * BPT)
        self.out_shapes = [(1, N, Do)]

    def build(self, seed):
        import mot_b200
        torch.manual_seed(seed)
        return mot_b200.MoTProjEmbedding(self.V, VB, self.Dt, self.bd, self.Do, BPT, variant="V1").to(dev()).bfloat16()

    def ref_forward(self, params, tok, ids):
        Et, Eb, W = params["embed_tokens.weight"], params["embed_bytes.weight"], params["byte_mixin_weight"]
        return [_v1_chain(Et, Eb, W, tok, ids.view(self.N, BPT), self.N)[None]]


class _ByteFc(_Family):
    """MoTByteFcEmbedding V3f (runs/71051): rms_norm(E_tok[tok] + F.linear(cat_k E_byte[ids[k]], W)), ids [bpt, N]."""
    tol = TOL_CHAIN

    def __init__(self, V, N, bd=32):
        super().__init__(V, N)
        self.D, self.bd = BPT * bd, bd
        self.ids_shape = (BPT, N)
        self.out_shapes = [(1, N, self.D)]

    def build(self, seed):
        import mot_b200
        torch.manual_seed(seed)
        return mot_b200.MoTByteFcEmbedding(self.V, VB, self.D, self.bd, BPT).to(dev()).bfloat16()

    def ref_forward(self, params, tok, ids):
        Et, Eb, W = params["embed_tokens.weight"], params["embed_bytes.weight"], params["byte_fc"]
        c = _rows(Eb, ids.t()).reshape(self.N, -1)
        return [F.rms_norm(_rows(Et, tok) + F.linear(c, W), (self.D,), eps=EPS)[None]]


class _MotValue(_Family):
    """MoTValueEmbeddings (runs/9, V6) with n_tables V1 chains, every one with the same workspace geometry."""
    tol = TOL_CHAIN

    def __init__(self, V, N, n_tables, Dt=128, bd=16):
        super().__init__(V, N)
        self.Dt, self.bd, self.n_tables = Dt, bd, n_tables
        self.ids_shape = (1, N * BPT)
        self.out_shapes = [(1, N, Dt)] * n_tables

    def build(self, seed):
        import mot_b200
        torch.manual_seed(seed)
        return mot_b200.MoTValueEmbeddings(self.V, VB, self.Dt, self.bd, BPT, n_tables=self.n_tables).to(dev()).bfloat16()

    def ref_forward(self, params, tok, ids):
        # the byte value tables have token-vocabulary rows; ids < VB index only the live ones
        return [_v1_chain(params[f"value_embeds_toks.{i}.weight"], params[f"value_embeds_bytes.{i}.weight"],
                          params[f"value_byte_mixin_weights.{i}"], tok, ids.view(self.N, BPT), self.N)[None]
                for i in range(self.n_tables)]


FAMILIES = {
    "sum_saved": _Sum(1500, 2048, saved=True),          # N <= 4V: saved-output backward
    "sum_recompute": _Sum(300, 2048, saved=False),      # N > 4V: recompute backward
    "value": _Value(1000, 1536),
    "proj": _Proj(800, 1024),
    "byte_fc": _ByteFc(1000, 1024),
}


# ------------------------------------------------------------------------------------------- helpers
def _outputs(out):
    return list(out) if isinstance(out, (list, tuple)) else [out]


def _zero_grads(m):
    for p in m.parameters():
        p.grad = None


def _step(m, fam, tok, ids, gouts):
    torch.autograd.backward(_outputs(m(*fam.args(tok, ids))), gouts)


def _quiesce():
    # objects of earlier tests (graphs with private pools, tensors last used on a side stream) must not be finalised in
    # the middle of a capture: the caching allocator would query their events, which invalidates a global-mode capture
    gc.collect()
    torch.cuda.synchronize()


def _rows(E, idx):
    """E[idx] after a host-side bounds check of the ids (a reference that indexes out of range fails here)."""
    idx = idx.long()
    lo, hi = int(idx.min()), int(idx.max())
    assert 0 <= lo and hi < E.shape[0], f"ids in [{lo}, {hi}] index a table of {E.shape[0]} rows"
    return E[idx]


def _ref_grads(fam, m, tok, ids, gouts):
    """float64 dense gradients of every parameter of m (m.parameters() order) for one batch."""
    params = {name: p.detach().double().requires_grad_(True) for name, p in m.named_parameters()}
    if hasattr(fam, "ref_grads"):
        grads = fam.ref_grads(params, tok, ids, gouts)
    else:
        torch.autograd.backward(fam.ref_forward(params, tok, ids), [g.double() for g in gouts])
        grads = {name: p.grad for name, p in params.items()}
    return [grads[name] if grads.get(name) is not None else torch.zeros_like(params[name])
            for name, _ in m.named_parameters()]


def _check(what, got, want, tol, scale=1.0):
    """Normalised max-abs error of every gradient within tol; rows of a table the batch never gathered (zero rows of
    the float64 gradient) exactly zero."""
    errs, cold_rows = [], []
    for a, w in zip(got, want):
        w = w * scale
        a = a.detach().double()
        errs.append(float((a - w).abs().max() / w.abs().max().clamp_min(1e-300)))
        cold = (w == 0).all(1) if w.dim() == 2 else None
        cold_rows.append(0 if cold is None or not bool(cold.any()) else int((a[cold] != 0).any(1).sum()))
    assert all(e <= tol for e in errs), f"{what}: normalised max-abs errors {['%.3e' % e for e in errs]} (bar {tol:.3e})"
    assert not any(cold_rows), f"{what}: non-zero rows where no position gathered: {cold_rows}"


def _check_module(what, fam, m, batch, scale=1.0):
    tok, ids, gouts = batch
    _check(what, [p.grad for p in m.parameters()], _ref_grads(fam, m, tok, ids, gouts), fam.tol, scale)


def _capture_step(fam, m, static):
    """torch.cuda.graph around one whole step (forward, backward, gradients allocated in the graph's pool) after a
    warm-up on a side stream, as bench.py's end-to-end arm does.  Returns (graph, the gradients it writes)."""
    tok, ids, gouts = static
    _quiesce()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            _zero_grads(m)
            _step(m, fam, tok, ids, gouts)
    torch.cuda.current_stream().wait_stream(side)
    _quiesce()
    _zero_grads(m)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _step(m, fam, tok, ids, gouts)
    return graph, [p.grad for p in m.parameters()]


def _replay_fresh_batches(fam, m, gen, kinds):
    static = fam.batch("uniform", gen)
    graph, grads = _capture_step(fam, m, static)
    for kind in kinds:
        batch = fam.batch(kind, gen)
        for s, b in zip((static[0], static[1], *static[2]), (batch[0], batch[1], *batch[2])):
            if s is not None:
                s.copy_(b)
        graph.replay()
        torch.cuda.synchronize()
        _check(f"replay with a {kind} batch", grads, _ref_grads(fam, m, *batch), fam.tol)
    del graph


def _graphed(fam, m, gen):
    """m with its forward and backward captured by torch.cuda.make_graphed_callables."""
    tok, ids, _ = fam.batch("uniform", gen)
    _quiesce()
    g = torch.cuda.make_graphed_callables(m, fam.args(tok, ids))
    _quiesce()
    return g


# ------------------------------------------------------------------------------------------- a. fresh batches per replay
@pytest.mark.parametrize("fam_name", sorted(FAMILIES))
def test_captured_step_replays_fresh_batches(fam_name, dispatch):
    """One captured step replayed with a different batch each time: the captured plan reruns on every replay, and the
    workspace's self-cleaning contract (zero head, reset partial slots and work counters) holds when the token
    distribution changes from one replay to the next."""
    fam = FAMILIES[fam_name]
    gen = torch.Generator(device="cuda").manual_seed(101)
    m = fam.build(1)
    if isinstance(fam, _Sum):
        fam.check_kernel(m, *fam.batch("uniform", gen)[:2])
    _replay_fresh_batches(fam, m, gen, BATCHES)


def test_captured_step_replays_fresh_batches_at_baseline_shape(dispatch):
    """The headline shape (49152 tokens, V = 50257, 768 = 16 x 48, bf16, saved-output backward), including one token
    at all 49152 positions: a single row spanning every stream chunk of the saved-output kernel."""
    fam = _Sum(50257, 49152, Dt=768, bd=48, saved=True)
    gen = torch.Generator(device="cuda").manual_seed(102)
    m = fam.build(2)
    fam.check_kernel(m, *fam.batch("uniform", gen)[:2])
    _replay_fresh_batches(fam, m, gen, BATCHES)


# ------------------------------------------------------------------------------------------- b, c. eager and replay interleaved
@pytest.mark.parametrize("fam_name", sorted(FAMILIES))
def test_eager_forward_replay_eager_backward(fam_name, dispatch):
    """An eager forward, then a replayed step of a graphed module of the same geometry, then the eager backward: the
    replay must not overwrite the eager call's plan."""
    fam = FAMILIES[fam_name]
    gen = torch.Generator(device="cuda").manual_seed(103)
    m_g, m_e = fam.build(3), fam.build(4)
    graphed = _graphed(fam, m_g, gen)
    be, bg = fam.batch("uniform", gen), fam.batch("zipf", gen)
    _zero_grads(m_g)
    _zero_grads(m_e)
    outs_e = _outputs(m_e(*fam.args(be[0], be[1])))
    torch.cuda.synchronize()
    _step(graphed, fam, *bg)
    torch.autograd.backward(outs_e, be[2])
    torch.cuda.synchronize()
    _check_module("eager gradients", fam, m_e, be)
    _check_module("graphed gradients", fam, m_g, bg)


@pytest.mark.parametrize("fam_name", sorted(FAMILIES))
def test_replayed_forward_eager_step_replayed_backward(fam_name, dispatch):
    """A replayed forward, a complete eager step of a module of the same geometry, then the replayed backward: the
    eager step must not overwrite the graph's plan."""
    fam = FAMILIES[fam_name]
    gen = torch.Generator(device="cuda").manual_seed(104)
    m_g, m_e = fam.build(5), fam.build(6)
    graphed = _graphed(fam, m_g, gen)
    bg, be = fam.batch("zipf", gen), fam.batch("uniform", gen)
    _zero_grads(m_g)
    _zero_grads(m_e)
    outs_g = _outputs(graphed(*fam.args(bg[0], bg[1])))
    torch.cuda.synchronize()
    _step(m_e, fam, *be)
    torch.cuda.synchronize()
    torch.autograd.backward(outs_g, bg[2])
    torch.cuda.synchronize()
    _check_module("graphed gradients", fam, m_g, bg)
    _check_module("eager gradients", fam, m_e, be)


# ------------------------------------------------------------------------------------------- d. two graphs of one geometry
@pytest.mark.parametrize("fam_name", sorted(FAMILIES))
def test_two_modules_of_one_geometry_graphed_separately(fam_name, dispatch):
    """Two modules with identical shapes and different weights, each graphed by its own make_graphed_callables call,
    in one step: forward A, forward B, backward B, backward A.  Each graph keeps its own plan."""
    fam = FAMILIES[fam_name]
    gen = torch.Generator(device="cuda").manual_seed(105)
    m_a, m_b = fam.build(7), fam.build(8)
    graphed_a = _graphed(fam, m_a, gen)
    graphed_b = _graphed(fam, m_b, gen)
    ba, bb = fam.batch("uniform", gen), fam.batch("zipf", gen)
    _zero_grads(m_a)
    _zero_grads(m_b)
    outs_a = _outputs(graphed_a(*fam.args(ba[0], ba[1])))
    outs_b = _outputs(graphed_b(*fam.args(bb[0], bb[1])))
    # f(o) = sum(o * w) in fp32: the gradient reaching each output is w itself (bf16)
    loss = sum((o.float() * w.float()).sum() for o, w in zip(outs_a, ba[2])) + \
        sum((o.float() * w.float()).sum() for o, w in zip(outs_b, bb[2]))
    loss.backward()
    torch.cuda.synchronize()
    _check_module("module A", fam, m_a, ba)
    _check_module("module B", fam, m_b, bb)


# ------------------------------------------------------------------------------------------- e. retain_graph
@pytest.mark.parametrize("fam_name", sorted(FAMILIES))
def test_retain_graph_second_backward(fam_name, dispatch):
    """loss.backward(retain_graph=True) then loss.backward(): the first backward leaves the forward's plan intact (the
    operator path reuses that workspace as planned and clean), so the accumulated gradient is twice the reference."""
    fam = FAMILIES[fam_name]
    gen = torch.Generator(device="cuda").manual_seed(106)
    m = fam.build(9)
    batch = fam.batch("zipf", gen)
    _zero_grads(m)
    outs = _outputs(m(*fam.args(batch[0], batch[1])))
    loss = sum((o.float() * w.float()).sum() for o, w in zip(outs, batch[2]))
    loss.backward(retain_graph=True)
    first = [p.grad.clone() for p in m.parameters()]
    loss.backward()
    torch.cuda.synchronize()
    want = _ref_grads(fam, m, *batch)
    _check("first backward", first, want, fam.tol)
    _check("accumulated after the second backward", [p.grad for p in m.parameters()], want, fam.tol, scale=2.0)


# ------------------------------------------------------------------------------------------- f. many same-key workspaces
def test_many_same_key_workspaces_in_one_capture(dispatch):
    """MoTValueEmbeddings with six tables: six workspaces of one geometry in flight inside one captured step, more than
    the eager pool keeps.  Each belongs to the graph; replays with two different batches match the reference."""
    fam = _MotValue(800, 1024, n_tables=6)
    gen = torch.Generator(device="cuda").manual_seed(107)
    m = fam.build(10)
    _replay_fresh_batches(fam, m, gen, ("uniform", "zipf"))
