"""GATConv's backward against float64: the C entries gnnb_gat_aggregate(+_bwd) against the oracle's closed-form pullback
(orc_gat_aggregate_bwd) on every dispatch branch, the logit-term gate against what csrc/gatlogit.cu accepts, and the layer's
gradients (dx, dW, da, db) against torch float64 autograd of a plain restatement of gat_conv, up to config-3 scale.

Bounds.  Outputs without cancellation (out, alpha, dWx, dx, dW, db) are held to 1e-5 normwise of fp64, the reference's own
gradient tolerance (GraphNeuralNetworks/test/test_module.jl:81-121).  del, der and da sum dz = α (dα − T) lrelu'(z), a
difference of O(1) terms: each is held to max(1e-5, 4 e32), where e32 is the error of the same formula run in float32 on the
CPU against fp64 on the same inputs — the conditioning of the quantity, measured, not guessed — and e32 itself must stay under
1e-4 so the bound cannot turn vacuous.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

BAR = 1e-5


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape and np.isfinite(a).all()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def check_plain(name, got, ref):
    err = rel(got, ref)
    assert err < BAR, f"{name}: err {err:.2e} >= {BAR:.0e}"
    return err


def check_cancelling(name, got, ref, ref32, record=None):
    """got: the GPU's fp32 result; ref: fp64; ref32: the fp32 CPU restatement on the same inputs"""
    err, e32 = rel(got, ref), rel(ref32, ref)
    if record is not None:
        record(f"err_{name}", f"{err:.3e}")
        record(f"e32_{name}", f"{e32:.3e}")
    assert e32 < 1e-4, f"{name}: e32 {e32:.2e} (err {err:.2e}): the fp32 formula itself is ill-conditioned here"
    assert err <= max(BAR, 4 * e32), f"{name}: err {err:.2e} > max(1e-5, 4 e32 = {4 * e32:.2e})"
    return err, e32


# ------------------------------------------------------------------------------------------------------- graphs
def make_graph(rng, n, E, hubs=0, hub_deg=0, empty_frac=0.3, src_hubs=0):
    """random multigraph; the top `empty_frac` of the node ids receive no edges; `hubs` targets get hub_deg extra in-edges,
    `src_hubs` sources hub_deg extra out-edges (long rows of the transposed plan)"""
    hi = max(1, int(n * (1 - empty_frac)))
    s = rng.integers(1, n + 1, E)
    t = rng.integers(1, hi + 1, E)
    for h in range(hubs):
        s = np.concatenate([s, rng.integers(1, n + 1, hub_deg)])
        t = np.concatenate([t, np.full(hub_deg, 1 + 3 * h)])
    for h in range(src_hubs):
        s = np.concatenate([s, np.full(hub_deg, 2 + 5 * h)])
        t = np.concatenate([t, rng.integers(1, hi + 1, hub_deg)])
    p = rng.permutation(len(s))
    return s[p].astype(np.int64), t[p].astype(np.int64)


GRAPHS = {
    "small": dict(n=37, E=150),
    "empty_rows": dict(n=200, E=300, empty_frac=0.6),
    "hubs": dict(n=500, E=3000, hubs=3, hub_deg=1000, src_hubs=2),
    "sparse": dict(n=5000, E=40),
}

# in- and out-degrees at the 128-edge chunk boundaries, empty rows and rows far longer than a chunk, in both plans
DEGREES = [0, 1, 127, 128, 129, 255, 256, 257, 1000]


def degree_graph(rng):
    """node i has in-degree DEGREES[i] and out-degree DEGREES[perm[i]] exactly; filler nodes have neither"""
    n = len(DEGREES) + 20
    perm = rng.permutation(len(DEGREES))
    t = np.repeat(np.arange(1, len(DEGREES) + 1), DEGREES)
    s = np.repeat(np.arange(1, len(DEGREES) + 1), [DEGREES[j] for j in perm])
    s = s[rng.permutation(len(s))]
    q = rng.permutation(len(s))
    return s[q].astype(np.int64), t[q].astype(np.int64), n


def _graph_case(oracle, key):
    """(s, t, n) in 1-based COO for a case key: '<name>+loops' / '<name>' (without self loops) / 'degrees' / 'chunk32'
    (`hubs` with self loops, planned with 32-edge chunks)"""
    if key == "degrees":
        return degree_graph(np.random.default_rng(99))
    name = "hubs" if key == "chunk32" else key.split("+")[0]
    rng = np.random.default_rng(list(GRAPHS).index(name))
    kw = GRAPHS[name]
    s, t = make_graph(rng, **kw)
    if key.endswith("+loops") or key == "chunk32":
        s, t = oracle.add_self_loops(s, t, kw["n"])
    return s, t, kw["n"]


GRAPH_KEYS = [k + sfx for k in GRAPHS for sfx in ("+loops", "")] + ["degrees", "chunk32"]


def test_degree_graph_hits_the_degrees():
    s, t, n = degree_graph(np.random.default_rng(99))
    din, dout = np.bincount(t - 1, minlength=n), np.bincount(s - 1, minlength=n)
    assert sorted(din[:len(DEGREES)]) == sorted(DEGREES) and sorted(dout[:len(DEGREES)]) == sorted(DEGREES)
    assert not din[len(DEGREES):].any() and not dout[len(DEGREES):].any()


# ----------------------------------------------------------------------------------------- the C entries, all branches
CH_PAIRS = [
    (1, 4), (2, 3), (2, 32), (2, 64),            # scalar path, K = 1 / 1 / 2 / 4 (C in {1, 2})
    (128, 3), (64, 16), (4, 128),                # vec4 chunk kernels with grid.y > 1 (D = 384, 1024; H > 64 at D = 512)
    (32, 4), (64, 4), (64, 8),                   # lean kernels at D = 128 / 256 / 512
    (4, 64), (8, 64),                            # lean at H = 64: the largest dynamic shared memory of the pullback
    (128, 1), (128, 4),                          # lean with C = 128 (one head per warp slice)
]


def _run_c_abi(gnn, oracle, s, t, n, Cc, H, slope, *, logit_scale=1.0, a_zero=False, misalign=False, chunk=None,
               record=None):
    """forward + pullback through the C entries against the oracle; returns (out, Wx, del, der64)"""
    lib = gnn._lib.lib
    E = len(s)
    rng = np.random.default_rng(Cc * 1000 + H * 10 + int(slope * 10))
    Wx = rng.standard_normal((n, H, Cc)).astype(np.float32)
    el = (rng.standard_normal((n, H)) * logit_scale).astype(np.float32)
    er = (rng.standard_normal((n, H)) * logit_scale).astype(np.float32)
    if a_zero:
        el[:] = 0.0
        er[:] = 0.0
    dout = rng.standard_normal((n, H, Cc)).astype(np.float32)
    dev = lambda a: torch.as_tensor(a).cuda().contiguous()
    if misalign:       # a one-float offset view: the fused entries take the scalar path
        buf = torch.empty(n * H * Cc + 1, device="cuda")
        Wx_d = buf[1:].view(n, H, Cc)
        Wx_d.copy_(torch.as_tensor(Wx))
        assert Wx_d.data_ptr() % 16 != 0
    else:
        Wx_d = dev(Wx)
    el_d, er_d, do_d = dev(el), dev(er), dev(dout)
    if chunk is not None:
        gnn._lib.check(lib.gnnb_set_chunk_edges(chunk))
    try:
        g = gnn.GNNGraph(s, t, num_nodes=n).to("cuda")
        p = g.plan()
        out = torch.empty(n, H, Cc, device="cuda"); alpha = torch.empty(E, H, device="cuda")
        smax = torch.empty(n, H, device="cuda"); ssum = torch.empty(n, H, device="cuda")
        gnn._lib.check(lib.gnnb_gat_aggregate(p.h, Wx_d.data_ptr(), el_d.data_ptr(), er_d.data_ptr(), Cc, H, slope,
                                              out.data_ptr(), alpha.data_ptr(), smax.data_ptr(), ssum.data_ptr(), None))
        res = []
        for _ in range(2):            # the pullback is deterministic: two runs, same bits
            dWx = torch.full((n, H, Cc), float("nan"), device="cuda")
            del_ = torch.full((n, H), float("nan"), device="cuda"); der = torch.full((n, H), float("nan"), device="cuda")
            gnn._lib.check(lib.gnnb_gat_aggregate_bwd(p.h, Wx_d.data_ptr(), el_d.data_ptr(), er_d.data_ptr(), smax.data_ptr(),
                                                      ssum.data_ptr(), out.data_ptr(), do_d.data_ptr(), Cc, H, slope,
                                                      dWx.data_ptr(), del_.data_ptr(), der.data_ptr(), None))
            res.append((dWx, del_, der))
        torch.cuda.synchronize()
    finally:
        if chunk is not None:
            lib.gnnb_set_chunk_edges(128)          # the library default (csrc/plan.cu)
    for a_, b_ in zip(*res):
        assert torch.equal(a_, b_)
    dWx, del_, der = (x.cpu().numpy() for x in res[0])
    f64 = lambda a: a.astype(np.float64)
    r64 = oracle.gat_aggregate_bwd(s, t, n, f64(Wx), f64(dout), slope, el=f64(el), er=f64(er))
    r32 = oracle.gat_aggregate_bwd(s, t, n, Wx, dout, slope, el=el, er=er)
    dWx64, del64, der64, alpha64 = r64
    out64 = np.stack([oracle.propagate_unfused("+", s, t, n, f64(Wx[:, h]), w=alpha64[:, h]) for h in range(H)], axis=1)
    check_plain("out", out.cpu().numpy(), out64)
    check_plain("alpha", alpha.cpu().numpy(), alpha64)
    check_plain("dWx", dWx, dWx64)
    if not a_zero:           # with a = 0 every logit of a row ties and del is 0 in exact arithmetic (checked by the caller)
        check_cancelling("del", del_, del64, r32[1], record)
    check_cancelling("der", der, der64, r32[2], record)
    return out.cpu().numpy(), Wx, del_, der64


@pytest.mark.parametrize("slope", [0.2, 0.0])
@pytest.mark.parametrize("Cc,H", CH_PAIRS)
@pytest.mark.parametrize("gkey", GRAPH_KEYS)
def test_gat_aggregate_bwd_against_fp64(gnn, oracle, record_property, gkey, Cc, H, slope):
    s, t, n = _graph_case(oracle, gkey)
    _run_c_abi(gnn, oracle, s, t, n, Cc, H, slope, chunk=32 if gkey == "chunk32" else None, record=record_property)


@pytest.mark.parametrize("Cc,H", [(8, 16), (4, 8), (1, 4)])
@pytest.mark.parametrize("gkey", ["hubs+loops", "degrees"])
def test_gat_aggregate_bwd_misaligned_wx(gnn, oracle, record_property, gkey, Cc, H):
    """Wx one float off 16 B: the scalar kernels serve C = 8 at D <= 128"""
    s, t, n = _graph_case(oracle, gkey)
    _run_c_abi(gnn, oracle, s, t, n, Cc, H, 0.2, misalign=True, record=record_property)


@pytest.mark.parametrize("Cc,H", [(64, 8), (4, 64), (128, 3), (2, 3)])
@pytest.mark.parametrize("gkey", ["hubs+loops", "hubs"])
def test_gat_aggregate_bwd_large_logits(gnn, oracle, record_property, gkey, Cc, H):
    """logits near ±80 (el, er × 50): exp without the max shift would overflow fp32.  At this scale a short row's softmax
    is one-hot, and del_i = Σ α (dα − T) vanishes to rounding: on `small` or `degrees` (whose rows draw on 9 sources only)
    the fp32 formula's own error e32 exceeds 1e-4, a quantity no relative bound applies to.  The hub graphs keep
    e32 ≈ 2e-5."""
    s, t, n = _graph_case(oracle, gkey)
    _run_c_abi(gnn, oracle, s, t, n, Cc, H, 0.2, logit_scale=50.0, record=record_property)


@pytest.mark.parametrize("Cc,H", [(64, 8), (128, 3), (2, 3)])
@pytest.mark.parametrize("gkey", ["hubs+loops", "empty_rows"])
def test_gat_zero_attention_is_the_mean(gnn, oracle, gkey, Cc, H):
    """a = 0 (el = er = 0): α = 1 / in-degree, so out is propagate(copy_xj, mean) of Wx; and del = Σ_k α (dα_k − mean dα)
    slope = 0 exactly, so it must vanish to rounding on the scale of der (the same dz terms, summed by source)"""
    s, t, n = _graph_case(oracle, gkey)
    out, Wx, del_, der64 = _run_c_abi(gnn, oracle, s, t, n, Cc, H, 0.2, a_zero=True)
    assert np.linalg.norm(del_) <= BAR * np.linalg.norm(der64)
    mean = oracle.propagate_unfused("mean", s, t, n, Wx.reshape(n, H * Cc).astype(np.float64)).reshape(n, H, Cc)
    assert rel(out, mean) < 2e-6


# ------------------------------------------------------------------------------------------------ the logit-term gate
def _logit_entries_accept(gnn, Cc, H):
    lib = gnn._lib.lib
    N = 3
    Wx = torch.randn(N, H, Cc, device="cuda")
    a = torch.randn(H, 2 * Cc, device="cuda")
    el, er = torch.zeros(N, H, device="cuda"), torch.zeros(N, H, device="cuda")
    dWx = torch.zeros_like(Wx); da = torch.empty(H, 2 * Cc, device="cuda")
    f = lib.gnnb_gat_logit_terms(Wx.data_ptr(), a.data_ptr(), N, Cc, H, el.data_ptr(), er.data_ptr(), None)
    b = lib.gnnb_gat_logit_terms_bwd(Wx.data_ptr(), a.data_ptr(), el.data_ptr(), er.data_ptr(), N, Cc, H, dWx.data_ptr(),
                                     da.data_ptr(), None)
    torch.cuda.synchronize()
    for st in (f, b):
        assert st in (gnn._lib.OK, gnn._lib.EUNSUPPORTED), st
    return f == gnn._lib.OK and b == gnn._lib.OK


@pytest.mark.parametrize("Cc", [4, 8, 16, 32, 64, 128])
def test_gat_logit_gate_matches_the_c_entries(gnn, Cc):
    """gat_logit_fusable(C, H) holds exactly when both logit-term entries accept the shape: the layer never routes a shape
    to the fused forward whose pullback then refuses it, and never sends a shape both entries cover to the eager path"""
    from gnnb200.layers import gat_logit_fusable
    G = Cc // 4
    edges = {1024 // Cc, 4096 // Cc, 8 * 32 // G, 32 // G, 200 * 1024 // (64 * Cc)}
    Hs = sorted({h for e in edges for h in (e - 1, e, e + 1) if h >= 1} | set(range(1, 10)))
    bad = [(Cc, H, gat_logit_fusable(Cc, H)) for H in Hs if gat_logit_fusable(Cc, H) != _logit_entries_accept(gnn, Cc, H)]
    assert not bad, f"(C, H, python gate) disagreeing with the C entries: {bad}"


# -------------------------------------------------------------------------------------------- the layer, end to end
def gat_conv_torch(s, t, n, x, W, a, b, slope, concat, mask):
    """gat_conv (GNNlib/src/layers/conv.jl:112-150) in plain torch on the CPU, in x's dtype: W·x, per-edge logits
    a·vcat(Wxi, Wxj), leakyrelu, neighbourhood softmax (scatter_reduce max, exp, index_add), α-weighted index_add,
    mean over heads if !concat, bias, σ.  σ = relu is applied as the mask of the GPU forward (None: identity), so a sign
    flip at 0 is not counted as backward error.  (s, t) already hold the self loops; x is (n, din) rows."""
    Cc, H = a.shape[0] // 2, a.shape[1]
    s0, t0 = torch.as_tensor(s - 1), torch.as_tensor(t - 1)
    Wx = (x @ W.t()).reshape(n, H, Cc)
    Wi, Wj = Wx[t0], Wx[s0]
    z = (Wi * a[:Cc].t()).sum(-1) + (Wj * a[Cc:].t()).sum(-1)
    u = torch.nn.functional.leaky_relu(z, slope)
    m = torch.full((n, H), -torch.inf, dtype=u.dtype).scatter_reduce(0, t0[:, None].expand(-1, H), u.detach(), "amax")
    ex = torch.exp(u - m[t0])
    den = torch.zeros(n, H, dtype=u.dtype).index_add(0, t0, ex)
    alpha = ex / den[t0]
    out = torch.zeros(n, H, Cc, dtype=u.dtype).index_add(0, t0, alpha[:, :, None] * Wj)
    out = out.reshape(n, H * Cc) if concat else out.mean(1)
    pre = out + b
    return pre if mask is None else pre * mask


LAYER_SHAPES = [
    (16, 64, 2),      # fused lean (D = 128), fused logit terms
    (32, 32, 4),      # fused lean (D = 128), 4 heads
    (8, 16, 3),       # fused chunk kernels (D = 48), fused logit terms
    (8, 128, 3),      # fused chunk kernels with grid.y = 3, fused logit terms
    (5, 2, 3),        # scalar kernels, logit halves by broadcast (C % 4 != 0)
    (16, 128, 16),    # C = 128, 16 heads: the fused logit pullback refuses 16 passes -> broadcast halves
    (16, 64, 32),     # C = 64, 32 heads: likewise
    (6, 4, 20),       # C = 4, 20 heads: one pass of 32 heads, fused logit terms
    (3, 5, 2),        # not fusable: the reference's composition on the generic kernels
]


@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("concat", [True, False])
@pytest.mark.parametrize("din,chout,heads", LAYER_SHAPES)
@pytest.mark.parametrize("gname", ["small", "hubs"])
def test_gat_conv_backward_against_fp64(gnn, oracle, record_property, gname, din, chout, heads, concat, relu):
    s, t, n = _graph_case(oracle, gname)
    torch.manual_seed(din * 100 + chout + heads)
    from gnnb200.layers import identity
    l = gnn.GATConv(din, chout, torch.relu if relu else identity, heads=heads, concat=concat, device="cuda")
    with torch.no_grad():
        l.bias.normal_()
    rng = np.random.default_rng(7)
    x = rng.standard_normal((n, din)).astype(np.float32)
    g = gnn.GNNGraph(s, t, num_nodes=n).to("cuda")
    xt = gnn.unrows(torch.as_tensor(x).cuda()).requires_grad_(True)
    y = l(g, xt)
    dy = rng.standard_normal(tuple(reversed(y.shape))).astype(np.float32)    # rows (n, Dout)
    y.backward(gnn.unrows(torch.as_tensor(dy).cuda()))
    yg = gnn.rows(y.detach()).cpu().numpy()
    s2, t2 = oracle.add_self_loops(s, t, n)
    params = [l.dense_x.weight, l.a, l.bias]
    mask = torch.as_tensor(yg > 0) if relu else None

    def ref(dtype):
        leaves = [torch.as_tensor(x, dtype=dtype).requires_grad_(True)] + \
                 [p.detach().cpu().to(dtype).requires_grad_(True) for p in params]
        yr = gat_conv_torch(s2, t2, n, leaves[0], *leaves[1:], float(l.negative_slope), concat,
                            None if mask is None else mask.to(dtype))
        return yr.detach().numpy(), torch.autograd.grad(yr, leaves, torch.as_tensor(dy, dtype=dtype))

    y64, (dx64, dW64, da64, db64) = ref(torch.float64)
    _, (_, _, da32, _) = ref(torch.float32)
    check_plain("y", yg, y64)
    check_plain("dx", gnn.rows(xt.grad).cpu().numpy(), dx64.numpy())
    check_plain("dW", l.dense_x.weight.grad.cpu().numpy(), dW64.numpy())
    check_plain("db", l.bias.grad.cpu().numpy(), db64.numpy())
    check_cancelling("da", l.a.grad.cpu().numpy(), da64.numpy(), da32.numpy(), record_property)


# --------------------------------------------------------------------------------------------------- config-3 scale
def test_at_scale_gat_backward_against_fp64(gnn, oracle, record_property):
    """GATConv 512 -> 8 heads x 64, relu, on RMAT N = 100 k, E = 1 M (config-3 shape): the layer's dx, dW, da, db and the C
    entry's dWx, del, der against fp64 built from orc_gat_aggregate_bwd, the linear logit chain, the dense part and the bias"""
    n, E, H, Cc = 100_000, 1_000_000, 8, 64
    D = H * Cc
    s, t = oracle.rmat(n, E, 17)
    g = gnn.GNNGraph(s, t, num_nodes=n).cuda()
    rng = np.random.default_rng(4)
    x = rng.standard_normal((n, D)).astype(np.float32)
    dy = rng.standard_normal((n, D)).astype(np.float32)
    torch.manual_seed(0)
    layer = gnn.GATConv(D, Cc, torch.relu, heads=H, device="cuda")
    with torch.no_grad():
        layer.bias.normal_()
    xt = gnn.unrows(torch.as_tensor(x).cuda()).requires_grad_(True)
    y = layer(g, xt)
    y.backward(gnn.unrows(torch.as_tensor(dy).cuda()))
    yg = gnn.rows(y.detach()).cpu().numpy()
    got = dict(dx=gnn.rows(xt.grad).cpu().numpy(), dW=layer.dense_x.weight.grad.cpu().numpy(),
               da=layer.a.grad.cpu().numpy(), db=layer.bias.grad.cpu().numpy())
    del y, xt
    s2, t2 = oracle.add_self_loops(s, t, n)
    Wd32 = layer.dense_x.weight.detach().cpu().numpy()
    a32 = np.ascontiguousarray(layer.a.detach().cpu().numpy().T)                    # rows (H, 2C)

    def layer_grads(dtype, only_da=False):
        """the layer's pullback in `dtype` on the CPU; relu' on the GPU forward's mask"""
        Wd, a, xx = Wd32.astype(dtype), a32.astype(dtype), x.astype(dtype)
        Wx = (xx @ Wd.T).reshape(n, H, Cc)
        dpre = dy.astype(dtype) * (yg > 0)
        dWx, del_, der, _ = oracle.gat_aggregate_bwd(s2, t2, n, Wx, dpre.reshape(n, H, Cc), 0.2, a=a)
        dWx = dWx + del_[:, :, None] * a[None, :, :Cc] + der[:, :, None] * a[None, :, Cc:]
        da = np.concatenate([np.einsum("nh,nhc->hc", del_, Wx), np.einsum("nh,nhc->hc", der, Wx)], axis=1).T   # (2C, H)
        if only_da:
            return dict(da=da)
        dWx = dWx.reshape(n, D)
        return dict(dx=dWx @ Wd, dW=dWx.T @ xx, da=da, db=dpre.sum(0))

    r64 = layer_grads(np.float64)
    for k in ("dx", "dW", "db"):
        check_plain(k, got[k], r64[k])
    da32 = layer_grads(np.float32, only_da=True)["da"]
    check_cancelling("da", got["da"], r64["da"], da32, record_property)
    del r64, da32
    # the C entry on the layer's own projection, with a fresh upstream gradient
    Wx = (x @ Wd32.T).reshape(n, H, Cc)
    el, er = oracle.gat_logit_halves(Wx, a32)
    dout = rng.standard_normal((n, H, Cc)).astype(np.float32)
    g2 = gnn.add_self_loops(g)
    p = g2.plan()
    lib = gnn._lib.lib
    dev = lambda v: torch.as_tensor(np.ascontiguousarray(v)).cuda()
    Wx_d, el_d, er_d, do_d = dev(Wx), dev(el), dev(er), dev(dout)
    out = torch.empty_like(Wx_d); smax = torch.empty(n, H, device="cuda"); ssum = torch.empty(n, H, device="cuda")
    dWx = torch.empty_like(Wx_d); del_ = torch.empty(n, H, device="cuda"); der = torch.empty(n, H, device="cuda")
    gnn._lib.check(lib.gnnb_gat_aggregate(p.h, Wx_d.data_ptr(), el_d.data_ptr(), er_d.data_ptr(), Cc, H, 0.2, out.data_ptr(),
                                          None, smax.data_ptr(), ssum.data_ptr(), None))
    gnn._lib.check(lib.gnnb_gat_aggregate_bwd(p.h, Wx_d.data_ptr(), el_d.data_ptr(), er_d.data_ptr(), smax.data_ptr(),
                                              ssum.data_ptr(), out.data_ptr(), do_d.data_ptr(), Cc, H, 0.2, dWx.data_ptr(),
                                              del_.data_ptr(), der.data_ptr(), None))
    f64 = lambda v: v.astype(np.float64)
    r64 = oracle.gat_aggregate_bwd(s2, t2, n, f64(Wx), f64(dout), 0.2, el=f64(el), er=f64(er))
    r32 = oracle.gat_aggregate_bwd(s2, t2, n, Wx, dout, 0.2, el=el, er=er)
    check_plain("dWx", dWx.cpu().numpy(), r64[0])
    check_cancelling("del", del_.cpu().numpy(), r64[1], r32[1], record_property)
    check_cancelling("der", der.cpu().numpy(), r64[2], r32[2], record_property)
