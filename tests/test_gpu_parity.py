"""Parity of the CUDA path (through the Python mirror -> C ABI -> sm_100a kernels) with the CPU oracle.

Bar (BASELINE.json north_star): bit-exact for index arithmetic; fp32 aggregations within 1e-5 relative
(normwise, the reference's `isapprox` semantics, GNNlib/test/test_module.jl:75-151) of the fp64 oracle — the
tests below use the tighter 2e-6 — and bit-exact against the fp32 oracle wherever a row is reduced by a single
group in COO order (rows <= chunk edges, sum/max/min).
"""
import ctypes as C
import operator

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 2e-6


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    fin = np.isfinite(b)
    assert (np.isfinite(a) == fin).all() and (a[~fin] == b[~fin]).all()
    return np.linalg.norm(a[fin] - b[fin]) / max(np.linalg.norm(b[fin]), 1e-30)


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


def jl(x_rows, dev="cuda"):
    """numpy rows (N, ...) -> Julia-shaped column-major device tensor (..., N)"""
    import gnnb200
    return gnnb200.unrows(torch.as_tensor(np.ascontiguousarray(x_rows), dtype=torch.float32).to(dev))


def np_rows(x_jl):
    import gnnb200
    return gnnb200.rows(x_jl.detach()).cpu().numpy()


GRAPHS = {
    "small": dict(n=37, E=150),
    "empty_rows": dict(n=200, E=300, empty_frac=0.6),
    "hubs": dict(n=500, E=3000, hubs=3, hub_deg=1000, src_hubs=2),   # rows far longer than the 128-edge chunk, both plans
    "sparse": dict(n=5000, E=40),                          # rows >> edges: row-parallel empty fill path
}


@pytest.fixture(scope="module", params=list(GRAPHS))
def graph(request, gnn):
    rng = np.random.default_rng(list(GRAPHS).index(request.param))
    kw = GRAPHS[request.param]
    s, t = make_graph(rng, **kw)
    g = gnn.GNNGraph(s, t, num_nodes=kw["n"]).to("cuda")
    return request.param, s, t, kw["n"], g


@pytest.fixture(scope="module", params=[k for k in GRAPHS if k != "sparse"])
def graph_with_edges(request, gnn):
    """the graphs whose targets mostly have in-edges (GAT always runs with self loops; `sparse` adds nothing there)"""
    rng = np.random.default_rng(list(GRAPHS).index(request.param))
    kw = GRAPHS[request.param]
    s, t = make_graph(rng, **kw)
    return request.param, s, t, kw["n"], gnn.GNNGraph(s, t, num_nodes=kw["n"]).to("cuda")


@pytest.fixture(scope="module")
def small_graph(gnn):
    rng = np.random.default_rng(0)
    kw = GRAPHS["small"]
    s, t = make_graph(rng, **kw)
    return "small", s, t, kw["n"], gnn.GNNGraph(s, t, num_nodes=kw["n"]).to("cuda")


# ------------------------------------------------------------------------------------------ index work
def test_csr_bit_exact(graph, oracle, gnn):
    _, s, t, n, g = graph
    p = g.plan()
    E = len(s)
    for transposed, key, other in ((0, t, s), (1, s, t)):
        rowptr = np.empty(n + 1, np.int32)
        col = np.empty(E, np.int32)
        eid = np.empty(E, np.int32)
        gnn._lib.check(gnn._lib.lib.gnnb_graph_csr(p.h, transposed, rowptr.ctypes.data, col.ctypes.data,
                                                   eid.ctypes.data, None))
        r0, c0, p0 = oracle.csr(key, other, n)
        assert (rowptr == r0).all() and (col == c0).all() and (eid == p0).all()
    # rowptr differences == degree(g; dir=:in) exactly
    assert (gnn.degree(g, dir="in").cpu().numpy() == oracle.degree(s, t, n, "in").astype(np.int64)).all()
    assert (gnn.degree(g, dir="out").cpu().numpy() == oracle.degree(s, t, n, "out").astype(np.int64)).all()
    assert (gnn.degree(g, dir="both").cpu().numpy() == oracle.degree(s, t, n, "both").astype(np.int64)).all()


def test_self_loop_plan_bit_exact(graph, oracle, gnn):
    _, s, t, n, g = graph
    g.plan()
    gnn._lib.check(gnn._lib.lib.gnnb_graph_csr(g.plan().h, 1, None, None, None, None))   # build by_src too
    g2 = gnn.add_self_loops(g)
    s2, t2 = oracle.add_self_loops(s, t, n)
    assert (g2.s.cpu().numpy() == s2).all() and (g2.t.cpu().numpy() == t2).all()
    E2 = len(s2)
    for transposed, key, other in ((0, t2, s2), (1, s2, t2)):
        rowptr = np.empty(n + 1, np.int32); col = np.empty(E2, np.int32); eid = np.empty(E2, np.int32)
        gnn._lib.check(gnn._lib.lib.gnnb_graph_csr(g2.plan().h, transposed, rowptr.ctypes.data, col.ctypes.data,
                                                   eid.ctypes.data, None))
        r0, c0, p0 = oracle.csr(key, other, n)
        assert (rowptr == r0).all() and (col == c0).all() and (eid == p0).all()


def test_index_inputs_and_validation(gnn, oracle):
    s = np.array([1, 1, 2, 3]); t = np.array([2, 2, 2, 4])
    ref = oracle.csr(t, s, 4)
    for dt in (torch.int64, torch.int32):
        for dev in ("cpu", "cuda"):
            g = gnn.GNNGraph(torch.as_tensor(s, dtype=dt, device=dev), torch.as_tensor(t, dtype=dt, device=dev))
            rowptr = np.empty(5, np.int32); col = np.empty(4, np.int32); eid = np.empty(4, np.int32)
            gnn._lib.check(gnn._lib.lib.gnnb_graph_csr(g.plan().h, 0, rowptr.ctypes.data, col.ctypes.data,
                                                       eid.ctypes.data, None))
            assert (rowptr == ref[0]).all() and (col == ref[1]).all() and (eid == ref[2]).all()
    # 1 <= idx <= num_nodes (GNNGraphs/src/convert.jl:49-54) -> AssertionError
    for bad_s, bad_t in (([0, 1], [1, 2]), ([1, 2], [1, 5])):
        with pytest.raises(AssertionError):
            gnn.GNNGraph(bad_s, bad_t, num_nodes=4).plan()


def test_degree_golden(gnn):
    # GNNGraphs/test/query.jl:49-58,71-87 on the GPU
    s, t = [1, 1, 2, 3], [2, 2, 2, 4]
    g = gnn.GNNGraph(s, t).cuda()
    assert gnn.degree(g).tolist() == [2, 1, 1, 0] == gnn.degree(g, dir="out").tolist()
    assert gnn.degree(g, dir="in").tolist() == [0, 3, 0, 1]
    assert gnn.degree(g, dir="both").tolist() == [2, 4, 1, 1]
    assert gnn.degree(g, torch.float32).dtype == torch.float32
    w = torch.tensor([0.1, 2.1, 1.2, 1.0])
    gw = gnn.GNNGraph((s, t, w)).cuda()
    np.testing.assert_allclose(gnn.degree(gw).cpu(), [2.2, 1.2, 1.0, 0.0], rtol=1e-6)
    assert gnn.degree(gw, edge_weight=False).tolist() == [2, 1, 1, 0]
    np.testing.assert_allclose(gnn.degree(gw, edge_weight=2 * w.cuda()).cpu(), [4.4, 2.4, 2.0, 0.0], rtol=1e-6)


def test_rmat_gpu_equals_cpu(gnn, oracle):
    for n, E in ((1000, 5000), (100000, 300000)):
        g = gnn.rmat_graph(n, E, 17)
        s, t = oracle.rmat(n, E, 17)
        assert (g.s.cpu().numpy() == s).all() and (g.t.cpu().numpy() == t).all()


# ---------------------------------------------------------------------------------------- fused propagate
def _check_propagate_copy_xj(graph, oracle, gnn, D, aggr):
    name, s, t, n, g = graph
    rng = np.random.default_rng(D)
    x = rng.standard_normal((n, D)).astype(np.float32)
    got = np_rows(gnn.propagate(gnn.copy_xj, g, aggr, xj=jl(x)))
    ref64 = oracle.propagate_unfused(aggr, s, t, n, x.astype(np.float64))
    assert rel(got, ref64) < TOL
    if aggr in ("max", "min"):       # order independent: bit-exact
        assert (got == oracle.propagate_unfused(aggr, s, t, n, x)).all()
    elif name in ("small", "empty_rows", "sparse"):   # rows <= chunk: same summation order as NNlib's CPU scatter
        assert (got == oracle.propagate_unfused(aggr, s, t, n, x)).all()


@pytest.mark.parametrize("D", [1, 3, 7, 10, 16, 20, 64, 128, 132, 256, 300])
@pytest.mark.parametrize("aggr", ["+", "mean", "max", "min"])
def test_propagate_copy_xj(graph, oracle, gnn, D, aggr):
    _check_propagate_copy_xj(graph, oracle, gnn, D, aggr)


@pytest.mark.parametrize("D", [512, 1433])
@pytest.mark.parametrize("aggr", ["+", "mean", "max", "min"])
def test_propagate_copy_xj_wide_rows(small_graph, oracle, gnn, D, aggr):
    _check_propagate_copy_xj(small_graph, oracle, gnn, D, aggr)


@pytest.mark.parametrize("D", [1, 5, 16, 128, 260])
@pytest.mark.parametrize("aggr", ["+", "mean", "max", "min"])
@pytest.mark.parametrize("fn", ["w_mul_xj", "e_mul_xj"])
def test_propagate_weighted(graph, oracle, gnn, D, aggr, fn):
    name, s, t, n, g = graph
    rng = np.random.default_rng(D + 1)
    x = rng.standard_normal((n, D)).astype(np.float32)
    w = rng.random(len(s)).astype(np.float32) - 0.3
    wt = torch.as_tensor(w).cuda()
    if fn == "w_mul_xj":
        got = gnn.propagate(gnn.w_mul_xj, gnn.set_edge_weight(g, wt), aggr, xj=jl(x))
    else:
        got = gnn.propagate(gnn.e_mul_xj, g, aggr, xj=jl(x), e=wt)
    got = np_rows(got)
    ref64 = oracle.propagate_unfused(aggr, s, t, n, x.astype(np.float64), w.astype(np.float64))
    assert rel(got, ref64) < TOL
    if aggr != "mean" and name != "hubs":
        assert (got == oracle.propagate_unfused(aggr, s, t, n, x, w)).all()


def test_propagate_matches_dense_adjacency(gnn, oracle):
    # GNNlib/test/msgpass.jl:69-116 on the GPU: ≈ X * Adj and ≈ X * A
    n = 128
    rng = np.random.default_rng(0)
    A = (rng.random((n, n)) < 0.1) * rng.random((n, n))
    g = gnn.GNNGraph(A.astype(np.float32)).cuda()
    X = rng.random((10, n)).astype(np.float32)
    Xd = gnn.colmajor(torch.as_tensor(X).cuda())
    Adj = (A > 0).astype(np.float64)
    y = gnn.propagate(gnn.copy_xj, g, operator.add, xj=Xd).cpu().numpy()
    assert rel(y, X.astype(np.float64) @ Adj) < TOL
    y = gnn.propagate(lambda xi, xj, e: xj, g, operator.add, xj=Xd).cpu().numpy()       # unfused path
    assert rel(y, X.astype(np.float64) @ Adj) < TOL
    ref = X.astype(np.float64) @ A.astype(np.float32).astype(np.float64)
    y = gnn.propagate(gnn.w_mul_xj, g, operator.add, xj=Xd).cpu().numpy()
    assert rel(y, ref) < TOL
    y = gnn.propagate(gnn.e_mul_xj, g, operator.add, xj=Xd, e=g.w).cpu().numpy()
    assert rel(y, ref) < TOL
    y = gnn.propagate(lambda xi, xj, e: e.reshape(1, -1) * xj, g, operator.add, xj=Xd, e=g.w).cpu().numpy()
    assert rel(y, ref) < TOL


def test_propagate_shapes_isolated_nodes_and_empty_graph(gnn):
    # GNNlib/test/msgpass.jl:10-26
    g1 = gnn.GNNGraph(list(range(1, 6)), list(range(1, 6)), num_nodes=6).cuda()
    x1 = gnn.colmajor(torch.rand(1, 6).cuda())
    y1 = gnn.propagate(lambda xi, xj, e: xj, g1, operator.add, xj=x1)
    assert y1.shape == (1, 6) and y1[0, 5] == 0
    y1 = gnn.propagate(gnn.copy_xj, g1, operator.add, xj=x1)
    assert y1.shape == (1, 6) and y1[0, 5] == 0 and torch.equal(y1[:, :5], x1[:, :5])
    g0 = gnn.GNNGraph(torch.empty(0, dtype=torch.int64), torch.empty(0, dtype=torch.int64), num_nodes=5).cuda()
    x0 = gnn.colmajor(torch.rand(4, 5).cuda())
    assert (gnn.propagate(gnn.copy_xj, g0, operator.add, xj=x0) == 0).all()
    assert (gnn.propagate(gnn.copy_xj, g0, max, xj=x0) == -float("inf")).all()
    assert (gnn.propagate(gnn.copy_xj, g0, min, xj=x0) == float("inf")).all()
    # 3-D features (C, H, N): last dimension is the node dimension
    x3 = gnn.jl_randn(3, 2, 6, device="cuda")
    y3 = gnn.propagate(gnn.copy_xj, g1, gnn.mean, xj=x3)
    assert y3.shape == (3, 2, 6) and torch.equal(y3[..., :5], x3[..., :5])


def test_generic_message_functions(graph, oracle, gnn):
    # apply_edges with NamedTuple-like containers, xi/xj/e all used (GNNlib/test/msgpass.jl:28-53)
    _, s, t, n, g = graph
    rng = np.random.default_rng(7)
    x = rng.standard_normal((n, 6)).astype(np.float32)
    e = rng.standard_normal((len(s), 6)).astype(np.float32)
    m = gnn.apply_edges(lambda xi, xj, e: {"a": xi["u"] - xj["u"], "b": gnn.xi_dot_xj(xi["u"], xj["u"], None) + e[:1]},
                        g, xi={"u": jl(x)}, xj={"u": jl(x), "v": jl(2 * x)}, e=jl(e))
    a_ref = x[t - 1] - x[s - 1]
    b_ref = (x[t - 1] * x[s - 1]).sum(1, keepdims=True) + e[:, :1]
    assert rel(np_rows(m["a"]), a_ref) < TOL and rel(np_rows(m["b"]), b_ref) < TOL
    out = gnn.aggregate_neighbors(g, gnn.mean, m)
    assert rel(np_rows(out["a"]), oracle.scatter("mean", a_ref.astype(np.float64), t, n)) < TOL
    assert rel(np_rows(out["b"]), oracle.scatter("mean", b_ref.astype(np.float64), t, n)) < TOL
    assert gnn.aggregate_neighbors(g, operator.add, None) is None
    # gather / scatter primitives, bit-exact data movement
    xe = gnn.apply_edges(gnn.copy_xi, g, xi=jl(x))
    assert (np_rows(xe) == x[t - 1]).all()
    for aggr in ("+", "max", "min"):
        got = np_rows(gnn.aggregate_neighbors(g, aggr, jl(e)))
        assert rel(got, oracle.scatter(aggr, e.astype(np.float64), t, n)) < TOL


# ------------------------------------------------------------------------------------------- pullbacks
@pytest.mark.parametrize("aggr", ["+", "mean", "max", "min"])
@pytest.mark.parametrize("D", [3, 16, 128, 256, 512])
def test_propagate_gradients(graph, oracle, gnn, aggr, D):
    """Zygote/NNlib pullbacks restated through the oracle's gather/scatter (SURVEY.md §9)."""
    name, s, t, n, g = graph
    rng = np.random.default_rng(11)
    x = rng.standard_normal((n, D)).astype(np.float32)
    if aggr in ("max", "min"):   # create exact ties
        x = np.round(x * 2) / 2
    dout = rng.standard_normal((n, D)).astype(np.float32)
    w = (rng.random(len(s)) + 0.5).astype(np.float32)
    for weighted in (False, True):
        xt = jl(x).requires_grad_(True)
        wt = torch.as_tensor(w).cuda().requires_grad_(True)
        if weighted:
            y = gnn.propagate(gnn.e_mul_xj, g, aggr, xj=xt, e=wt)
        else:
            y = gnn.propagate(gnn.copy_xj, g, aggr, xj=xt)
        if aggr in ("max", "min"):
            dd = np.where(np.isfinite(np_rows(y)), dout, 0).astype(np.float32)   # no gradient through ∓Inf rows
        else:
            dd = dout
        if weighted and aggr in ("max", "min"):
            wt2 = wt.detach()   # dw for max/min runs through the generic path only
            y = gnn.propagate(gnn.e_mul_xj, g, aggr, xj=xt, e=wt2)
        y.backward(jl(dd))
        # oracle: m = w .* gather(x, s); out = scatter(aggr, m, t)
        x64, w64, d64 = x.astype(np.float64), w.astype(np.float64), dd.astype(np.float64)
        m = oracle.gather(x64, s) * (w64[:, None] if weighted else 1.0)
        dg = oracle.gather(d64, t)
        if aggr == "mean":
            cnt = np.maximum(oracle.degree(s, t, n, "in", None, np.float64), 1)
            dm = dg / cnt[t - 1][:, None]
        elif aggr in ("max", "min"):
            out = oracle.scatter(aggr, m, t, n)
            dm = dg * (m == oracle.gather(out, t))
        else:
            dm = dg
        dx_ref = oracle.scatter("+", dm * (w64[:, None] if weighted else 1.0), s, n)
        assert rel(np_rows(xt.grad), dx_ref) < 5e-6
        if weighted and aggr in ("+", "mean"):
            dw_ref = (dm * oracle.gather(x64, s)).sum(1)
            assert rel(wt.grad.cpu().numpy(), dw_ref) < 5e-6


def test_generic_path_gradients(graph, oracle, gnn):
    """gather/scatter autograd (the path an arbitrary message function takes) ≈ fused path gradients."""
    _, s, t, n, g = graph
    rng = np.random.default_rng(12)
    x = rng.standard_normal((n, 8)).astype(np.float32)
    dout = jl(rng.standard_normal((n, 8)).astype(np.float32))
    for aggr in ("+", "mean", "max"):
        a = jl(x).requires_grad_(True)
        b = jl(x).requires_grad_(True)
        ya = gnn.propagate(gnn.copy_xj, g, aggr, xj=a)
        yb = gnn.propagate(lambda xi, xj, e: xj, g, aggr, xj=b)
        fin = torch.isfinite(ya)
        assert torch.equal(fin, torch.isfinite(yb))
        d = torch.where(fin, dout, torch.zeros_like(dout))
        ya.backward(d); yb.backward(d)
        assert rel(ya.detach().cpu(), yb.detach().cpu()) < TOL
        assert rel(a.grad.cpu(), b.grad.cpu()) < 5e-6


# ---------------------------------------------------------------------------------------- edge softmax
def test_softmax_edge_neighbors_golden(gnn):
    # GNNlib/test/utils.jl:58-67
    g2 = gnn.GNNGraph([1, 2, 3, 4], [5, 5, 6, 6]).cuda()
    e2 = gnn.jl_randn(3, g2.num_edges, device="cuda")
    z = gnn.softmax_edge_neighbors(g2, e2)
    assert z.shape == e2.shape
    assert torch.allclose(z[:, 0:2], torch.softmax(e2[:, 0:2], dim=1), rtol=1e-6, atol=1e-7)
    assert torch.allclose(z[:, 2:4], torch.softmax(e2[:, 2:4], dim=1), rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("K", [1, 3, 8])
def test_softmax_edge_neighbors_parity_and_grad(graph, oracle, gnn, K):
    _, s, t, n, g = graph
    rng = np.random.default_rng(K)
    e = (3 * rng.standard_normal((len(s), K))).astype(np.float32)
    et = jl(e).requires_grad_(True)
    z = gnn.softmax_edge_neighbors(g, et)
    ref = oracle.softmax_edge_neighbors(t, n, e.astype(np.float64))
    assert rel(np_rows(z), ref) < TOL
    da = rng.standard_normal((len(s), K))
    z.backward(jl(da.astype(np.float32)))
    # de_k = a_k (da_k - sum_{k' in N(i)} a_k' da_k')
    T = oracle.scatter("+", ref * da, t, n)
    de_ref = ref * (da - oracle.gather(T, t))
    assert rel(np_rows(et.grad), de_ref) < 2e-5


# ------------------------------------------------------------------------------------------------ layers
class _NT:
    """a Lux-style NamedTuple layer `l` (duck typing, GNNLux/src/layers/conv.jl:131-139)"""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def test_gcn_closed_form_and_conv_weight(gnn):
    # GraphNeuralNetworks/test/layers/conv.jl:30-44
    s, t = [2, 3, 1, 3, 1, 2], [1, 1, 2, 2, 3, 3]
    w = torch.tensor([1, 2, 3, 4, 5, 6], dtype=torch.float32)
    g = gnn.GNNGraph((s, t, w)).cuda()
    x = gnn.colmajor(torch.ones(1, 3).cuda())
    l = gnn.GCNConv(1, 1, add_self_loops=False, use_edge_weight=True, device="cuda")
    with torch.no_grad():
        l.weight.fill_(1)
    d = gnn.degree(g, dir="in", edge_weight=True).cpu().numpy()
    y = l(g, x).detach().cpu().numpy()
    wn = w.numpy()
    np.testing.assert_allclose(y[0, 0], wn[0] / np.sqrt(d[0] * d[1]) + wn[1] / np.sqrt(d[0] * d[2]), rtol=1e-6)
    np.testing.assert_allclose(y[0, 1], wn[2] / np.sqrt(d[1] * d[0]) + wn[3] / np.sqrt(d[1] * d[2]), rtol=1e-6)
    y2 = l(g, x, w.cuda(), norm_fn=lambda d: 1 / torch.sqrt(d)).detach().cpu().numpy()
    np.testing.assert_allclose(y, y2, rtol=1e-6)
    # gradient w.r.t. the edge weights exists and is a vector (conv.jl:47-52)
    wv = torch.rand(6, device="cuda", requires_grad=True)
    l(g, gnn.colmajor(torch.rand(1, 3).cuda()), wv).sum().backward()
    assert wv.grad.shape == (6,) and wv.grad.dtype == torch.float32
    # conv_weight = 0 => output == 0 == w*x exactly (conv.jl:55-65), on the reference's TEST_GRAPHS
    adj1 = np.array([[0, 1, 0, 1], [1, 0, 1, 0], [0, 1, 0, 1], [1, 0, 1, 0]])
    adj2 = np.array([[0, 0, 0, 1], [0, 0, 0, 0], [0, 0, 0, 1], [1, 0, 1, 0]])
    l = gnn.GCNConv(3, 5, device="cuda")
    wz = torch.zeros(5, 3, device="cuda")
    for adj in (adj1, adj2):
        gg = gnn.GNNGraph(adj).cuda()
        xx = gnn.colmajor(torch.rand(3, 4).cuda())
        assert (l(gg, xx, conv_weight=wz) == 0).all()
        assert l(gg, xx).shape == (5, 4)


@pytest.mark.parametrize("din,dout", [(3, 5), (16, 7), (128, 128), (40, 16)])
def test_gcn_conv_parity_and_grad(graph, oracle, gnn, din, dout):
    _check_gcn_conv_parity_and_grad(graph, oracle, gnn, din, dout, True)


@pytest.mark.parametrize("din,dout", [(3, 5), (16, 7), (128, 128), (40, 16)])
def test_gcn_conv_parity_and_grad_without_self_loops(small_graph, oracle, gnn, din, dout):
    """without self loops isolated nodes give c = Inf (the reference tests skip such graphs too): the small graph, with
    every node made a target once"""
    _check_gcn_conv_parity_and_grad(small_graph, oracle, gnn, din, dout, False)


def _check_gcn_conv_parity_and_grad(graph, oracle, gnn, din, dout, loops):
    name, s, t, n, g = graph
    rng = np.random.default_rng(din)
    if not loops:   # make every node a target at least once
        s = np.concatenate([s, np.arange(1, n + 1)]); t = np.concatenate([t, np.roll(np.arange(1, n + 1), 1)])
        g = gnn.GNNGraph(s, t, num_nodes=n).cuda()
    x = rng.standard_normal((n, din)).astype(np.float32)
    W = (rng.standard_normal((dout, din)) / np.sqrt(din)).astype(np.float32)
    b = rng.standard_normal(dout).astype(np.float32)
    l = _NT(weight=torch.as_tensor(W).cuda().requires_grad_(True), bias=torch.as_tensor(b).cuda(), σ=torch.relu,
            add_self_loops=loops, use_edge_weight=False)
    xt = jl(x).requires_grad_(True)
    y = gnn.gcn_conv(l, g, xt)
    # oracle composition (GNNlib/src/layers/conv.jl:14-72) in fp64
    s2, t2 = oracle.add_self_loops(s, t, n) if loops else (s, t)
    x64, W64 = x.astype(np.float64), W.astype(np.float64)
    h = x64 @ W64.T if dout < din else x64
    p, c = oracle.gcn_propagate(s2, t2, n, h, None, fused=True)
    pre = (p @ W64.T if dout >= din else p) + b
    ref = np.maximum(pre, 0)
    assert rel(np_rows(y), ref) < 5e-6
    # gradient of sum(y .* r): dP = c .* A^T-propagate(c .* dPre) etc.
    r = rng.standard_normal(ref.shape)
    (y * jl(r.astype(np.float32))).sum().backward()
    dpre = r * (pre > 0)
    dp = dpre @ W64 if dout >= din else dpre
    dh = oracle.propagate_unfused("+", t2, s2, n, dp * c[:, None]) * c[:, None]      # transposed graph
    dx_ref = dh @ W64 if dout < din else dh
    dW_ref = dpre.T @ p if dout >= din else dh.T @ x64
    assert rel(np_rows(xt.grad), dx_ref) < 1e-5
    assert rel(l.weight.grad.cpu().numpy(), dW_ref) < 1e-5


@pytest.mark.parametrize("aggr", ["mean", "+"])
def test_sage_conv_parity(graph, oracle, gnn, aggr):
    _, s, t, n, g = graph
    rng = np.random.default_rng(3)
    din, dout = 16, 9
    x = rng.standard_normal((n, din)).astype(np.float32)
    W = rng.standard_normal((dout, 2 * din)).astype(np.float32) / 4
    b = rng.standard_normal(dout).astype(np.float32)
    l = _NT(weight=torch.as_tensor(W).cuda(), bias=torch.as_tensor(b).cuda(), σ=torch.relu,
            aggr={"mean": gnn.mean, "+": operator.add}[aggr])
    y = np_rows(gnn.sage_conv(l, g, jl(x)))
    m = oracle.propagate_unfused(aggr, s, t, n, x.astype(np.float64))
    ref = np.maximum(np.concatenate([x.astype(np.float64), m], 1) @ W.astype(np.float64).T + b, 0)
    assert rel(y, ref) < 5e-6
    mod = gnn.SAGEConv(din, dout, torch.relu, device="cuda")
    assert mod(g, jl(x)).shape == (dout, n)


# ----------------------------------------------------------------------------------- C-ABI host entries
def test_host_buffer_entries(graph, oracle, gnn):
    _, s, t, n, g = graph
    lib = gnn._lib.lib
    rng = np.random.default_rng(5)
    D = 32
    x = rng.standard_normal((n, D)).astype(np.float32)
    out = np.empty_like(x)
    gnn._lib.check(lib.gnnb_propagate_host(g.plan().h, 0, gnn._lib.COPY_XJ, gnn._lib.MEAN, x.ctypes.data, None, D,
                                           out.ctypes.data))
    assert rel(out, oracle.propagate_unfused("mean", s, t, n, x.astype(np.float64))) < TOL
    g2 = gnn.add_self_loops(g)
    s2, t2 = oracle.add_self_loops(s, t, n)
    gnn._lib.check(lib.gnnb_gcn_propagate_host(g2.plan().h, 0, x.ctypes.data, None, D, out.ctypes.data))
    ref, c = oracle.gcn_propagate(s2, t2, n, x.astype(np.float64))
    assert rel(out, ref) < TOL
    gnn._lib.check(lib.gnnb_gcn_propagate_host(g2.plan().h, 1, x.ctypes.data, None, D, out.ctypes.data))
    ref_t = oracle.propagate_unfused("+", t2, s2, n, x.astype(np.float64) * c[:, None]) * c[:, None]
    assert rel(out, ref_t) < TOL


def test_determinism(graph, gnn):
    _, s, t, n, g = graph
    x = gnn.jl_randn(128, n, device="cuda")
    a = gnn.propagate(gnn.copy_xj, g, operator.add, xj=x)
    for _ in range(3):
        assert torch.equal(a, gnn.propagate(gnn.copy_xj, g, operator.add, xj=x))


def test_launch_counter(gnn):
    before = gnn.launch_count()
    g = gnn.GNNGraph([1, 2, 3], [2, 3, 1]).cuda()
    gnn.propagate(gnn.copy_xj, g, operator.add, xj=gnn.jl_randn(4, 3, device="cuda"))
    assert gnn.launch_count() > before


# ------------------------------------------------------------------------------------------------- GAT
def _gat_reference_bwd(oracle, s, t, n, Wx, el, er, dout, slope):
    """fp64 closed form of the GAT edge part and its pullback (SURVEY.md §9)."""
    z = el[t - 1] + er[s - 1]                                   # (E, H)
    u = np.where(z > 0, z, slope * z)
    alpha = oracle.softmax_edge_neighbors(t, n, u)
    out = oracle.scatter("+", alpha[:, :, None] * Wx[s - 1], t, n)
    dalpha = (dout[t - 1] * Wx[s - 1]).sum(-1)
    T = oracle.scatter("+", alpha * dalpha, t, n)
    dz = alpha * (dalpha - T[t - 1]) * np.where(z > 0, 1.0, slope)
    del_ = oracle.scatter("+", dz, t, n)
    der = oracle.scatter("+", dz, s, n)
    dWx = oracle.scatter("+", alpha[:, :, None] * dout[t - 1], s, n)
    return out, alpha, dWx, del_, der


@pytest.mark.parametrize("Cc,H", [(64, 8), (16, 4), (8, 2), (4, 1), (32, 2), (128, 1), (128, 4), (2, 3), (1, 4), (16, 1), (32, 4), (64, 4),
                                  (16, 8), (4, 32)])
def test_gat_aggregate_c_abi(graph_with_edges, oracle, gnn, Cc, H):
    name, s, t, n, g = graph_with_edges
    lib = gnn._lib.lib
    rng = np.random.default_rng(Cc * 10 + H)
    s2, t2 = oracle.add_self_loops(s, t, n)
    g2 = gnn.add_self_loops(g)
    E2 = len(s2)
    Wx = rng.standard_normal((n, H, Cc)).astype(np.float32)
    el = rng.standard_normal((n, H)).astype(np.float32)
    er = rng.standard_normal((n, H)).astype(np.float32)
    dout = rng.standard_normal((n, H, Cc)).astype(np.float32)
    slope = 0.2
    dev = lambda a: torch.as_tensor(a).cuda().contiguous()
    Wx_d, el_d, er_d, do_d = dev(Wx), dev(el), dev(er), dev(dout)
    out = torch.empty_like(Wx_d); alpha = torch.empty(E2, H, device="cuda")
    smax = torch.empty(n, H, device="cuda"); ssum = torch.empty(n, H, device="cuda")
    p = g2.plan()
    gnn._lib.check(lib.gnnb_gat_aggregate(p.h, Wx_d.data_ptr(), el_d.data_ptr(), er_d.data_ptr(), Cc, H, slope,
                                          out.data_ptr(), alpha.data_ptr(), smax.data_ptr(), ssum.data_ptr(), None))
    f64 = lambda a: a.astype(np.float64)
    o_ref, a_ref, dWx_ref, del_ref, der_ref = _gat_reference_bwd(oracle, s2, t2, n, f64(Wx), f64(el), f64(er),
                                                                 f64(dout), slope)
    assert rel(out.cpu().numpy(), o_ref) < 5e-6
    assert rel(alpha.cpu().numpy(), a_ref) < 5e-6
    dWx = torch.empty_like(Wx_d); del_ = torch.empty(n, H, device="cuda"); der = torch.empty(n, H, device="cuda")
    gnn._lib.check(lib.gnnb_gat_aggregate_bwd(p.h, Wx_d.data_ptr(), el_d.data_ptr(), er_d.data_ptr(), smax.data_ptr(),
                                              ssum.data_ptr(), out.data_ptr(), do_d.data_ptr(), Cc, H, slope,
                                              dWx.data_ptr(), del_.data_ptr(), der.data_ptr(), None))
    assert rel(dWx.cpu().numpy(), dWx_ref) < 1e-5
    # dz is a difference of O(1) terms: del / der are held to 4x the error of the fp32 oracle on the same inputs
    from test_gpu_gat_backward import check_cancelling
    _, del32, der32, _ = oracle.gat_aggregate_bwd(s2, t2, n, Wx, dout, slope, el=el, er=er)
    check_cancelling("del", del_.cpu().numpy(), del_ref, del32)
    check_cancelling("der", der.cpu().numpy(), der_ref, der32)


def test_gat_unsupported_shape_is_loud(gnn):
    g = gnn.GNNGraph([1, 2], [2, 1]).cuda()
    z = torch.zeros(2, 2, 5, device="cuda")
    with pytest.raises(gnn.GNNBError):
        gnn._lib.check(gnn._lib.lib.gnnb_gat_aggregate(g.plan().h, z.data_ptr(), z.data_ptr(), z.data_ptr(), 5, 2, 0.2,
                                                       z.data_ptr(), None, z.data_ptr(), z.data_ptr(), None))


@pytest.mark.parametrize("din,chout", [(3, 5), (8, 16), (16, 64)])
@pytest.mark.parametrize("heads", [1, 2])
@pytest.mark.parametrize("concat", [True, False])
def test_gat_conv_layer(graph_with_edges, oracle, gnn, din, chout, heads, concat):
    """GraphNeuralNetworks/test/layers/conv.jl:154-170 (heads x concat sweep): output size, fused == the reference's
    own composition (generic gather/softmax/scatter path), gradients of both paths ≈ fp64 autograd, forward ≈ fp64 oracle."""
    name, s, t, n, g = graph_with_edges
    torch.manual_seed(0)
    l = gnn.GATConv(din, chout, torch.relu, heads=heads, concat=concat, device="cuda")
    with torch.no_grad():
        l.bias.normal_()
    rng = np.random.default_rng(1)
    x = rng.standard_normal((n, din)).astype(np.float32)
    xa = jl(x).requires_grad_(True)
    xb = jl(x).requires_grad_(True)
    ya = l(g, xa)                       # fused when the shape allows, else generic
    yb = l(g, xb, fused=False)          # the reference's composition
    assert ya.shape == ((chout * heads) if concat else chout, n)
    assert rel(ya.detach().cpu(), yb.detach().cpu()) < 1e-5
    r_rows = rng.standard_normal((n, ya.shape[0])).astype(np.float32)
    r = jl(r_rows)
    ga = torch.autograd.grad((ya * r).sum(), [xa, l.dense_x.weight, l.a])
    gb = torch.autograd.grad((yb * r).sum(), [xb, l.dense_x.weight, l.a])
    # both paths' gradients against torch float64 autograd of gat_conv (relu' on the fused forward's mask); da cancels
    from test_gpu_gat_backward import check_cancelling, check_plain, gat_conv_torch
    s2, t2 = oracle.add_self_loops(s, t, n)
    mask = torch.as_tensor(np_rows(ya) > 0)

    def ref(dtype):
        leaves = [torch.as_tensor(x, dtype=dtype).requires_grad_(True)] + \
                 [p_.detach().cpu().to(dtype).requires_grad_(True) for p_ in (l.dense_x.weight, l.a)]
        yr = gat_conv_torch(s2, t2, n, *leaves, l.bias.detach().cpu().to(dtype), 0.2, concat, mask.to(dtype))
        return torch.autograd.grad(yr, leaves, torch.as_tensor(r_rows, dtype=dtype))

    (dx64, dW64, da64), da32 = ref(torch.float64), ref(torch.float32)[2]
    for gx, gW, ga_ in (ga, gb):
        check_plain("dx", np_rows(gx), dx64.numpy())
        check_plain("dW", gW.cpu().numpy(), dW64.numpy())
        check_cancelling("da", ga_.cpu().numpy(), da64.numpy(), da32.numpy())
    # forward against the fp64 oracle (GNNlib/src/layers/conv.jl:112-167 restated)
    W = l.dense_x.weight.detach().cpu().numpy().astype(np.float64)          # (C*H, din)
    Wx = (x.astype(np.float64) @ W.T).reshape(n, heads, chout)
    a_rows = l.a.detach().cpu().numpy().astype(np.float64).T                # (H, 2C)
    o, _ = oracle.gat_aggregate(s2, t2, n, Wx, a_rows, 0.2)
    o = o.reshape(n, heads * chout) if concat else o.mean(1)
    ref = np.maximum(o + l.bias.detach().cpu().numpy(), 0)
    assert rel(np_rows(ya), ref) < 1e-5


# ------------------------------------------------------------------------ kernel variants and halo addressing
@pytest.fixture
def variant(gnn):
    yield lambda v: gnn._lib.check(gnn._lib.lib.gnnb_set_kernel_variant(v))
    gnn._lib.lib.gnnb_set_kernel_variant(DEFAULT_VARIANT)


DEFAULT_VARIANT = 0


@pytest.mark.parametrize("D", [128, 256, 512])
@pytest.mark.parametrize("aggr", ["+", "mean", "max", "min"])
def test_tma_staged_variant_is_bit_identical(graph, oracle, gnn, variant, D, aggr):
    """The cp.async.bulk/mbarrier kernel (segbulk.cu, variant 1) against the register-staged one (12): same bits."""
    name, s, t, n, g = graph
    rng = np.random.default_rng(D)
    x = jl(rng.standard_normal((n, D)).astype(np.float32))
    w = torch.as_tensor(rng.random(len(s)).astype(np.float32) + 0.1).cuda()
    variant(12)
    base = gnn.propagate(gnn.copy_xj, g, aggr, xj=x)
    base_w = gnn.propagate(gnn.e_mul_xj, g, aggr, xj=x, e=w)
    assert rel(np_rows(base), oracle.propagate_unfused(aggr, s, t, n, np_rows(x).astype(np.float64))) < TOL
    for v in (1, 5, 0):
        variant(v)
        assert torch.equal(gnn.propagate(gnn.copy_xj, g, aggr, xj=x), base), f"variant {v}"
        assert torch.equal(gnn.propagate(gnn.e_mul_xj, g, aggr, xj=x, e=w), base_w), f"variant {v} weighted"


def test_tma_staged_variant_large_chunks(gnn, oracle, variant):
    """long chunks (many ring wrap-arounds), long rows, GCN scales — both variants, several chunk sizes"""
    rng = np.random.default_rng(0)
    n = 3000
    s, t = make_graph(rng, n, 60000, hubs=2, hub_deg=5000)
    x = rng.standard_normal((n, 128)).astype(np.float32)
    s2, t2 = oracle.add_self_loops(s, t, n)
    ref, _ = oracle.gcn_propagate(s2, t2, n, x.astype(np.float64))
    try:
        for chunk in (32, 128, 1024, 4096):
            gnn._lib.check(gnn._lib.lib.gnnb_set_chunk_edges(chunk))
            g = gnn.GNNGraph(s, t, num_nodes=n).cuda()
            l = gnn.GCNConv(128, 128, device="cuda")
            outs = []
            for v in (12, 1, 5, 0):
                variant(v)
                g2 = gnn.add_self_loops(g)
                c = gnn.layers._gcn_c(g2)
                out = torch.empty(n, 128, device="cuda")
                xr = torch.as_tensor(x).cuda()
                for tr in (0, 1):
                    gnn._lib.check(gnn._lib.lib.gnnb_gcn_propagate(g2.plan().h, tr, xr.data_ptr(), None, c.data_ptr(), 128,
                                                                   out.data_ptr(), None))
                    if tr == 0:
                        assert rel(out.cpu().numpy(), ref) < TOL, (chunk, v)
                outs.append(out.clone())
            assert all(torch.equal(outs[0], o) for o in outs[1:])
    finally:
        gnn._lib.lib.gnnb_set_chunk_edges(128)


@pytest.mark.parametrize("D", [128, 256, 512])
@pytest.mark.parametrize("aggr", ["+", "mean", "max", "min"])
def test_lean_kernel_is_bit_identical(graph, oracle, gnn, variant, D, aggr):
    """The work-item kernel (seglean.cu, variants 0 / 10, and 13 = its TMA gather4 staging) against seg_reduce_kernel (variant 12): same bits for every message /
    aggregation / scale combination, and both against the oracle."""
    name, s, t, n, g = graph
    lib = gnn._lib.lib
    rng = np.random.default_rng(D + 1)
    x = jl(rng.standard_normal((n, D)).astype(np.float32))
    w = torch.as_tensor(rng.random(len(s)).astype(np.float32) + 0.1).cuda()
    cs = torch.rand(n, device="cuda") + 0.5
    ct = torch.rand(n, device="cuda") + 0.5
    p = g.plan()
    A = {"+": gnn._lib.SUM, "mean": gnn._lib.MEAN, "max": gnn._lib.MAX, "min": gnn._lib.MIN}[aggr]

    def scaled(tr, wt):
        out = torch.empty(n, D, device="cuda")
        gnn._lib.check(lib.gnnb_propagate(p.h, tr, gnn._lib.W_MUL_XJ if wt is not None else gnn._lib.COPY_XJ, A,
                                          gnn.rows(x).data_ptr(), None if wt is None else wt.data_ptr(), cs.data_ptr(),
                                          ct.data_ptr(), D, out.data_ptr(), None))
        return out

    def run():
        return [gnn.propagate(gnn.copy_xj, g, aggr, xj=x), gnn.propagate(gnn.e_mul_xj, g, aggr, xj=x, e=w),
                scaled(0, None), scaled(1, None), scaled(0, w), scaled(1, w)]

    variant(12)
    base = run()
    assert rel(np_rows(base[0]), oracle.propagate_unfused(aggr, s, t, n, np_rows(x).astype(np.float64))) < TOL
    for v in (0, 10, 13):                # 13: rows staged by TMA tile::gather4 (plain / node-scaled sums; the rest as 0)
        variant(v)
        for i, (a, b) in enumerate(zip(run(), base)):
            assert torch.equal(a, b), f"variant {v} case {i}"


@pytest.mark.parametrize("D", [128, 256])
def test_lean_kernel_gcn_plan_norm_and_chunks(gnn, oracle, variant, D):
    """GCN core with the plan-owned normalisation (c = NULL: per-edge scale stream) on a graph with hubs (long rows, every
    kind of work item), several chunk sizes: variants 0 / 10 == variant 12 bit for bit, forward and transposed."""
    rng = np.random.default_rng(3)
    n = 3000
    s, t = make_graph(rng, n, 60000, hubs=2, hub_deg=5000)
    x = rng.standard_normal((n, D)).astype(np.float32)
    s2, t2 = oracle.add_self_loops(s, t, n)
    ref, _ = oracle.gcn_propagate(s2, t2, n, x.astype(np.float64))
    lib = gnn._lib.lib
    try:
        for chunk in (32, 128, 1024):
            gnn._lib.check(lib.gnnb_set_chunk_edges(chunk))
            g2 = gnn.add_self_loops(gnn.GNNGraph(s, t, num_nodes=n).cuda())
            c = gnn.layers._gcn_c(g2)
            xr = torch.as_tensor(x).cuda()
            outs = {}
            for v, cp in ((12, c), (10, c), (0, c), (0, None), (13, None), (13, c), (12, None)):
                variant(v)
                for tr in (0, 1):
                    out = torch.empty(n, D, device="cuda")
                    gnn._lib.check(lib.gnnb_gcn_propagate(g2.plan().h, tr, xr.data_ptr(), None,
                                                          None if cp is None else cp.data_ptr(), D, out.data_ptr(), None))
                    if tr == 0:
                        assert rel(out.cpu().numpy(), ref) < TOL, (chunk, v)
                    outs.setdefault(tr, []).append(out)
            for tr in (0, 1):
                assert all(torch.equal(outs[tr][0], o) for o in outs[tr][1:]), (chunk, tr)
    finally:
        lib.gnnb_set_chunk_edges(128)


def test_lean_kernel_halo_bases(graph, gnn, variant):
    """gnnb_propagate_halo through the lean kernel: two source bases, node scales gathered per edge"""
    name, s, t, n, g = graph
    lib = gnn._lib.lib
    D = 128
    rng = np.random.default_rng(9)
    x = torch.as_tensor(rng.standard_normal((n, D)).astype(np.float32)).cuda()
    n_local = n // 3
    x_local, x_halo = x[:n_local].clone(), x[n_local:].clone()
    cs = torch.rand(n, device="cuda") + 0.5
    ct = torch.rand(n, device="cuda") + 0.5
    p = g.plan()
    outs = []
    for v in (12, 0):
        variant(v)
        out = torch.empty_like(x)
        gnn._lib.check(lib.gnnb_propagate_halo(p.h, gnn._lib.COPY_XJ, gnn._lib.SUM, x_local.data_ptr(), x_halo.data_ptr(),
                                               n_local, None, cs.data_ptr(), ct.data_ptr(), D, out.data_ptr(), None))
        outs.append(out)
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("D", [5, 16, 128, 256])
def test_halo_addressing_and_gather_rows(graph, oracle, gnn, variant, D):
    """gnnb_propagate_halo: sources < n_local read x_local, the rest x_halo (the [local | halo] space of a shard)."""
    name, s, t, n, g = graph
    lib = gnn._lib.lib
    rng = np.random.default_rng(D)
    x = torch.as_tensor(rng.standard_normal((n, D)).astype(np.float32)).cuda()
    n_local = n // 3
    x_local, x_halo = x[:n_local].clone(), x[n_local:].clone()
    cs = torch.rand(n, device="cuda") + 0.5
    ct = torch.rand(n, device="cuda") + 0.5
    ref = torch.empty_like(x)
    p = g.plan()
    for v in (0, 1, 5, 12):
        variant(v)
        gnn._lib.check(lib.gnnb_propagate(p.h, 0, gnn._lib.COPY_XJ, gnn._lib.SUM, x.data_ptr(), None, cs.data_ptr(),
                                          ct.data_ptr(), D, ref.data_ptr(), None))
        out = torch.empty_like(x)
        gnn._lib.check(lib.gnnb_propagate_halo(p.h, gnn._lib.COPY_XJ, gnn._lib.SUM, x_local.data_ptr(),
                                               x_halo.data_ptr(), n_local, None, cs.data_ptr(), ct.data_ptr(), D,
                                               out.data_ptr(), None))
        assert torch.equal(out, ref)
    idx = torch.as_tensor(rng.integers(0, n, 77).astype(np.int32)).cuda()
    packed = torch.empty(77, D, device="cuda")
    gnn._lib.check(lib.gnnb_gather_rows(idx.data_ptr(), 77, x.data_ptr(), D, packed.data_ptr(), None))
    assert torch.equal(packed, x[idx.long()])


# --------------------------------------------------------------------------------------------- dense layer part
@pytest.mark.parametrize("N,Din,Dout", [(1000, 128, 128), (777, 16, 8), (5000, 64, 256), (33, 1432, 16), (0, 8, 8),
                                        (4096, 64, 128), (130000, 128, 64), (300, 32, 16), (129, 96, 48), (1, 128, 128),
                                        (400000, 128, 128), (70001, 96, 128),
                                        # the wide tcgen05 kernel (K or Nout above 128, N >= 2048): GATConv 512 -> 8 x 64, config 5
                                        (40000, 512, 512), (3000, 256, 256), (20001, 512, 128), (2048, 160, 384),
                                        (9000, 1024, 1024)])
@pytest.mark.parametrize("relu_flag,with_bias", [(1, True), (0, True), (1, False), (0, False)])
@pytest.mark.parametrize("emulate", [1, 0])
def test_linear_c_abi(gnn, N, Din, Dout, relu_flag, with_bias, emulate):
    # emulate=1: hand-written tcgen05 3xTF32 kernel where the shape allows, cuBLASLt fp32-emulated GEMM elsewhere;
    # emulate=0: cuBLASLt SIMT sgemm only (tensor-core kernel switched off)
    """gnnb_linear / gnnb_linear_bwd (σ.(W*x .+ b), conv.jl:69-71) against fp64: the fp32-emulated tensor-core GEMM must
    stay inside the 1e-5 bar, like the SIMT sgemm."""
    lib = gnn._lib.lib
    lib.gnnb_dense_set_emulation(emulate)
    lib.gnnb_dense_set_tensor_core_kernel(emulate)
    try:
        gen = torch.Generator(device="cuda").manual_seed(N + Din)
        x = torch.randn(N, Din, device="cuda", generator=gen)
        W = torch.randn(Dout, Din, device="cuda", generator=gen) / Din ** 0.5
        b = torch.randn(Dout, device="cuda", generator=gen) if with_bias else None
        dy = torch.randn(N, Dout, device="cuda", generator=gen)
        y = torch.empty(N, Dout, device="cuda")
        gnn._lib.check(lib.gnnb_linear(x.data_ptr(), W.data_ptr(), None if b is None else b.data_ptr(), relu_flag, N, Din,
                                       Dout, y.data_ptr(), None))
        pre = x.double() @ W.double().t() + (0 if b is None else b.double())
        ref = pre.clamp(min=0) if relu_flag else pre
        if N:
            assert rel(y.cpu(), ref.cpu()) < 5e-6
        ws = torch.empty_like(dy); dx = torch.empty_like(x); dW = torch.empty_like(W); db = torch.empty(Dout, device="cuda")
        gnn._lib.check(lib.gnnb_linear_bwd(dy.data_ptr(), y.data_ptr(), x.data_ptr(), W.data_ptr(), relu_flag, N, Din, Dout,
                                           ws.data_ptr(), dx.data_ptr(), dW.data_ptr(), db.data_ptr(), None))
        dpre = dy.double() * (y > 0) if relu_flag else dy.double()
        if N:
            assert rel(dx.cpu(), (dpre @ W.double()).cpu()) < 5e-6
            assert rel(dW.cpu(), (dpre.t() @ x.double()).cpu()) < 5e-6
            assert rel(db.cpu(), dpre.sum(0).cpu()) < 5e-6
        else:
            assert (db == 0).all()
        assert lib.gnnb_dense_emulation_active() in (-1, 0, 1)
        assert lib.gnnb_dense_tc_error() == 0          # the tcgen05 pipeline never timed out
    finally:
        lib.gnnb_dense_set_emulation(1)
        lib.gnnb_dense_set_tensor_core_kernel(1)


def test_linear_wide_accumulation_drift(gnn):
    """All-positive operands at K = 512: every product has the same sign, the case in which the tensor core's truncating
    accumulator drifts most.  The wide kernel keeps the full-magnitude chain at K/8 accumulations; the bar stays 5e-6."""
    lib = gnn._lib.lib
    N, K, Nout = 30000, 512, 512
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = torch.rand(N, K, device="cuda", generator=gen) + 0.5
    W = torch.rand(Nout, K, device="cuda", generator=gen) + 0.5
    y = torch.empty(N, Nout, device="cuda")
    n0 = gnn.launch_count()
    gnn._lib.check(lib.gnnb_linear(x.data_ptr(), W.data_ptr(), None, 0, N, K, Nout, y.data_ptr(), None))
    assert gnn.launch_count() == n0 + 2                      # the W-image pre-pass + the hand-written kernel, not the library GEMM
    ref = x.double() @ W.double().t()
    assert rel(y.cpu(), ref.cpu()) < 5e-6
    assert float(((y.double() - ref) / ref).abs().max()) < 2e-5
    assert lib.gnnb_dense_tc_error() == 0


# ---------------------------------------------------------------------------------- full-size properties (config 2)
def test_full_size_properties(gnn):
    """BASELINE configs[1] sizes (RMAT N=10M, E=100M, D=128): size-independent properties instead of an oracle run —
    propagate(ones) == in-degree exactly (integers are exact in fp32), GCN normalisation of ones, linearity, and
    <A x, y> == <x, A^T y> between the forward and the transposed plan."""
    n, E, D = 10_000_000, 100_000_000, 128
    g = gnn.rmat_graph(n, E, 17)
    deg = gnn.degree(g, torch.float32, dir="in")
    assert int(deg.double().sum().item()) == E                     # checksum of the whole edge list
    ones = gnn.unrows(torch.ones(n, 8, device="cuda"))
    out = gnn.propagate(gnn.copy_xj, g, operator.add, xj=ones)
    assert torch.equal(gnn.rows(out)[:, 0], deg) and torch.equal(gnn.rows(out)[:, 7], deg)
    m = gnn.propagate(gnn.copy_xj, g, gnn.mean, xj=ones)
    assert torch.equal(gnn.rows(m)[:, 0], (deg > 0).float())       # mean of ones is 1 where there are in-edges, else 0
    del ones, out, m
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(n, D, device="cuda", generator=gen)
    y = torch.randn(n, D, device="cuda", generator=gen)
    px = gnn.rows(gnn.propagate(gnn.copy_xj, g, operator.add, xj=gnn.unrows(x)))
    # linearity: P(2x + y) == 2 P(x) + P(y) up to rounding
    py = gnn.rows(gnn.propagate(gnn.copy_xj, g, operator.add, xj=gnn.unrows(y)))
    pz = gnn.rows(gnn.propagate(gnn.copy_xj, g, operator.add, xj=gnn.unrows(2 * x + y)))
    assert float((pz - (2 * px + py)).norm() / pz.norm()) < 1e-6
    del py, pz
    # adjointness between the two plans: <P x, y> == <x, P^T y>
    lib = gnn._lib.lib
    pty = torch.empty_like(x)
    gnn._lib.check(lib.gnnb_propagate(g.plan().h, 1, gnn._lib.COPY_XJ, gnn._lib.SUM, y.data_ptr(), None, None, None, D,
                                      pty.data_ptr(), None))
    a = float((px.double() * y.double()).sum()); b = float((x.double() * pty.double()).sum())
    assert abs(a - b) <= 1e-6 * max(abs(a), abs(b), 1.0)


# ---------------------------------------------------------------------------------- oracle parity at scale
def test_at_scale_propagate_against_the_oracle(gnn, oracle):
    """RMAT N = 1 M, E = 10 M, D = 128 (real hubs of 10^4-10^5 edges, thousands of long rows through the fix-up kernel, every
    kind of work item): `+` against the oracle's fused CPU path (CSC rebuild + dense x CSC, fp64), mean / max against the
    unfused gather -> scatter path on the first 4 M edges; CSR integers with ==."""
    n, E, D = 1_000_000, 10_000_000, 128
    g = gnn.rmat_graph(n, E, 17)
    s, t = oracle.rmat(n, E, 17)
    assert np.array_equal(g.s.cpu().numpy(), s) and np.array_equal(g.t.cpu().numpy(), t)       # generator: GPU == CPU
    rowptr = np.empty(n + 1, np.int32)
    gnn._lib.check(gnn._lib.lib.gnnb_graph_csr(g.plan().h, 0, rowptr.ctypes.data, None, None, None))
    assert np.array_equal(np.diff(rowptr), np.bincount(t - 1, minlength=n))                      # in-degrees, exact
    rng = np.random.default_rng(0)
    x = rng.standard_normal((n, D)).astype(np.float32)
    out = gnn.propagate(gnn.copy_xj, g, operator.add, xj=jl(x))
    assert rel(np_rows(out), oracle.propagate_fused(s, t, n, x.astype(np.float64))) < TOL
    del out
    Em = 4_000_000
    gm = gnn.GNNGraph(s[:Em], t[:Em], num_nodes=n).cuda()
    for aggr in ("mean", "max"):
        out = gnn.propagate(gnn.copy_xj, gm, aggr, xj=jl(x))
        assert rel(np_rows(out), oracle.propagate_unfused(aggr, s[:Em], t[:Em], n, x.astype(np.float64))) < TOL, aggr


def test_at_scale_gcn_layer_against_the_oracle(gnn, oracle):
    """GCNConv 128 -> 128 forward + backward on RMAT N = 1 M, E = 10 M against the oracle composition in fp64 (bar 1e-5)."""
    n, E, D = 1_000_000, 10_000_000, 128
    s, t = oracle.rmat(n, E, 17)
    g = gnn.GNNGraph(s, t, num_nodes=n).cuda()
    rng = np.random.default_rng(1)
    x = rng.standard_normal((n, D)).astype(np.float32)
    dy = rng.standard_normal((n, D)).astype(np.float32)
    layer = gnn.GCNConv(D, D, torch.relu, device="cuda")
    with torch.no_grad():
        layer.bias.normal_()
    W, b = layer.weight.detach().cpu().numpy().astype(np.float64), layer.bias.detach().cpu().numpy().astype(np.float64)
    xt = jl(x).requires_grad_(True)
    y = layer(g, xt)
    y.backward(jl(dy))
    s2, t2 = oracle.add_self_loops(s, t, n)
    p, c = oracle.gcn_propagate(s2, t2, n, x.astype(np.float64))
    pre = p @ W.T + b
    yg = np_rows(y)
    assert rel(yg, np.maximum(pre, 0)) < 1e-5
    # relu' is discontinuous at 0: where |pre| is below fp32 resolution the GPU's mask and the fp64 one may differ (a
    # handful of the 128 M elements, each worth O(1e-3) of a bias-gradient entry) — the pullback is checked on the mask of
    # the forward output it belongs to, the disagreements are counted
    assert int(((yg > 0) != (pre > 0)).sum()) < 1e-6 * pre.size
    dpre = dy.astype(np.float64) * (yg > 0)
    assert rel(layer.weight.grad.cpu().numpy(), dpre.T @ p) < 1e-5
    assert rel(layer.bias.grad.cpu().numpy(), dpre.sum(0)) < 1e-5
    dp = (dpre @ W) * c[:, None]
    dx = oracle.propagate_fused(t2, s2, n, dp) * c[:, None]                  # A' through the transposed edge list
    assert rel(np_rows(xt.grad), dx) < 1e-5


def test_at_scale_gat_layer_against_the_oracle(gnn, oracle):
    """GATConv 8 heads x 64 on RMAT N = 100 k, E = 1 M (config-3 shape): forward against the oracle's step-by-step
    restatement of gat_conv / gat_message in fp64."""
    n, E, H, Cc = 100_000, 1_000_000, 8, 64
    D = H * Cc
    s, t = oracle.rmat(n, E, 17)
    g = gnn.GNNGraph(s, t, num_nodes=n).cuda()
    rng = np.random.default_rng(2)
    x = rng.standard_normal((n, D)).astype(np.float32)
    layer = gnn.GATConv(D, Cc, torch.relu, heads=H, device="cuda")
    with torch.no_grad():
        y = layer(g, jl(x))
    Wd = layer.dense_x.weight.detach().cpu().numpy().astype(np.float64)
    a = layer.a.detach().cpu().numpy().astype(np.float64)
    s2, t2 = oracle.add_self_loops(s, t, n)
    Wx = (x.astype(np.float64) @ Wd.T).reshape(n, H, Cc)
    o, _ = oracle.gat_aggregate(s2, t2, n, Wx, np.ascontiguousarray(a.T))
    ref = np.maximum(o.reshape(n, D) + layer.bias.detach().cpu().numpy(), 0)
    assert rel(np_rows(y), ref) < 1e-5


def test_at_scale_sage_on_batched_graphs_against_the_oracle(gnn, oracle):
    """SAGEConv mean on a config-4-shaped batch (1024 graphs x 1000 nodes, 5000 edges): mean aggregation and the layer
    output against the oracle (unfused gather -> scatter(mean), vcat, GEMM) in fp64."""
    G, n1, e1, D = 1024, 1000, 5000, 128
    n = G * n1
    rng = np.random.default_rng(3)
    off = np.repeat(np.arange(G) * n1, e1)
    s = rng.integers(0, n1, G * e1) + off + 1
    t = rng.integers(0, n1, G * e1) + off + 1
    g = gnn.GNNGraph(s, t, num_nodes=n).cuda()
    x = rng.standard_normal((n, D)).astype(np.float32)
    m_ref = oracle.propagate_unfused("mean", s, t, n, x.astype(np.float64))
    m = gnn.propagate(gnn.copy_xj, g, gnn.mean, xj=jl(x))
    assert rel(np_rows(m), m_ref) < TOL
    layer = gnn.SAGEConv(D, D, torch.relu, device="cuda")
    with torch.no_grad():
        y = layer(g, jl(x))
    W, b = layer.weight.detach().cpu().numpy().astype(np.float64), layer.bias.detach().cpu().numpy().astype(np.float64)
    ref = np.maximum(np.concatenate([x.astype(np.float64), m_ref], axis=1) @ W.T + b, 0)
    assert rel(np_rows(y), ref) < 1e-5


@pytest.mark.parametrize("Cc,H,n", [(64, 8, 777), (4, 3, 100), (128, 2, 50), (16, 5, 1000), (8, 1, 33)])
def test_gat_logit_terms_c_abi(gnn, Cc, H, n):
    """gnnb_gat_logit_terms(+_bwd): el / er = the two halves of sum(a .* vcat(Wxi, Wxj), dims=1) (conv.jl:157-163) per node,
    the in-place dWx accumulation and the deterministic da reduction, against float64 torch."""
    lib = gnn._lib.lib
    gen = torch.Generator(device="cuda").manual_seed(Cc * 31 + H)
    Wx = torch.randn(n, H, Cc, device="cuda", generator=gen)
    a = torch.randn(2 * Cc, H, device="cuda", generator=gen)            # Julia-shaped (2C, H)
    a_jl = a.t().contiguous()                                            # its column-major memory
    el, er = torch.empty(n, H, device="cuda"), torch.empty(n, H, device="cuda")
    gnn._lib.check(lib.gnnb_gat_logit_terms(Wx.data_ptr(), a_jl.data_ptr(), n, Cc, H, el.data_ptr(), er.data_ptr(), None))
    W64, a64 = Wx.double(), a.double()
    el_ref = (W64 * a64[:Cc].t().unsqueeze(0)).sum(-1)
    er_ref = (W64 * a64[Cc:].t().unsqueeze(0)).sum(-1)
    assert float((el.double() - el_ref).norm() / el_ref.norm()) < 2e-6
    assert float((er.double() - er_ref).norm() / er_ref.norm()) < 2e-6
    dl = torch.randn(n, H, device="cuda", generator=gen)
    dr = torch.randn(n, H, device="cuda", generator=gen)
    dWx0 = torch.randn(n, H, Cc, device="cuda", generator=gen)
    outs = []
    for _ in range(2):                                                   # twice: the reduction is deterministic
        dWx = dWx0.clone()
        da = torch.empty(H, 2 * Cc, device="cuda")
        gnn._lib.check(lib.gnnb_gat_logit_terms_bwd(Wx.data_ptr(), a_jl.data_ptr(), dl.data_ptr(), dr.data_ptr(), n, Cc, H,
                                                    dWx.data_ptr(), da.data_ptr(), None))
        outs.append((dWx, da))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    dWx_ref = dWx0.double() + dl.double()[:, :, None] * a64[:Cc].t().unsqueeze(0) + dr.double()[:, :, None] * a64[Cc:].t().unsqueeze(0)
    da_ref = torch.cat([(dl.double()[:, :, None] * W64).sum(0), (dr.double()[:, :, None] * W64).sum(0)], dim=1)   # (H, 2C)
    assert float((outs[0][0].double() - dWx_ref).norm() / dWx_ref.norm()) < 2e-6
    assert float((outs[0][1].double() - da_ref).norm() / da_ref.norm()) < 5e-6


@pytest.mark.parametrize("N,D1,D2", [(70001, 128, 128), (5000, 96, 32), (129, 128, 64)])
@pytest.mark.parametrize("relu_flag,with_bias", [(1, True), (0, False)])
def test_linear2_c_abi(gnn, N, D1, D2, relu_flag, with_bias):
    """gnnb_linear2 / gnnb_linear2_bwd — σ.(W * vcat(x1, x2) .+ b) as two accumulating tcgen05 passes over the column blocks
    of W (sage_conv, conv.jl:281) — against float64."""
    lib = gnn._lib.lib
    Dout = 128
    gen = torch.Generator(device="cuda").manual_seed(N + D1)
    x1 = torch.randn(N, D1, device="cuda", generator=gen)
    x2 = torch.randn(N, D2, device="cuda", generator=gen)
    W = torch.randn(Dout, D1 + D2, device="cuda", generator=gen) / (D1 + D2) ** 0.5
    b = torch.randn(Dout, device="cuda", generator=gen) if with_bias else None
    dy = torch.randn(N, Dout, device="cuda", generator=gen)
    y = torch.empty(N, Dout, device="cuda")
    gnn._lib.check(lib.gnnb_linear2(x1.data_ptr(), x2.data_ptr(), W.data_ptr(), None if b is None else b.data_ptr(), relu_flag,
                                    N, D1, D2, Dout, y.data_ptr(), None))
    pre = torch.cat([x1, x2], 1).double() @ W.double().t() + (0 if b is None else b.double())
    ref = pre.clamp(min=0) if relu_flag else pre
    assert rel(y.cpu(), ref.cpu()) < 5e-6
    ws = torch.empty_like(dy); dx1 = torch.empty_like(x1); dx2 = torch.empty_like(x2)
    dW = torch.empty_like(W); db = torch.empty(Dout, device="cuda")
    gnn._lib.check(lib.gnnb_linear2_bwd(dy.data_ptr(), y.data_ptr(), x1.data_ptr(), x2.data_ptr(), W.data_ptr(), relu_flag, N, D1,
                                        D2, Dout, ws.data_ptr(), dx1.data_ptr(), dx2.data_ptr(), dW.data_ptr(),
                                        db.data_ptr() if with_bias else None, None))
    dpre = dy.double() * (y > 0) if relu_flag else dy.double()
    assert rel(dx1.cpu(), (dpre @ W.double()[:, :D1]).cpu()) < 5e-6
    assert rel(dx2.cpu(), (dpre @ W.double()[:, D1:]).cpu()) < 5e-6
    assert rel(dW.cpu(), (dpre.t() @ torch.cat([x1, x2], 1).double()).cpu()) < 5e-6
    if with_bias:
        assert rel(db.cpu(), dpre.sum(0).cpu()) < 5e-6
    assert lib.gnnb_dense_tc_error() == 0


@pytest.mark.parametrize("N,D", [(70001, 512), (1, 4), (4099, 36), (0, 64)])
@pytest.mark.parametrize("relu_flag,with_bias", [(1, True), (0, True), (1, False)])
def test_bias_act_c_abi(gnn, N, D, relu_flag, with_bias):
    """gnnb_bias_act / gnnb_bias_act_bwd — σ.(x .+ b), the closing line of GATConv (conv.jl:149): exact forward (one add, one
    max), exact mask product, deterministic bias gradient against float64."""
    lib = gnn._lib.lib
    gen = torch.Generator(device="cuda").manual_seed(N + D)
    x = torch.randn(N, D, device="cuda", generator=gen)
    b = torch.randn(D, device="cuda", generator=gen) if with_bias else None
    dy = torch.randn(N, D, device="cuda", generator=gen)
    y = torch.full((N, D), float("nan"), device="cuda")
    gnn._lib.check(lib.gnnb_bias_act(x.data_ptr() if N else None, None if b is None else b.data_ptr(), relu_flag, N, D,
                                     y.data_ptr() if N else None, None))
    pre = x if b is None else x + b
    assert torch.equal(y, pre.clamp(min=0) if relu_flag else pre)
    dpre = torch.full((N, D), float("nan"), device="cuda")
    dbs = []
    for _ in range(2):
        db = torch.full((D,), float("nan"), device="cuda")
        gnn._lib.check(lib.gnnb_bias_act_bwd(dy.data_ptr() if N else None, y.data_ptr() if N else None, relu_flag, N, D,
                                             dpre.data_ptr() if (N and relu_flag) else None, db.data_ptr() if with_bias else None, None))
        dbs.append(db)
    ref = dy * (y > 0) if relu_flag else dy
    if relu_flag:
        assert torch.equal(dpre, ref)
    if with_bias:
        assert torch.equal(dbs[0], dbs[1])
        if N:
            assert rel(dbs[0].cpu(), ref.double().sum(0).cpu()) < 2e-6
        else:
            assert float(dbs[0].abs().max()) == 0.0


def test_gat_conv_closing_line_uses_the_fused_pass(gnn, small_graph):
    """GATConv's σ.(x .+ bias) goes through gnnb_bias_act (one kernel) and differentiates like the torch composition"""
    _, _, _, n, g = small_graph
    torch.manual_seed(3)
    l = gnn.GATConv(32, 16, torch.relu, heads=4, device="cuda")
    with torch.no_grad():
        l.bias.normal_()
    x = torch.randn(32, n, device="cuda", requires_grad=True)
    n0 = gnn.launch_count()
    y = gnn.gat_conv(l, g, x)
    assert gnn.launch_count() > n0
    dy = torch.randn_like(y)
    gx, ga, gb, gw = torch.autograd.grad(y, [x, l.a, l.bias, l.dense_x.weight], dy)
    from gnnb200 import layers as L
    saved = L._bias_act
    try:
        L._bias_act = lambda ll, out: L._sigma(ll)(L._add_bias(out, L._bias(ll)))
        y2 = gnn.gat_conv(l, g, x)
        gx2, ga2, gb2, gw2 = torch.autograd.grad(y2, [x, l.a, l.bias, l.dense_x.weight], dy)
    finally:
        L._bias_act = saved
    assert torch.equal(y, y2)
    for a_, b_ in ((gx, gx2), (ga, ga2), (gw, gw2), (gb, gb2)):
        assert rel(a_.cpu(), b_.cpu()) < 2e-6
