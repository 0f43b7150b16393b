"""The fp64 pullback of the GAT edge part in the CPU oracle (orc_gat_aggregate_bwd), pinned before any GPU test leans on it:
against central finite differences of the oracle's own step-by-step forward (orc_gat_aggregate), and against torch float64
autograd of an independent restatement of gat_conv's edge part (GNNlib/src/layers/conv.jl:136-141,152-167)."""
import numpy as np
import pytest
import torch


def _graph(rng):
    """a small multigraph with a hub target, duplicate edges, a node without in-edges and one without out-edges"""
    n = 14
    s = list(rng.integers(1, n - 1, 30))                 # node n never sends
    t = list(rng.integers(1, n - 2, 30))                 # nodes n-1, n never receive
    s += list(rng.integers(1, n - 1, 25)); t += [3] * 25   # hub
    s += [5, 5, 5]; t += [7, 7, 7]                       # duplicates: tied logits
    p = rng.permutation(len(s))
    return np.asarray(s, np.int64)[p], np.asarray(t, np.int64)[p], n


def _inputs(seed, H, Cc, ties):
    rng = np.random.default_rng(seed)
    s, t, n = _graph(rng)
    Wx = rng.standard_normal((n, H, Cc))
    if ties:      # logits from a few values: many edges of a row share the maximum; |z| >= 0.5 keeps FD off the kink
        el = rng.choice([-1.0, 0.5, 2.0], (n, H))
        er = rng.choice([-1.0, 0.5, 2.0], (n, H))
    else:
        el = rng.standard_normal((n, H))
        er = rng.standard_normal((n, H))
    dout = rng.standard_normal((n, H, Cc))
    return s, t, n, Wx, el, er, dout


def _loss(oracle, s, t, n, Wx, el, er, dout, slope):
    """<out, dout> through the oracle's forward, whose logits are a·vcat(Wxi, Wxj): el and er ride in two extra channels
    whose `a` entries are 1 (target half, channel C) and 1 (source half, channel C+1), every other entry 0 — the sums are
    then exactly el[t] + er[s], and the extra output channels carry no upstream gradient"""
    N, H, Cc = Wx.shape
    Wa = np.concatenate([Wx, el[:, :, None], er[:, :, None]], axis=2)
    a = np.zeros((H, 2 * (Cc + 2)))
    a[:, Cc] = 1.0
    a[:, (Cc + 2) + Cc + 1] = 1.0
    out, _ = oracle.gat_aggregate(s, t, n, Wa, a, slope)
    return float((out[:, :, :Cc] * dout).sum())


def _fd(f, x, h=1e-5):
    g = np.empty_like(x)
    for i in np.ndindex(x.shape):
        x0 = x[i]
        x[i] = x0 + h; fp = f()
        x[i] = x0 - h; fm = f()
        x[i] = x0
        g[i] = (fp - fm) / (2 * h)
    return g


def _rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


@pytest.mark.parametrize("slope", [0.2, 0.0])
@pytest.mark.parametrize("H,Cc,ties", [(2, 3, False), (1, 4, True), (3, 2, True)])
def test_pullback_matches_finite_differences(oracle, H, Cc, ties, slope):
    s, t, n, Wx, el, er, dout = _inputs(H * 10 + Cc, H, Cc, ties)
    dWx, del_, der, _ = oracle.gat_aggregate_bwd(s, t, n, Wx, dout, slope, el=el, er=er)
    f = lambda: _loss(oracle, s, t, n, Wx, el, er, dout, slope)
    for got, x in ((dWx, Wx), (del_, el), (der, er)):
        ref = _fd(f, x)
        assert _rel(got, ref) < 1e-7
    assert np.abs(del_[[n - 2, n - 1]]).max() == 0 and np.abs(der[n - 1]).max() == 0 and np.abs(dWx[n - 1]).max() == 0


def _edge_part_torch(s, t, n, Wx, el, er, slope):
    """gat_conv's edge part in plain torch: per-edge logits, leakyrelu, neighbourhood softmax by scatter_reduce / index_add,
    α-weighted sum by index_add"""
    s0, t0 = torch.as_tensor(s - 1), torch.as_tensor(t - 1)
    H = Wx.shape[1]
    z = el[t0] + er[s0]
    u = torch.nn.functional.leaky_relu(z, slope)
    m = torch.full((n, H), -torch.inf, dtype=u.dtype).scatter_reduce(0, t0[:, None].expand(-1, H), u.detach(), "amax")
    ex = torch.exp(u - m[t0])
    den = torch.zeros(n, H, dtype=u.dtype).index_add(0, t0, ex)
    alpha = ex / den[t0]
    out = torch.zeros_like(Wx).index_add(0, t0, alpha[:, :, None] * Wx[s0])
    return out, alpha


@pytest.mark.parametrize("slope", [0.2, 0.0])
@pytest.mark.parametrize("H,Cc,ties", [(2, 3, False), (4, 8, False), (3, 2, True)])
def test_pullback_matches_torch_autograd(oracle, H, Cc, ties, slope):
    s, t, n, Wx, el, er, dout = _inputs(H * 100 + Cc, H, Cc, ties)
    dWx, del_, der, alpha = oracle.gat_aggregate_bwd(s, t, n, Wx, dout, slope, el=el, er=er)
    leaves = [torch.tensor(v, requires_grad=True) for v in (Wx, el, er)]
    out, al = _edge_part_torch(s, t, n, *leaves, slope)
    grads = torch.autograd.grad((out * torch.as_tensor(dout)).sum(), leaves)
    assert _rel(alpha, al.detach().numpy()) < 1e-12
    for got, ref in zip((dWx, del_, der), grads):
        assert _rel(got, ref.numpy()) < 1e-12


def test_pullback_through_the_attention_vector(oracle):
    """with `a` given the logits are its two halves against Wx; the chain dWx += del a_t + der a_s, da = [Σ del Wx, Σ der Wx]
    (what the GPU tests apply to the pullback) matches finite differences of the oracle's forward in Wx and a"""
    H, Cc, slope = 2, 3, 0.2
    s, t, n, Wx, _, _, dout = _inputs(7, H, Cc, False)
    a = np.random.default_rng(8).standard_normal((H, 2 * Cc))
    dWx, del_, der, _ = oracle.gat_aggregate_bwd(s, t, n, Wx, dout, slope, a=a)
    dWx_full = dWx + del_[:, :, None] * a[None, :, :Cc] + der[:, :, None] * a[None, :, Cc:]
    da = np.concatenate([np.einsum("nh,nhc->hc", del_, Wx), np.einsum("nh,nhc->hc", der, Wx)], axis=1)
    f = lambda: float((oracle.gat_aggregate(s, t, n, Wx, a, slope)[0] * dout).sum())
    assert _rel(dWx_full, _fd(f, Wx)) < 1e-7
    assert _rel(da, _fd(f, a)) < 1e-7


def test_fp32_pullback_tracks_fp64(oracle):
    """the fp32 instantiation (the measured conditioning of the GPU bounds) runs the same sequence in float32"""
    s, t, n, Wx, el, er, dout = _inputs(11, 4, 8, False)
    r64 = oracle.gat_aggregate_bwd(s, t, n, Wx, dout, 0.2, el=el, er=er)
    f32 = lambda v: v.astype(np.float32)
    r32 = oracle.gat_aggregate_bwd(s, t, n, f32(Wx), f32(dout), 0.2, el=f32(el), er=f32(er))
    for a32, a64 in zip(r32, r64):
        assert a32.dtype == np.float32
        assert 0 < _rel(a32.astype(np.float64), a64) < 1e-5
