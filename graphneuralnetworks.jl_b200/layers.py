"""The three functional layers that ride on the hot path, with the reference's signatures:

    gcn_conv(l, g, x, edge_weight, norm_fn, conv_weight)   GNNlib/src/layers/conv.jl:14-72
    gat_conv(l, g, x, e)  + gat_message                    GNNlib/src/layers/conv.jl:112-167
    sage_conv(l, g, x)                                     GNNlib/src/layers/conv.jl:277-283

``l`` is duck-typed exactly as in the reference (a Flux struct or a Lux NamedTuple there; any object with the
same field names here): GCN ``weight, bias, σ|sigma, add_self_loops, use_edge_weight``; GAT ``dense_x, dense_e, a,
bias, σ, negative_slope, channel, heads, concat, add_self_loops, dropout``; SAGE ``weight, bias, σ, aggr``.
``GCNConv`` / ``GATConv`` / ``SAGEConv`` are thin parameter holders mirroring the Flux constructors
(GraphNeuralNetworks/src/layers/conv.jl:77-104, 309-346, 770-787).

Arrays are Julia-shaped and column-major: x is (Din, N), weight is (Dout, Din), GAT's ``a`` is (2C, H).
The dense contractions `σ.(W*x .+ b)` go through gnnb_linear / gnnb_linear_bwd (hand-written tcgen05 3xTF32 kernels with
the bias/relu epilogue; cuBLASLt for shapes they do not cover) when the shape allows, torch's fp32 matmul otherwise.

Further down: the layers SURVEY.md §8f ranks first because they re-parameterise the same kernels — graph_conv, gin_conv,
sgc_conv / sg_conv, tag_conv, gated_graph_conv, agnn_conv, gatv2_conv, transformer_conv — with their parameter holders.
"""
from __future__ import annotations

import math
import operator
from typing import Callable, Optional

import torch

from . import _lib
from ._lib import lib
from .graph import GNNGraph, _stream, add_self_loops, degree, rows, unrows
from .msgpass import (Fix1, _GCNPropagateFn, _f32, aggregate_neighbors, apply_edges, check_num_nodes, copy_xj,
                      e_mul_xj, expand_srcdst, mean, propagate, softmax_edge_neighbors, w_mul_xj)


def identity(x):
    return x


def relu(x):
    return torch.relu(x)


def _sigma(l) -> Callable:
    for name in ("σ", "sigma", "activation"):
        if hasattr(l, name):
            return getattr(l, name)
    return identity


def _bias(l):
    b = getattr(l, "bias", None)
    if b is None or b is False:
        return None
    return b


def _matmul(W: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """Julia `W * x` for W (Dout, Din), x (Din, N) column-major -> (Dout, N) column-major (rows @ W^T)."""
    return unrows(rows(x) @ W.t())


def _add_bias(x: torch.Tensor, b) -> torch.Tensor:
    if b is None:
        return x
    return x + b.reshape(-1, 1)


class _LinearFn(torch.autograd.Function):
    """σ.(W * x .+ b) for σ ∈ {identity, relu} through gnnb_linear / gnnb_linear_bwd (cuBLASLt GEMM with the bias and
    relu in the epilogue, fp32-emulated on bf16 tensor cores when available; hand-written relu/bias-grad pullback)."""

    @staticmethod
    def forward(ctx, x_rows, W, bias, relu_flag):
        N, Din = x_rows.shape
        Dout = W.shape[0]
        y = torch.empty((N, Dout), dtype=torch.float32, device=x_rows.device)
        Wc = W.contiguous()
        with torch.cuda.device(x_rows.device):
            _lib.check(lib.gnnb_linear(x_rows.data_ptr(), Wc.data_ptr(), None if bias is None else bias.data_ptr(),
                                       int(relu_flag), N, Din, Dout, y.data_ptr(), _stream(x_rows.device)))
        ctx.relu_flag, ctx.has_bias = bool(relu_flag), bias is not None
        ctx.save_for_backward(x_rows, Wc, y if relu_flag else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_rows, W, y = ctx.saved_tensors
        dy = dy.contiguous()
        N, Din = x_rows.shape
        Dout = W.shape[0]
        need_dx, need_dW, need_db = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        dx = torch.empty_like(x_rows) if need_dx else None
        dW = torch.empty_like(W) if need_dW else None
        db = torch.empty(Dout, dtype=torch.float32, device=dy.device) if need_db else None
        ws = torch.empty_like(dy) if ctx.relu_flag else None
        p = lambda t: None if t is None else t.data_ptr()
        with torch.cuda.device(dy.device):
            _lib.check(lib.gnnb_linear_bwd(dy.data_ptr(), p(y), x_rows.data_ptr(), W.data_ptr(), int(ctx.relu_flag), N, Din,
                                           Dout, p(ws), p(dx), p(dW), p(db), _stream(dy.device)))
        return dx, dW, db, None


class _BiasActFn(torch.autograd.Function):
    """σ.(x .+ b) on node rows for σ ∈ {identity, relu} (gnnb_bias_act / gnnb_bias_act_bwd): the closing line of the layers
    whose last step is an aggregation (GATConv, conv.jl:149).  One pass forward, one pass backward."""

    @staticmethod
    def forward(ctx, x_rows, bias, relu_flag):
        N, D = x_rows.shape
        y = torch.empty_like(x_rows)
        with torch.cuda.device(x_rows.device):
            _lib.check(lib.gnnb_bias_act(x_rows.data_ptr(), None if bias is None else bias.data_ptr(), int(relu_flag), N, D,
                                         y.data_ptr(), _stream(x_rows.device)))
        ctx.relu_flag, ctx.has_bias = bool(relu_flag), bias is not None
        ctx.save_for_backward(y if relu_flag else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        dy = dy.contiguous()
        N, D = dy.shape
        need_db = ctx.has_bias and ctx.needs_input_grad[1]
        if not ctx.relu_flag and not need_db:
            return dy, None, None
        dpre = torch.empty_like(dy) if ctx.relu_flag else dy
        db = torch.empty(D, dtype=torch.float32, device=dy.device) if need_db else None
        p = lambda t: None if t is None else t.data_ptr()
        with torch.cuda.device(dy.device):
            _lib.check(lib.gnnb_bias_act_bwd(dy.data_ptr(), p(y), int(ctx.relu_flag), N, D, p(dpre) if ctx.relu_flag else None,
                                             p(db), _stream(dy.device)))
        return dpre, db, None


def _bias_act(l, x: torch.Tensor) -> torch.Tensor:
    """`l.σ.(x .+ l.bias)` on Julia-shaped (D, N) x: the fused pass for fp32 CUDA rows with D % 4 == 0 (<= 1024) and
    σ ∈ {identity, relu}; the same arithmetic through torch otherwise."""
    sig, b = _sigma(l), _bias(l)
    xr = rows(x)
    if (x.dim() == 2 and xr.is_cuda and xr.dtype == torch.float32 and xr.is_contiguous() and xr.shape[1] % 4 == 0
            and xr.shape[1] <= 1024 and xr.data_ptr() % 16 == 0 and (sig is identity or _is_relu(sig))
            and (b is None or (b.dtype == torch.float32 and b.is_contiguous())) and (b is not None or _is_relu(sig))):
        return unrows(_BiasActFn.apply(xr, b, _is_relu(sig)))
    return sig(_add_bias(x, b))


def _is_relu(f) -> bool:
    return f in (relu, torch.relu, torch.nn.functional.relu)


def _linear(l, W: torch.Tensor, x: torch.Tensor, with_bias_act: bool) -> torch.Tensor:
    """`σ.(W * x .+ b)` (with_bias_act) or `W * x` on Julia-shaped x.  The library GEMM path needs fp32 CUDA tensors,
    Dout % 4 == 0 and σ ∈ {identity, relu}; anything else is the same arithmetic through torch."""
    sig = _sigma(l) if with_bias_act else identity
    b = _bias(l) if with_bias_act else None
    xr = rows(x)
    Dout = W.shape[0]
    fusable = (xr.is_cuda and xr.dtype == torch.float32 and W.dtype == torch.float32 and Dout % 4 == 0 and Dout <= 1024
               and (sig is identity or _is_relu(sig)) and W.shape[1] % 4 == 0)
    if fusable:
        bb = None if b is None else b.contiguous()
        return unrows(_LinearFn.apply(xr, W, bb, _is_relu(sig)))
    out = _matmul(W, x)
    return sig(_add_bias(out, b)) if with_bias_act else out


def default_norm_fn(d: torch.Tensor) -> torch.Tensor:
    """d -> 1 ./ sqrt.(d) — GraphNeuralNetworks/src/layers/conv.jl:99."""
    return 1.0 / torch.sqrt(d)


# ------------------------------------------------------------------------------------------- GCNConv
def check_gcnconv_input(g: GNNGraph, edge_weight) -> None:
    """GNNlib/src/layers/conv.jl:3-12."""
    if edge_weight is not None and edge_weight.numel() != g.num_edges:
        raise ValueError(f"Wrong number of edge weights (expected {g.num_edges} but given {edge_weight.numel()})")


def _gcn_c(g: GNNGraph) -> torch.Tensor:
    """c = 1 ./ sqrt.(degree(g; dir=:in, edge_weight=false)) on the device, cached on the (immutable) graph."""
    c = getattr(g, "_gcn_c_cache", None)
    if c is None:
        p = g.plan()
        c = torch.empty(g.num_nodes, dtype=torch.float32, device=p.device)
        with torch.cuda.device(p.device):
            _lib.check(lib.gnnb_gcn_norm(p.h, None, c.data_ptr(), _stream(p.device)))
        g._gcn_c_cache = c
    return c


def gcn_conv(l, g: GNNGraph, x: torch.Tensor, edge_weight: Optional[torch.Tensor] = None,
             norm_fn: Optional[Callable] = None, conv_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:14-72, statement for statement; the unweighted default-norm case runs the
    fused kernel (degree from rowptr, both 1/sqrt(d) scalings folded into the load/store of one pass)."""
    check_gcnconv_input(g, edge_weight)
    if conv_weight is None:
        weight = l.weight
    else:
        weight = conv_weight
        if tuple(weight.shape) != tuple(l.weight.shape):
            raise ValueError(f"The weight matrix has the wrong size. Expected {tuple(l.weight.shape)} "
                             f"but got {tuple(weight.shape)}")
    if l.add_self_loops:
        g = add_self_loops(g)
        if edge_weight is not None:
            edge_weight = torch.cat([edge_weight, torch.ones(g.num_nodes, dtype=edge_weight.dtype,
                                                             device=edge_weight.device)])
            assert edge_weight.numel() == g.num_edges
    Dout, Din = weight.shape
    if Dout < Din:
        x = _linear(l, weight, x, False)  # multiply before convolution if it is more convenient
    xj, xi = expand_srcdst(g, x)
    check_num_nodes(g, xj)
    use_w = bool(getattr(l, "use_edge_weight", False)) and g.w is not None
    if edge_weight is None and not use_w and norm_fn is None:
        plan = g.plan()
        out = unrows(_GCNPropagateFn.apply(_f32(rows(xj), plan.device), plan, None))   # c: the plan's own
    else:
        nf = norm_fn or default_norm_fn
        if edge_weight is not None:
            d = degree(g, torch.float32, dir="in", edge_weight=edge_weight)
        else:
            d = degree(g, torch.float32, dir="in", edge_weight=bool(getattr(l, "use_edge_weight", False)))
        c = nf(d)
        xs = xj * c.reshape(1, -1)
        if edge_weight is not None:
            out = propagate(e_mul_xj, g, operator.add, xj=xs, e=edge_weight)
        elif use_w:
            out = propagate(w_mul_xj, g, operator.add, xj=xs)
        else:
            out = propagate(copy_xj, g, operator.add, xj=xs)
        out = out * c.reshape(1, -1)
    if Dout >= Din:
        return _linear(l, weight, out, True)      # σ.(W * x .+ b): one GEMM with the bias/relu epilogue
    return _bias_act(l, out)


def glorot_uniform(*shape, device=None) -> torch.Tensor:
    """Flux.glorot_uniform: U(-s, s), s = sqrt(24 / (fan_in + fan_out)) / 2... = sqrt(6/(fan_in+fan_out))."""
    fan_out, fan_in = shape[0], shape[1] if len(shape) > 1 else shape[0]
    s = math.sqrt(6.0 / (fan_in + fan_out))
    return (torch.rand(*shape, device=device) * 2 - 1) * s


class GCNConv(torch.nn.Module):
    """GCNConv(in => out, σ=identity; bias=true, add_self_loops=true, use_edge_weight=false)
    — GraphNeuralNetworks/src/layers/conv.jl:77-104."""

    def __init__(self, ch_in: int, ch_out: int, sigma: Callable = identity, *, bias: bool = True,
                 add_self_loops: bool = True, use_edge_weight: bool = False, device=None):
        super().__init__()
        self.weight = torch.nn.Parameter(glorot_uniform(ch_out, ch_in, device=device))
        self.bias = torch.nn.Parameter(torch.zeros(ch_out, device=device)) if bias else None
        self.sigma = sigma
        self.add_self_loops = add_self_loops
        self.use_edge_weight = use_edge_weight

    def forward(self, g: GNNGraph, x: torch.Tensor, edge_weight=None, *, norm_fn=None, conv_weight=None):
        return gcn_conv(self, g, x, edge_weight, norm_fn, conv_weight)


# ------------------------------------------------------------------------------------------- GATConv
class _GATAggregateFn(torch.autograd.Function):
    """Fused logits -> leakyrelu -> neighbourhood softmax -> α-weighted sum: gnnb_gat_aggregate(+_bwd)."""

    @staticmethod
    def forward(ctx, Wx_rows, el_rows, er_rows, plan, slope):
        N, H, Cc = Wx_rows.shape
        out = torch.empty_like(Wx_rows)
        smax = torch.empty((N, H), dtype=torch.float32, device=Wx_rows.device)
        ssum = torch.empty((N, H), dtype=torch.float32, device=Wx_rows.device)
        with torch.cuda.device(plan.device):
            _lib.check(lib.gnnb_gat_aggregate(plan.h, Wx_rows.data_ptr(), el_rows.data_ptr(), er_rows.data_ptr(),
                                              Cc, H, slope, out.data_ptr(), None, smax.data_ptr(),
                                              ssum.data_ptr(), _stream(plan.device)))
        ctx.plan, ctx.slope, ctx.dims = plan, slope, (Cc, H)
        ctx.save_for_backward(Wx_rows, el_rows, er_rows, smax, ssum, out)
        return out

    @staticmethod
    def backward(ctx, dout):
        Wx_rows, el_rows, er_rows, smax, ssum, out = ctx.saved_tensors
        Cc, H = ctx.dims
        dout = dout.contiguous()
        dWx = torch.empty_like(Wx_rows)
        del_ = torch.empty_like(el_rows)
        der = torch.empty_like(er_rows)
        with torch.cuda.device(ctx.plan.device):
            _lib.check(lib.gnnb_gat_aggregate_bwd(ctx.plan.h, Wx_rows.data_ptr(), el_rows.data_ptr(),
                                                  er_rows.data_ptr(), smax.data_ptr(), ssum.data_ptr(),
                                                  out.data_ptr(), dout.data_ptr(), Cc, H, ctx.slope, dWx.data_ptr(),
                                                  del_.data_ptr(), der.data_ptr(), _stream(ctx.plan.device)))
        return dWx, del_, der, None, None


class _GATCoreFn(torch.autograd.Function):
    """The whole edge part of gat_conv for one projection Wx (N, H, C) and attention vector a (2C, H): per-node logit
    halves (gnnb_gat_logit_terms, one pass over Wx), then the fused logits -> leakyrelu -> neighbourhood softmax ->
    α-weighted sum (gnnb_gat_aggregate).  Backward: gnnb_gat_aggregate_bwd, then gnnb_gat_logit_terms_bwd adds the el / er
    chain into dWx in place and reduces da — no (C,H,N) temporaries, no eager broadcast-multiply-reduce."""

    @staticmethod
    def forward(ctx, Wx_rows, a, plan, slope):
        N, H, Cc = Wx_rows.shape
        dev = Wx_rows.device
        a_jl = a.detach().t().contiguous()                 # Julia (2C, H) column-major memory = rows (H, 2C)
        el = torch.empty((N, H), dtype=torch.float32, device=dev)
        er = torch.empty_like(el)
        out = torch.empty_like(Wx_rows)
        smax, ssum = torch.empty_like(el), torch.empty_like(el)
        with torch.cuda.device(plan.device):
            st = _stream(plan.device)
            _lib.check(lib.gnnb_gat_logit_terms(Wx_rows.data_ptr(), a_jl.data_ptr(), N, Cc, H, el.data_ptr(), er.data_ptr(), st))
            _lib.check(lib.gnnb_gat_aggregate(plan.h, Wx_rows.data_ptr(), el.data_ptr(), er.data_ptr(), Cc, H, slope,
                                              out.data_ptr(), None, smax.data_ptr(), ssum.data_ptr(), st))
        ctx.plan, ctx.slope, ctx.dims = plan, slope, (Cc, H)
        ctx.save_for_backward(Wx_rows, a_jl, el, er, smax, ssum, out)
        return out

    @staticmethod
    def backward(ctx, dout):
        Wx_rows, a_jl, el, er, smax, ssum, out = ctx.saved_tensors
        Cc, H = ctx.dims
        N = Wx_rows.shape[0]
        dout = dout.contiguous()
        dWx = torch.empty_like(Wx_rows)
        del_, der = torch.empty_like(el), torch.empty_like(er)
        da_jl = torch.empty_like(a_jl)
        with torch.cuda.device(ctx.plan.device):
            st = _stream(ctx.plan.device)
            _lib.check(lib.gnnb_gat_aggregate_bwd(ctx.plan.h, Wx_rows.data_ptr(), el.data_ptr(), er.data_ptr(), smax.data_ptr(),
                                                  ssum.data_ptr(), out.data_ptr(), dout.data_ptr(), Cc, H, ctx.slope,
                                                  dWx.data_ptr(), del_.data_ptr(), der.data_ptr(), st))
            _lib.check(lib.gnnb_gat_logit_terms_bwd(Wx_rows.data_ptr(), a_jl.data_ptr(), del_.data_ptr(), der.data_ptr(), N, Cc,
                                                    H, dWx.data_ptr(), da_jl.data_ptr(), st))
        return dWx, da_jl.t(), None, None


def gat_logit_fusable(chout: int, heads: int) -> bool:
    """Shapes both gnnb_gat_logit_terms and gnnb_gat_logit_terms_bwd (csrc/gatlogit.cu) cover: G = C/4 a power of two <= 32,
    C*H <= 4096, at most 8 passes of 32/G heads per warp, and a block stage of 8 warps x 2*H*C floats = 64*H*C bytes
    <= 200 KiB (config 3, 64 x 8: 4 passes of 2 heads, 32 KiB).  Other shapes take the el / er broadcasts."""
    g = chout // 4
    if not (heads >= 1 and chout % 4 == 0 and g > 0 and (g & (g - 1)) == 0 and g <= 32 and chout * heads <= 4096):
        return False
    passes = -(-heads // (32 // g))
    return passes <= 8 and 64 * heads * chout <= 200 * 1024


def gat_fusable(chout: int, heads: int) -> bool:
    """Shapes the fused GAT kernels cover (csrc/gat.cu gat_shape): C/4 a power of two <= 32 (any number of heads), or
    C a power of two <= 32 with C*H <= 128.  Everything else takes the reference's own composition."""
    def pow2(v):
        return v > 0 and (v & (v - 1)) == 0
    if chout % 4 == 0 and pow2(chout // 4) and chout // 4 <= 32:
        return True
    return pow2(chout) and chout <= 32 and chout * heads <= 128


def gat_message(l, Wxi, Wxj, e):
    """GNNlib/src/layers/conv.jl:152-167 (generic path; arrays are (C, H, E))."""
    _, chout = l.channel
    heads = l.heads
    if e is None:
        Wxx = torch.cat([Wxi, Wxj], dim=0)
    else:
        We = l.dense_e(e)
        We = _jl_reshape3(We, chout, heads)  # chout × nheads × nedges
        Wxx = torch.cat([Wxi, Wxj, We], dim=0)
    aWW = (l.a.unsqueeze(-1) * Wxx).sum(dim=0, keepdim=True)  # 1 × nheads × nedges
    logα = torch.nn.functional.leaky_relu(aWW, float(l.negative_slope))
    return {"logα": logα, "Wxj": Wxj}


def _jl_reshape3(x: torch.Tensor, c: int, h: int) -> torch.Tensor:
    """Julia reshape((c*h, N) -> (c, h, N)) on column-major data = view rows (N, c*h) as (N, h, c)."""
    r = rows(x)
    return unrows(r.reshape(r.shape[0], h, c))


def gat_conv(l, g: GNNGraph, x: torch.Tensor, e: Optional[torch.Tensor] = None, *, fused: bool = True):
    """GNNlib/src/layers/conv.jl:112-150.  Without edge features the edge part (two gathers, vcat, logits,
    neighbourhood softmax, α .* Wxj, scatter) is ONE fused kernel; with edge features (or fused=False) the
    reference's own composition runs on the generic gather/scatter kernels."""
    check_num_nodes(g, x)
    dense_e = getattr(l, "dense_e", None)
    assert not (e is None and dense_e is not None), "Input edge features required for this layer"
    assert not (e is not None and dense_e is None), "Input edge features were not specified in the layer constructor"
    xj, xi = expand_srcdst(g, x)
    if l.add_self_loops:
        assert e is None, "Using edge features and setting add_self_loops=true at the same time is not yet supported."
        g = add_self_loops(g)
    _, chout = l.channel
    heads = l.heads
    Wxj = _jl_reshape3(l.dense_x(xj), chout, heads)  # chout × heads × N
    Wxi = Wxj
    if xi is not xj:
        Wxi = _jl_reshape3(l.dense_x(xi), chout, heads)
    if fused and e is None and xi is xj and gat_fusable(chout, heads) and float(getattr(l, "dropout", 0.0) or 0.0) == 0.0:
        plan = g.plan()
        Wr = _f32(rows(Wxj), plan.device)                       # (N, H, C)
        if Wr.data_ptr() % 16 != 0:                             # a misaligned view: the fused kernels take 16 B-aligned rows
            Wr = Wr.clone()
        a = l.a                                                 # (2C, H)
        if gat_logit_fusable(chout, heads) and a.dtype == torch.float32:
            out = unrows(_GATCoreFn.apply(Wr, a, plan, float(l.negative_slope)))
        else:
            el = (Wr * a[:chout, :].t().unsqueeze(0)).sum(-1)   # (N, H): rows 1..C pair with the target
            er = (Wr * a[chout:, :].t().unsqueeze(0)).sum(-1)   # rows C+1..2C pair with the source
            out = unrows(_GATAggregateFn.apply(Wr, el.contiguous(), er.contiguous(), plan, float(l.negative_slope)))
    else:
        m = apply_edges(Fix1(gat_message, l), g, Wxi, Wxj, e)
        α = softmax_edge_neighbors(g, m["logα"])
        p = float(getattr(l, "dropout", 0.0) or 0.0)
        if p > 0:
            α = torch.nn.functional.dropout(α, p, training=getattr(l, "training", True))
        β = α * m["Wxj"]
        out = aggregate_neighbors(g, operator.add, β)
    if not l.concat:
        out = out.mean(dim=1, keepdim=True)
    out = unrows(rows(out).reshape(out.shape[-1], -1))  # reshape(x, :, size(x, 3))
    return _bias_act(l, out)


class _Dense(torch.nn.Module):
    """Flux.Dense(in => out; bias) on Julia-shaped arrays."""

    def __init__(self, ch_in, ch_out, bias=True, device=None):
        super().__init__()
        self.weight = torch.nn.Parameter(glorot_uniform(ch_out, ch_in, device=device))
        self.bias = torch.nn.Parameter(torch.zeros(ch_out, device=device)) if bias else None

    def forward(self, x):
        return _linear(self, self.weight, x, True)     # W * x .+ b (σ = identity)


class GATConv(torch.nn.Module):
    """GATConv(in => out, σ=identity; heads=1, concat=true, negative_slope=0.2, add_self_loops=true, dropout=0)
    — GraphNeuralNetworks/src/layers/conv.jl:309-346 (ein = 0: no edge features)."""

    def __init__(self, ch_in: int, ch_out: int, sigma: Callable = identity, *, heads: int = 1,
                 concat: bool = True, negative_slope: float = 0.2, bias: bool = True,
                 add_self_loops: bool = True, dropout: float = 0.0, device=None):
        super().__init__()
        self.dense_x = _Dense(ch_in, ch_out * heads, bias=False, device=device)
        self.dense_e = None
        self.a = torch.nn.Parameter(glorot_uniform(2 * ch_out, heads, device=device))
        nb = ch_out * heads if concat else ch_out
        self.bias = torch.nn.Parameter(torch.zeros(nb, device=device)) if bias else None
        self.sigma = sigma
        self.negative_slope = negative_slope
        self.channel = (ch_in, ch_out)
        self.heads = heads
        self.concat = concat
        self.add_self_loops = add_self_loops
        self.dropout = dropout

    def forward(self, g: GNNGraph, x: torch.Tensor, e=None, **kw):
        return gat_conv(self, g, x, e, **kw)


# ------------------------------------------------------------------------------------------ SAGEConv
class _Linear2Fn(torch.autograd.Function):
    """σ.(W * vcat(x1, x2) .+ b) for σ ∈ {identity, relu} through gnnb_linear2 / gnnb_linear2_bwd: the two column blocks
    of W meet x1 and x2 in two accumulating passes of the tcgen05 kernel — no (Din1+Din2, N) vcat temporary."""

    @staticmethod
    def forward(ctx, x1, x2, W, bias, relu_flag):
        N, D1 = x1.shape
        D2 = x2.shape[1]
        Dout = W.shape[0]
        y = torch.empty((N, Dout), dtype=torch.float32, device=x1.device)
        Wc = W.contiguous()
        with torch.cuda.device(x1.device):
            _lib.check(lib.gnnb_linear2(x1.data_ptr(), x2.data_ptr(), Wc.data_ptr(), None if bias is None else bias.data_ptr(),
                                        int(relu_flag), N, D1, D2, Dout, y.data_ptr(), _stream(x1.device)))
        ctx.relu_flag, ctx.has_bias = bool(relu_flag), bias is not None
        ctx.save_for_backward(x1, x2, Wc, y if relu_flag else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x1, x2, W, y = ctx.saved_tensors
        dy = dy.contiguous()
        N, D1 = x1.shape
        D2, Dout = x2.shape[1], W.shape[0]
        dx1 = torch.empty_like(x1) if ctx.needs_input_grad[0] else None
        dx2 = torch.empty_like(x2) if ctx.needs_input_grad[1] else None
        dW = torch.empty_like(W) if ctx.needs_input_grad[2] else None
        db = torch.empty(Dout, dtype=torch.float32, device=dy.device) if (ctx.has_bias and ctx.needs_input_grad[3]) else None
        ws = torch.empty_like(dy) if ctx.relu_flag else None
        p = lambda t: None if t is None else t.data_ptr()
        with torch.cuda.device(dy.device):
            _lib.check(lib.gnnb_linear2_bwd(dy.data_ptr(), p(y), x1.data_ptr(), x2.data_ptr(), W.data_ptr(), int(ctx.relu_flag), N,
                                            D1, D2, Dout, p(ws), p(dx1), p(dx2), p(dW), p(db), _stream(dy.device)))
        return dx1, dx2, dW, db, None


def sage_conv(l, g: GNNGraph, x: torch.Tensor) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:277-283: σ.(W * vcat(xi, propagate(copy_xj, g, aggr, xj)) .+ b).
    W is (out, 2·in): its first `in` columns multiply x_i, the rest the aggregated neighbours."""
    check_num_nodes(g, x)
    xj, xi = expand_srcdst(g, x)
    m = propagate(copy_xj, g, l.aggr, xj=xj)
    W = l.weight
    sig, b = _sigma(l), _bias(l)
    r1, r2 = rows(xi), rows(m)
    D1, D2, Dout = r1.shape[1], r2.shape[1], W.shape[0]
    if (r1.is_cuda and r1.dtype == torch.float32 and W.dtype == torch.float32 and Dout == 128 and D1 % 32 == 0 and D2 % 32 == 0
            and D1 <= 128 and D2 <= 128 and (sig is identity or _is_relu(sig))):
        # the two column blocks of W in two accumulating tcgen05 passes: no vcat temporary
        return unrows(_Linear2Fn.apply(r1.contiguous(), r2.contiguous(), W, None if b is None else b.contiguous(), _is_relu(sig)))
    xm = unrows(torch.cat([r1, r2], dim=1))                   # vcat(xi, m): (2·in, N)
    return _linear(l, W, xm, True)                            # σ.(W * vcat(xi, m) .+ b): one GEMM, bias/σ in the epilogue


class SAGEConv(torch.nn.Module):
    """SAGEConv(in => out, σ=identity; aggr=mean, bias=true) — GraphNeuralNetworks/src/layers/conv.jl:770-787."""

    def __init__(self, ch_in: int, ch_out: int, sigma: Callable = identity, *, aggr=mean, bias: bool = True,
                 device=None):
        super().__init__()
        self.weight = torch.nn.Parameter(glorot_uniform(ch_out, 2 * ch_in, device=device))
        self.bias = torch.nn.Parameter(torch.zeros(ch_out, device=device)) if bias else None
        self.sigma = sigma
        self.aggr = aggr

    def forward(self, g: GNNGraph, x: torch.Tensor):
        return sage_conv(self, g, x)


# ------------------------------------------------------------------ layers that re-parameterise the same kernels (§8f rank 1)
def graph_conv(l, g: GNNGraph, x: torch.Tensor) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:102-108: σ.(W1*xi .+ W2*propagate(copy_xj, g, aggr, xj) .+ b)."""
    check_num_nodes(g, x)
    xj, xi = expand_srcdst(g, x)
    m = propagate(copy_xj, g, l.aggr, xj=xj)
    out = unrows(torch.addmm(rows(xi) @ l.weight1.t(), rows(m), l.weight2.t()))
    return _bias_act(l, out)


def gin_conv(l, g: GNNGraph, x: torch.Tensor) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:250-256: nn((1 + ϵ) .* xi .+ propagate(copy_xj, g, aggr, xj))."""
    check_num_nodes(g, x)
    xj, xi = expand_srcdst(g, x)
    m = propagate(copy_xj, g, l.aggr, xj=xj)
    eps = 0.0
    for name in ("\u03f5", "\u03b5", "eps"):     # ϵ (the reference's field; Python NFKC-normalises it to ε in identifiers)
        if hasattr(l, name):
            eps = getattr(l, name)
            break
    return l.nn((1 + eps) * xi + m)


def sgc_conv(l, g: GNNGraph, x: torch.Tensor, edge_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:407-448 (SGConv): k rounds of the normalised GCN propagate around one W; the
    unweighted case is k launches of the fused kernel (both 1/sqrt(d) scalings folded in)."""
    if edge_weight is not None:
        assert edge_weight.numel() == g.num_edges, \
            f"Wrong number of edge weights (expected {g.num_edges} but given {edge_weight.numel()})"
    if l.add_self_loops:
        g = add_self_loops(g)
        if edge_weight is not None:
            edge_weight = torch.cat([edge_weight, torch.ones(g.num_nodes, dtype=edge_weight.dtype, device=edge_weight.device)])
    W = l.weight
    Dout, Din = W.shape
    if Dout < Din:
        x = _linear(l, W, x, False)
    use_w = bool(getattr(l, "use_edge_weight", False)) and g.w is not None
    if edge_weight is None and not use_w:
        plan = g.plan()
        xr = _f32(rows(x), plan.device)
        c = _gcn_c(g)
        for _ in range(int(l.k)):
            xr = _GCNPropagateFn.apply(xr, plan, c)
        x = unrows(xr)
    else:
        d = degree(g, torch.float32, dir="in", edge_weight=edge_weight if edge_weight is not None else True)
        c = (1.0 / torch.sqrt(d)).reshape(1, -1)
        for _ in range(int(l.k)):
            x = x * c
            x = (propagate(e_mul_xj, g, operator.add, xj=x, e=edge_weight) if edge_weight is not None
                 else propagate(w_mul_xj, g, operator.add, xj=x))
            x = x * c
    if Dout >= Din:
        x = _linear(l, W, x, False)
    return _add_bias(x, _bias(l))


def agnn_conv(l, g: GNNGraph, x: torch.Tensor) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:337-352: cosine-similarity attention, neighbourhood softmax, weighted sum."""
    check_num_nodes(g, x)
    if l.add_self_loops:
        g = add_self_loops(g)
    from .msgpass import xi_dot_xj
    xn = x / torch.sqrt((x ** 2).sum(dim=0, keepdim=True))
    cos_dist = apply_edges(xi_dot_xj, g, xi=xn, xj=xn)
    alpha = softmax_edge_neighbors(g, l.β * cos_dist if hasattr(l, "β") else l.beta * cos_dist)
    return propagate(lambda xi, xj, a: a * xj, g, operator.add, xj=x, e=alpha)


def _k_hop_gcn(l, g: GNNGraph, x: torch.Tensor, edge_weight, each_hop: Callable) -> None:
    """The loop sg_conv and tag_conv share (conv.jl:521-536, 655-682): k rounds of  x <- c' .* A(c' .* x)  with
    c = 1/sqrt(in-degree); `each_hop(i, x)` sees the features after round i.  Unweighted graphs take the fused GCN
    kernel (both scalings folded into its load and store)."""
    use_w = bool(getattr(l, "use_edge_weight", False)) and g.w is not None
    if edge_weight is None and not use_w:
        plan = g.plan()
        xr = _f32(rows(x), plan.device)
        c = _gcn_c(g)
        for i in range(int(l.k)):
            xr = _GCNPropagateFn.apply(xr, plan, c)
            each_hop(i, unrows(xr))
        return
    d = degree(g, torch.float32, dir="in", edge_weight=edge_weight if edge_weight is not None else True)
    c = (1.0 / torch.sqrt(d)).reshape(1, -1)
    for i in range(int(l.k)):
        x = x * c
        x = (propagate(e_mul_xj, g, operator.add, xj=x, e=edge_weight) if edge_weight is not None
             else propagate(w_mul_xj, g, operator.add, xj=x))
        x = x * c
        each_hop(i, x)


def _loops_and_weights(l, g: GNNGraph, edge_weight):
    if edge_weight is not None:
        assert edge_weight.numel() == g.num_edges, \
            f"Wrong number of edge weights (expected {g.num_edges} but given {edge_weight.numel()})"
    if l.add_self_loops:
        g = add_self_loops(g)
        if edge_weight is not None:
            edge_weight = torch.cat([edge_weight, torch.ones(g.num_nodes, dtype=edge_weight.dtype,
                                                             device=edge_weight.device)])
            assert edge_weight.numel() == g.num_edges
    return g, edge_weight


def sg_conv(l, g: GNNGraph, x: torch.Tensor, edge_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:501-543 (SGConv): W applied on the cheaper side of k normalised propagation rounds."""
    g, edge_weight = _loops_and_weights(l, g, edge_weight)
    W = l.weight
    Dout, Din = W.shape
    if Dout < Din:
        x = _linear(l, W, x, False)
    last = [x]
    _k_hop_gcn(l, g, x, edge_weight, lambda i, h: last.__setitem__(0, h))
    x = last[0]
    if Dout >= Din:
        x = _linear(l, W, x, False)
    return _add_bias(x, _bias(l))


def tag_conv(l, g: GNNGraph, x: torch.Tensor, edge_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:634-686 (TAGConv), as the reference computes it: after round i the running sum
    S_i = Σ_{j<=i} Â^j x is multiplied by the ONE weight matrix and accumulated:  Σ_i W S_i  (+ bias)."""
    g, edge_weight = _loops_and_weights(l, g, edge_weight)
    W = l.weight
    state = {"pow": None, "total": None}

    def hop(i, h):
        if i == 0:
            state["pow"] = h
            state["total"] = _linear(l, W, h, False)
        else:
            state["pow"] = state["pow"] + h
            state["total"] = state["total"] + _linear(l, W, state["pow"], False)

    _k_hop_gcn(l, g, x, edge_weight, hop)
    if state["total"] is None:            # k = 0: the reference returns 0 .+ bias
        b = _bias(l)
        return torch.zeros((), dtype=x.dtype, device=x.device) if b is None else b.clone()
    return _add_bias(state["total"], _bias(l))


class _GRUCell(torch.nn.Module):
    """Flux.GRUCell(in => out) on Julia-shaped (D, N) arrays; returns (h', h') like Flux's cell.
        r = σ(Wi_r x + Wh_r h + b_r);  z = σ(Wi_z x + Wh_z h + b_z);  h~ = tanh(Wi_h x + r .* (Wh_h h) + b_h)
        h' = (1 - z) .* h~ + z .* h"""

    def __init__(self, ch_in: int, ch_out: int, device=None):
        super().__init__()
        self.Wi = torch.nn.Parameter(glorot_uniform(3 * ch_out, ch_in, device=device))
        self.Wh = torch.nn.Parameter(glorot_uniform(3 * ch_out, ch_out, device=device))
        self.b = torch.nn.Parameter(torch.zeros(3 * ch_out, device=device))
        self.ch_out = ch_out

    def forward(self, x, h):
        o = self.ch_out
        gx = _matmul(self.Wi, x)
        gh = _matmul(self.Wh, h)
        b = self.b.reshape(-1, 1)
        r = torch.sigmoid(gx[:o] + gh[:o] + b[:o])
        z = torch.sigmoid(gx[o:2 * o] + gh[o:2 * o] + b[o:2 * o])
        hc = torch.tanh(gx[2 * o:] + r * gh[2 * o:] + b[2 * o:])
        hn = (1 - z) * hc + z * h
        return hn, hn


def gated_graph_conv(l, g: GNNGraph, x: torch.Tensor) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:218-233: zero-pad x to `dims`, then num_layers rounds of
    m = propagate(copy_xj, g, aggr, xj = W_i * h);  h = gru(m, h).   l.weight is (dims, dims, num_layers)."""
    check_num_nodes(g, x)
    m_in, n = x.shape
    assert m_in <= l.dims, "number of input features must be less or equal to output features."
    if m_in < l.dims:
        x = unrows(torch.cat([rows(x), torch.zeros(n, l.dims - m_in, dtype=x.dtype, device=x.device)], dim=1))
    h = x
    for i in range(int(l.num_layers)):
        m = _linear(l, l.weight[:, :, i], h, False)
        m = propagate(copy_xj, g, l.aggr, xj=m)
        _, h = l.gru(m, h)
    return h


def gatv2_message(l, Wxi, Wxj, e):
    """GNNlib/src/layers/conv.jl:203-214 (arrays are (C, H, E))."""
    _, chout = l.channel
    Wx = Wxi + Wxj
    if e is not None:
        Wx = Wx + _jl_reshape3(l.dense_e(e), chout, l.heads)
    logα = (l.a.unsqueeze(-1) * torch.nn.functional.leaky_relu(Wx, float(l.negative_slope))).sum(dim=0, keepdim=True)
    return {"logα": logα, "Wxj": Wxj}


def _attention_tail(l, out: torch.Tensor) -> torch.Tensor:
    """`!concat -> mean over heads; reshape(x, :, N); σ.(x .+ bias)` shared by gat_conv and gatv2_conv."""
    if not l.concat:
        out = out.mean(dim=1, keepdim=True)
    out = unrows(rows(out).reshape(out.shape[-1], -1))
    return _bias_act(l, out)


def gatv2_conv(l, g: GNNGraph, x: torch.Tensor, e: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:171-201.  The logit a·leakyrelu(W_i x_i + W_j x_j) does not split into per-node
    terms, so the edge part is the reference's composition on the gather / neighbourhood-softmax / scatter kernels."""
    check_num_nodes(g, x)
    dense_e = getattr(l, "dense_e", None)
    assert not (e is None and dense_e is not None), "Input edge features required for this layer"
    assert not (e is not None and dense_e is None), "Input edge features were not specified in the layer constructor"
    xj, xi = expand_srcdst(g, x)
    if l.add_self_loops:
        assert e is None, "Using edge features and setting add_self_loops=true at the same time is not yet supported."
        g = add_self_loops(g)
    _, chout = l.channel
    Wxi = _jl_reshape3(l.dense_i(xi), chout, l.heads)
    Wxj = _jl_reshape3(l.dense_j(xj), chout, l.heads)
    m = apply_edges(Fix1(gatv2_message, l), g, Wxi, Wxj, e)
    α = softmax_edge_neighbors(g, m["logα"])
    p = float(getattr(l, "dropout", 0.0) or 0.0)
    if p > 0:
        α = torch.nn.functional.dropout(α, p, training=getattr(l, "training", True))
    out = aggregate_neighbors(g, operator.add, α * m["Wxj"])
    return _attention_tail(l, out)


def transformer_message_uij(l, xi, xj, e):
    """GNNlib/src/layers/conv.jl:614-621."""
    key = xj["W4x"]
    if e["W6e"] is not None:
        key = key + e["W6e"]
    return (xi["W3x"] * key).sum(dim=0, keepdim=True) / l.sqrt_out


def transformer_message_main(xi, xj, e):
    """GNNlib/src/layers/conv.jl:623-629."""
    val = xj["W2x"]
    if e["W6e"] is not None:
        val = val + e["W6e"]
    return e["α"] * val


def transformer_conv(l, g: GNNGraph, x: torch.Tensor, e: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GNNlib/src/layers/conv.jl:553-612: multi-head dot-product attention over each in-neighbourhood, then the
    root-weight / gating / skip / batch-norm / feed-forward tail (dense per-node work, left to torch like Flux's)."""
    check_num_nodes(g, x)
    if l.add_self_loops:
        g = add_self_loops(g)
    out = l.channels[1]
    heads = l.heads
    W1x = l.W1(x) if l.W1 is not None else None
    W2x = _jl_reshape3(l.W2(x), out, heads)
    W3x = _jl_reshape3(l.W3(x), out, heads)
    W4x = _jl_reshape3(l.W4(x), out, heads)
    W6e = _jl_reshape3(l.W6(e), out, heads) if l.W6 is not None else None
    m = apply_edges(Fix1(transformer_message_uij, l), g, xi={"W3x": W3x}, xj={"W4x": W4x}, e={"W6e": W6e})
    α = softmax_edge_neighbors(g, m)
    h = propagate(transformer_message_main, g, operator.add, xi={"W3x": W3x}, xj={"W2x": W2x}, e={"W6e": W6e, "α": α})
    if l.concat:
        h = unrows(rows(h).reshape(h.shape[-1], out * heads))
    else:
        h = h.mean(dim=1)                                          # (out, N)
    if W1x is not None:
        if l.W5 is not None:
            β = l.W5(torch.cat([h, W1x, h - W1x], dim=0))
            h = β * W1x + (1.0 - β) * h
        else:
            h = h + W1x
    if l.skip_connection:
        assert h.shape[0] == x.shape[0], \
            "In-channels must correspond to out-channels * heads if skip_connection is used"
        h = h + x
    if l.BN1 is not None:
        h = l.BN1(h)
    if l.FF is not None:
        h1 = h
        h = l.FF(h)
        if l.skip_connection:
            h = h + h1
        if l.BN2 is not None:
            h = l.BN2(h)
    return h


# ------------------------------------------------------------------ parameter holders for the layers above
class _DenseAct(_Dense):
    """Flux.Dense(in => out, σ; bias): `_linear` reads the activation from the `sigma` field."""

    def __init__(self, ch_in, ch_out, sigma: Callable = identity, bias=True, device=None):
        super().__init__(ch_in, ch_out, bias=bias, device=device)
        self.sigma = sigma


class _BatchNorm(torch.nn.Module):
    """Flux.BatchNorm(ch) on (ch, N) Julia-shaped arrays (normalises over the node dimension)."""

    def __init__(self, ch, device=None):
        super().__init__()
        self.bn = torch.nn.BatchNorm1d(ch, eps=1e-5, momentum=0.1, device=device)

    def forward(self, x):
        return unrows(self.bn(rows(x)))


class GraphConv(torch.nn.Module):
    """GraphConv(in => out, σ=identity; aggr=+, bias=true) — GraphNeuralNetworks/src/layers/conv.jl:226-251."""

    def __init__(self, ch_in, ch_out, sigma: Callable = identity, *, aggr=operator.add, bias=True, device=None):
        super().__init__()
        self.weight1 = torch.nn.Parameter(glorot_uniform(ch_out, ch_in, device=device))
        self.weight2 = torch.nn.Parameter(glorot_uniform(ch_out, ch_in, device=device))
        self.bias = torch.nn.Parameter(torch.zeros(ch_out, device=device)) if bias else None
        self.sigma, self.aggr = sigma, aggr

    def forward(self, g, x):
        return graph_conv(self, g, x)


class GINConv(torch.nn.Module):
    """GINConv(nn, ϵ; aggr=+) — GraphNeuralNetworks/src/layers/conv.jl:628-640 (ϵ is not trainable there either)."""

    def __init__(self, nn: Callable, eps: float = 0.0, *, aggr=operator.add):
        super().__init__()
        self.nn, self.eps, self.aggr = nn, float(eps), aggr

    def forward(self, g, x):
        return gin_conv(self, g, x)


class AGNNConv(torch.nn.Module):
    """AGNNConv(; init_beta=1, trainable=true, add_self_loops=true) — GraphNeuralNetworks/src/layers/conv.jl:988-1003."""

    def __init__(self, *, init_beta: float = 1.0, trainable: bool = True, add_self_loops: bool = True, device=None):
        super().__init__()
        b = torch.tensor([float(init_beta)], device=device)
        self.beta = torch.nn.Parameter(b) if trainable else b
        self.add_self_loops = add_self_loops
        self.trainable = trainable

    def forward(self, g, x):
        return agnn_conv(self, g, x)


class SGConv(torch.nn.Module):
    """SGConv(in => out, k=1; bias=true, add_self_loops=true, use_edge_weight=false) — conv.jl:1197-1222."""

    def __init__(self, ch_in, ch_out, k: int = 1, *, bias=True, add_self_loops=True, use_edge_weight=False,
                 device=None):
        super().__init__()
        self.weight = torch.nn.Parameter(glorot_uniform(ch_out, ch_in, device=device))
        self.bias = torch.nn.Parameter(torch.zeros(ch_out, device=device)) if bias else None
        self.k, self.add_self_loops, self.use_edge_weight = int(k), add_self_loops, use_edge_weight

    def forward(self, g, x, edge_weight=None):
        return sg_conv(self, g, x, edge_weight)


class TAGConv(SGConv):
    """TAGConv(in => out, k=3; bias=true, add_self_loops=true, use_edge_weight=false) — conv.jl:1265-1286."""

    def __init__(self, ch_in, ch_out, k: int = 3, **kw):
        super().__init__(ch_in, ch_out, k, **kw)

    def forward(self, g, x, edge_weight=None):
        return tag_conv(self, g, x, edge_weight)


class GatedGraphConv(torch.nn.Module):
    """GatedGraphConv(out, num_layers; aggr=+) — GraphNeuralNetworks/src/layers/conv.jl:515-530."""

    def __init__(self, dims: int, num_layers: int, *, aggr=operator.add, device=None):
        super().__init__()
        w = torch.stack([glorot_uniform(dims, dims, device=device) for _ in range(num_layers)], dim=2)
        self.weight = torch.nn.Parameter(w)                       # (dims, dims, num_layers)
        self.gru = _GRUCell(dims, dims, device=device)
        self.dims, self.num_layers, self.aggr = dims, num_layers, aggr

    def forward(self, g, x):
        return gated_graph_conv(self, g, x)


class GATv2Conv(torch.nn.Module):
    """GATv2Conv(in => out, σ=identity; heads=1, concat=true, negative_slope=0.2, bias=true, add_self_loops=true,
    dropout=0) and the (in, ein) => out form — GraphNeuralNetworks/src/layers/conv.jl:413-462."""

    def __init__(self, ch_in, ch_out: int, sigma: Callable = identity, *, heads: int = 1, concat: bool = True,
                 negative_slope: float = 0.2, bias: bool = True, add_self_loops: bool = True, dropout: float = 0.0,
                 device=None):
        super().__init__()
        cin, ein = ch_in if isinstance(ch_in, tuple) else (ch_in, 0)
        if add_self_loops:
            assert ein == 0, "Using edge features and setting add_self_loops=true at the same time is not yet supported."
        self.dense_i = _Dense(cin, ch_out * heads, bias=bias, device=device)
        self.dense_j = _Dense(cin, ch_out * heads, bias=False, device=device)
        self.dense_e = _Dense(ein, ch_out * heads, bias=False, device=device) if ein > 0 else None
        nb = ch_out * heads if concat else ch_out
        self.bias = torch.nn.Parameter(torch.zeros(nb, device=device)) if bias else None
        self.a = torch.nn.Parameter(glorot_uniform(ch_out, heads, device=device))
        self.sigma, self.negative_slope = sigma, negative_slope
        self.channel = ((cin, ein), ch_out)
        self.heads, self.concat, self.add_self_loops, self.dropout = heads, concat, add_self_loops, dropout

    def forward(self, g, x, e=None):
        return gatv2_conv(self, g, x, e)


class TransformerConv(torch.nn.Module):
    """TransformerConv((in, ein) => out; heads=1, concat=true, add_self_loops=false, bias_qkv=true, bias_root=true,
    root_weight=true, gating=false, skip_connection=false, batch_norm=false, ff_channels=0)
    — GraphNeuralNetworks/src/layers/conv.jl:1473-1539."""

    def __init__(self, ch_in, ch_out: int, *, heads: int = 1, concat: bool = True, add_self_loops: bool = False,
                 bias_qkv: bool = True, bias_root: bool = True, root_weight: bool = True, gating: bool = False,
                 skip_connection: bool = False, batch_norm: bool = False, ff_channels: int = 0, device=None):
        super().__init__()
        cin, ein = ch_in if isinstance(ch_in, tuple) else (ch_in, 0)
        if add_self_loops:
            assert ein == 0, "Using edge features and setting add_self_loops=true at the same time is not yet supported."
        out_mha = ch_out * (heads if concat else 1)
        self.W1 = _Dense(cin, out_mha, bias=bias_root, device=device) if root_weight else None
        self.W2 = _Dense(cin, ch_out * heads, bias=bias_qkv, device=device)
        self.W3 = _Dense(cin, ch_out * heads, bias=bias_qkv, device=device)
        self.W4 = _Dense(cin, ch_out * heads, bias=bias_qkv, device=device)
        self.W5 = _DenseAct(3 * out_mha, 1, torch.sigmoid, bias=False, device=device) if gating else None
        self.W6 = _Dense(ein, ch_out * heads, bias=bias_qkv, device=device) if ein > 0 else None
        self.FF = (torch.nn.Sequential(_DenseAct(out_mha, ff_channels, relu, device=device),
                                       _Dense(ff_channels, out_mha, device=device)) if ff_channels > 0 else None)
        self.BN1 = _BatchNorm(out_mha, device=device) if batch_norm else None
        self.BN2 = _BatchNorm(out_mha, device=device) if (batch_norm and ff_channels > 0) else None
        self.channels = ((cin, ein), ch_out)
        self.heads, self.add_self_loops, self.concat, self.skip_connection = heads, add_self_loops, concat, skip_connection
        self.sqrt_out = math.sqrt(ch_out)

    def forward(self, g, x, e=None):
        return transformer_conv(self, g, x, e)
