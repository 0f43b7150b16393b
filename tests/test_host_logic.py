"""Host-side mirror of the reference interface: size checks, containers, layout helpers, batching.
CPU only (no kernels run)."""
import operator
import sys

import numpy as np
import pytest
import torch


def test_colmajor_rows_roundtrip(gnn):
    x = torch.arange(12, dtype=torch.float32).reshape(3, 4)        # Julia (3, 4)
    xc = gnn.colmajor(x)
    assert xc.shape == (3, 4) and xc.stride() == (1, 3) and torch.equal(xc, x)
    r = gnn.rows(xc)
    assert r.shape == (4, 3) and r.is_contiguous() and r.data_ptr() == xc.data_ptr()   # zero copy
    assert torch.equal(gnn.unrows(r), x)
    z = gnn.jl_zeros(2, 3, 5)
    assert z.shape == (2, 3, 5) and z.stride() == (1, 2, 6)
    assert gnn.rows(z).shape == (5, 3, 2)


def test_graph_constructors(gnn):
    g = gnn.GNNGraph([1, 1, 2, 3], [2, 2, 2, 4])
    assert (g.num_nodes, g.num_edges) == (4, 4)
    g = gnn.GNNGraph(([1, 2], [2, 3], [0.5, 1.5]), num_nodes=5)
    assert g.num_nodes == 5 and g.w.tolist() == [0.5, 1.5]
    # adjacency matrix: A[i,j] != 0 <=> edge i -> j, column-major order (GNNlib/test/test_module.jl:153-178)
    adj1 = [[0, 1, 0, 1], [1, 0, 1, 0], [0, 1, 0, 1], [1, 0, 1, 0]]
    g = gnn.GNNGraph(np.array(adj1))
    s, t = gnn.edge_index(g)
    assert s.tolist() == [2, 4, 1, 3, 2, 4, 1, 3] and t.tolist() == [1, 1, 2, 2, 3, 3, 4, 4]
    with pytest.raises(AssertionError):
        gnn.GNNGraph([1, 2], [1, 2, 3])


def test_size_checks_raise_assertion_error(gnn):
    # GNNlib/test/msgpass.jl:55-66, 118-125: wrong last dimension -> AssertionError
    g = gnn.GNNGraph(np.array([[0, 1, 0, 1], [1, 0, 1, 0], [0, 1, 0, 1], [1, 0, 1, 0]]))
    x = torch.rand(3, g.num_nodes - 1)
    with pytest.raises(AssertionError):
        gnn.apply_edges(gnn.copy_xj, g, xj=x)
    with pytest.raises(AssertionError):
        gnn.apply_edges(gnn.copy_xj, g, xi=x)
    xs = {"a": torch.rand(3, g.num_nodes), "b": torch.rand(3, g.num_nodes + 1)}
    with pytest.raises(AssertionError):
        gnn.apply_edges(gnn.copy_xj, g, xj=xs)
    e = torch.rand(3, g.num_edges - 1)
    with pytest.raises(AssertionError):
        gnn.apply_edges(gnn.copy_xj, g, e=e)
    with pytest.raises(AssertionError):
        gnn.aggregate_neighbors(g, operator.add, torch.rand(2, g.num_edges - 1))
    with pytest.raises(AssertionError):
        gnn.aggregate_neighbors(g, operator.add, (torch.rand(2, g.num_edges + 1), None))
    with pytest.raises(AssertionError):
        gnn.propagate(gnn.copy_xj, g, operator.add, xj=x)


def test_aggr_codes(gnn):
    from gnnb200.msgpass import _aggr_code
    L = gnn._lib
    assert _aggr_code(operator.add) == L.SUM == _aggr_code("+")
    assert _aggr_code(gnn.mean) == L.MEAN and _aggr_code(max) == L.MAX and _aggr_code(min) == L.MIN
    with pytest.raises(ValueError):
        _aggr_code(operator.mul)


def test_message_functions(gnn):
    xi, xj = torch.rand(3, 5), torch.rand(3, 5)
    e = torch.rand(5)
    assert gnn.copy_xj(xi, xj, e) is xj and gnn.copy_xi(xi, xj, e) is xi
    assert torch.allclose(gnn.xi_dot_xj(xi, xj, None), (xi * xj).sum(0, keepdim=True))
    assert torch.equal(gnn.xi_sub_xj(xi, xj, None), xi - xj) and torch.equal(gnn.xj_sub_xi(xi, xj, None), xj - xi)
    assert torch.equal(gnn.e_mul_xj(xi, xj, e), e.reshape(1, 5) * xj)
    assert torch.equal(gnn.w_mul_xj(xi, xj, e), e.reshape(1, 5) * xj)
    assert gnn.w_mul_xj(xi, xj, None) is xj
    x3 = torch.rand(2, 3, 5)
    assert gnn.w_mul_xj(None, x3, e).shape == (2, 3, 5)
    assert gnn.Fix1(lambda a, b, c: (a, b, c), 1)(2, 3) == (1, 2, 3)
    with pytest.raises(ValueError):
        gnn.expand_srcdst(None, torch.rand(3))


def test_batch_offsets(gnn):
    # GNNGraphs/test/transform.jl:19-54: ids offset by cumulative node counts; graph_indicator 1,1,..,2,..
    rng = np.random.default_rng(0)

    def ring(n):
        s = np.arange(1, n + 1)
        return gnn.GNNGraph(s, np.roll(s, -1), ndata={"x": gnn.colmajor(torch.rand(16, n))})

    g1, g2, g3 = ring(10), ring(4), ring(7)
    g123 = gnn.batch([g1, g2, g3])
    assert g123.graph_indicator.tolist() == [1] * 10 + [2] * 4 + [3] * 7
    s, t = gnn.edge_index(g123)
    assert s.tolist() == g1.s.tolist() + (10 + g2.s).tolist() + (14 + g3.s).tolist()
    assert t.tolist() == g1.t.tolist() + (10 + g2.t).tolist() + (14 + g3.t).tolist()
    assert torch.equal(g123.ndata["x"][:, 10:14], g2.ndata["x"])
    g6 = gnn.batch([g123, g123])
    assert g6.num_graphs == 6
    assert g6.graph_indicator.tolist() == [1] * 10 + [2] * 4 + [3] * 7 + [4] * 10 + [5] * 4 + [6] * 7


def test_layer_argument_errors(gnn):
    # GNNlib/src/layers/conv.jl:3-10,22 -> ArgumentError (ValueError here), raised before any kernel runs
    l = gnn.GCNConv(3, 5)
    g = gnn.GNNGraph([1, 2, 3], [2, 3, 1])
    x = gnn.colmajor(torch.rand(3, 3))
    with pytest.raises(ValueError):
        l(g, x, torch.rand(2))
    with pytest.raises(ValueError):
        l(g, x, conv_weight=torch.zeros(5, 4))


def test_reference_arm_prints_the_contract_line():
    """bench.py --impl reference (the oracle port of the reference's CPU path) on a tiny bounded sample: one JSON line
    with the contract's keys; rank != 0 prints nothing."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
           "--cpu-nodes", "20000", "--cpu-edges", "100000", "--ref-sample"]
    out = subprocess.check_output(cmd, text=True, timeout=300)
    line = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "edges/s" and line["value"] > 0
    for key in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config", "cpu_baseline", "e2e"):
        assert key in line
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] == "port"
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    assert subprocess.check_output(cmd, text=True, timeout=300, env=env).strip() == ""


def _bench_module():
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(root, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_bench_reads_roofline_traffic_from_the_committed_ncu_extracts():
    """roofline.traffic must come from the committed CSV of the CURRENT kernel, selected by name — not a literal"""
    b = _bench_module()
    lean = b.ncu_traffic("r2_seg_lean_v0_ncu_raw.csv")
    assert lean is not None and 35e9 < lean < 45e9                        # config 2: 39.2 GB per launch
    fwd = b.ncu_traffic("r2_gat_lean_ncu_raw.csv", "gat_fwd_lean_kernel")
    bwd = b.ncu_traffic("r2_gat_lean_ncu_raw.csv", "gat_bwd_lean_kernel")
    assert fwd is not None and bwd is not None and bwd > fwd > 50e9       # config 3: 94.7 / 126.4 GB
    assert b.ncu_traffic("r2_gat_lean_ncu_raw.csv", "no_such_kernel") is None
    assert b.ncu_traffic("no_such_file.csv") is None
    assert b.ncu_traffic("r2_seg_lean_mean_c4_ncu_raw.csv") is not None   # config 4's mean kernel


def test_bench_argument_surface():
    """the flags the driver and the scripts rely on"""
    import sys
    b = _bench_module()
    old = sys.argv
    try:
        sys.argv = ["bench.py", "--gpus", "8", "--steps", "4", "--warmup", "3", "--config", "5", "--no-parity", "--no-cpu", "--no-e2e"]
        a = b.parse()
    finally:
        sys.argv = old
    assert (a.gpus, a.steps, a.warmup, a.config) == (8, 4, 3, 5)
    assert a.no_parity and a.no_cpu and a.no_e2e and a.impl != "reference"
    assert (a.nodes, a.edges, a.dim) == (100_000_000, 1_000_000_000, 256)     # config 5 = BASELINE configs[4]


def test_bench_dump_outputs_and_its_arguments(tmp_path, monkeypatch):
    """--dump-outputs: float32 files, one seeded row sample shared by the row arrays and the same on every call, the
    whole budget respected; all rows when they fit.  --steps must be a real count."""
    b = _bench_module()
    n, D = 1000, 3
    g = torch.Generator().manual_seed(0)
    y, dx = torch.randn(n, D, generator=g), torch.randn(n, D, generator=g)
    dW, db = torch.randn(D, D, generator=g), torch.randn(D, generator=g)
    monkeypatch.setattr(b, "DUMP_BYTES", 8000)
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), {"y": y, "dx": dx}, {"dW": dW, "db": db}, n)
    got = {f.stem: np.load(f) for f in (tmp_path / "a").glob("*.npy")}
    assert sorted(got) == ["dW", "db", "dx", "row_ids", "y"]
    assert all(v.dtype == (np.float64 if k == "row_ids" else np.float32) for k, v in got.items())
    ids = got["row_ids"].astype(np.int64)
    assert 100 < len(ids) < n and (np.diff(ids) > 0).all() and ids[-1] < n
    assert np.array_equal(got["y"], y.numpy()[ids]) and np.array_equal(got["dx"], dx.numpy()[ids])
    assert np.array_equal(got["dW"], dW.numpy()) and np.array_equal(got["db"], db.numpy())
    assert sum(v.nbytes for v in got.values()) <= 8000
    for k, v in got.items():
        assert np.array_equal(np.load(tmp_path / "b" / f"{k}.npy"), v)
    monkeypatch.setattr(b, "DUMP_BYTES", 60_000_000)
    b.dump_outputs(str(tmp_path / "c"), {"y": y}, {}, n)
    assert np.array_equal(np.load(tmp_path / "c" / "row_ids.npy"), np.arange(n))
    monkeypatch.setattr(b, "DUMP_BYTES", 10)
    with pytest.raises(SystemExit):
        b.dump_outputs(str(tmp_path / "d"), {"y": y}, {"dW": dW}, n)
    for argv in (["--steps", "0"], ["--warmup", "-1"], ["--config", "3", "--dump-outputs", str(tmp_path)],
                 ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        with pytest.raises(SystemExit):
            b.parse()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "1", "--steps", "7", "--warmup", "2", "--dump-outputs", "out"])
    a = b.parse()
    assert (a.steps, a.warmup, a.dump_outputs, a.config) == (7, 2, "out", 2)
