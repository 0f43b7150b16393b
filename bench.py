#!/usr/bin/env python
"""bench.py — edges/s for forward+backward of the layer of one BASELINE.json config, with the HBM roofline of its dominant
kernel, the reference's CPU path timed beside it, parity against the oracle and an end-to-end number on host buffers.

    python bench.py [--config 1..5] [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Default (what the driver runs): config 2 = BASELINE configs[1], the config the metric is quoted on — one GCNConv 128->128
(add_self_loops, relu, bias) forward + backward on RMAT N = 10 M, E = 100 M, fp32.
    1: 2-layer GCN 1433->16->7 on a Cora-shaped graph          3: GATConv 8 heads x 64 on RMAT N = 5 M, E = 50 M
    4: SAGEConv mean 128->128 on 1024 batched ER graphs         5: GCNConv 256->256 on RMAT N = 100 M, E = 1 B, 8 GPUs

`value`   : graph edges per second, every input resident in HBM (CUDA events around the K timed steps, max over ranks).
`e2e`     : the same step through the C ABI's host-buffer entry (config 2: gnnb_gcn_conv_step_host) or the public layer
            call on pinned host arrays (other configs): inputs H2D and results D2H inside the timed region.
`roofline`: the dominant kernel timed alone with CUDA events on its launch stream; achieved = algorithmic bytes per launch
            (SURVEY.md §8d gather model) / duration against MEASURED_PEAKS.json; `traffic` = DRAM bytes per launch read from
            the committed ncu capture of the same kernel (profiles/), never a literal.
`cpu_baseline`, `parity_rel_err`: the oracle's restatement of the reference's CPU algorithm on a bounded sample of the
            same workload, timed on the host cores; the GPU runs the same sample and the two results are compared.
`--impl reference`: the reference's CPU path (oracle port; Julia cannot run here) at the FULL size of the config when the
            host has the memory (config 2: ~60 GB), else the bounded sample (says which).
`--dump-outputs DIR`: after the timed steps of config 2, what the last step returned to its caller (y, dx, dW, db) as
            DIR/<name>.npy, float32; the row arrays as the same seeded sample of rows (row_ids.npy), under 64 MB in all.
            The inputs are seeded, so two builds run with the same arguments can be compared output for output.

bench.py writes nothing into the tree it runs from (the tree may be read-only): no bytecode caches either.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
SEED = 17
DUMP_BYTES = 60_000_000          # array data of --dump-outputs; the .npy headers add 128 bytes a file

# BASELINE.json configs (SURVEY.md §8: sizes BASELINE leaves open are this project's choice, stated with every number)
CFG = {
    1: dict(name="configs[0]: 2-layer GCNConv 1433->16->7, Cora-shaped graph", nodes=2708, edges=10556, dim=1433),
    2: dict(name="configs[1]: GCNConv 128->128, RMAT", nodes=10_000_000, edges=100_000_000, dim=128),
    3: dict(name="configs[2]: GATConv 8 heads x 64 (concat), RMAT", nodes=5_000_000, edges=50_000_000, dim=512),
    4: dict(name="configs[3]: SAGEConv mean 128->128, 1024 batched ER graphs (1000 nodes, 5000 edges each)",
            nodes=1_024_000, edges=5_120_000, dim=128),
    5: dict(name="configs[4]: GCNConv 256->256, RMAT, node-partitioned over 8 GPUs", nodes=100_000_000,
            edges=1_000_000_000, dim=256),
}
CPU_SAMPLE = {2: (1_000_000, 10_000_000), 3: (100_000, 1_000_000), 4: (64, None), 5: (1_000_000, 10_000_000)}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=sorted(CFG))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nodes", type=int, default=None)
    ap.add_argument("--edges", type=int, default=None)
    ap.add_argument("--dim", type=int, default=None)
    ap.add_argument("--cpu-nodes", type=int, default=None, help="bounded CPU sample: nodes")
    ap.add_argument("--cpu-edges", type=int, default=None, help="bounded CPU sample: edges")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity leg (debug)")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-size parity check of the partitioned path (debug)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (debug)")
    ap.add_argument("--ref-sample", action="store_true", help="--impl reference on the bounded sample instead of the full size")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (config 2, one GPU)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and (a.config != 2 or a.impl != "ours"):
        ap.error("--dump-outputs is written by the GPU run of config 2")
    c = CFG[a.config]
    a.nodes = a.nodes or c["nodes"]
    a.edges = a.edges or c["edges"]
    a.dim = a.dim or c["dim"]
    sn, se = CPU_SAMPLE.get(a.config, (None, None))
    a.cpu_nodes = a.cpu_nodes or sn
    a.cpu_edges = a.cpu_edges or se
    return a


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(name, kernel=None):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes) of one launch in a committed profiles/*_ncu_raw.csv: the first
    launch whose kernel name contains `kernel` (launch 1 if None); None if the file or the kernel is missing"""
    import csv
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    try:
        tot, col = 0.0, 2
        with open(os.path.join(ROOT, "profiles", name)) as f:
            for row in csv.reader(f):
                if row and row[0] == "Kernel Name" and kernel is not None:
                    col = next(i for i, v in enumerate(row) if i >= 2 and kernel in v)
                if row and row[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(row[col]) * unit[row[1]]
        return tot or None
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.check_output(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                               "-i", str(self.index)], text=True, timeout=5)
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def oracle_module():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    return oracle


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([int(i.get("num_threads", 1)) for i in threadpool_info() if i.get("user_api") == "blas"] or [1])
    except Exception:
        return os.cpu_count() or 1


def relerr(a, b):
    import numpy as np
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


# ======================================================================================================== CPU legs (oracle port)
def cpu_gcn_step_port(n, E, D, steps=1, keep=False):
    """The reference's CPU path for one GCNConv fwd+bwd, restated (oracle = test infrastructure, timed here only as the
    baseline): add_self_loops, degree scatter, x.*c, CSC rebuild (every forward) + serial dense x CSC product, .*c, BLAS
    GEMM, bias, relu; backward = Zygote's pullbacks (Δ*A' with the forward's A, dense GEMMs)."""
    import numpy as np
    oracle = oracle_module()
    s, t = oracle.rmat(n, E, SEED)
    rng = np.random.default_rng(0)
    x = rng.standard_normal((n, D), dtype=np.float32)
    W = (rng.standard_normal((D, D), dtype=np.float32) / np.sqrt(D)).astype(np.float32)
    b = np.zeros(D, np.float32)
    dy = rng.standard_normal((n, D), dtype=np.float32)
    times, res = [], None
    for _ in range(steps):
        t0 = time.perf_counter()
        s2, t2 = oracle.add_self_loops(s, t, n)                          # conv.jl:26-27
        d = oracle.degree(s2, t2, n, "in", None, np.float32)             # conv.jl:52-56
        c = (1.0 / np.sqrt(d)).astype(np.float32)
        xs = x * c[:, None]                                               # conv.jl:59
        A = oracle.csc_build(s2, t2, n, None, np.float32)                 # adjacency_matrix(g) per call, query.jl:227
        p = oracle.dense_times_csc(xs, A)                                 # xj * A, msgpass.jl:217
        p *= c[:, None]                                                   # conv.jl:67
        pre = p @ W.T + b                                                 # conv.jl:69-71
        y = np.maximum(pre, 0)
        dpre = dy * (pre > 0)                                             # backward
        dW = dpre.T @ p
        db = dpre.sum(0)
        dp = dpre @ W
        dp *= c[:, None]
        dxs = oracle.dense_times_csc(dp, A, transposed=True)              # Δ * A'
        dx = dxs * c[:, None]
        times.append(time.perf_counter() - t0)
        if keep:
            def pullback(mask):                                           # the same pullback on a given relu mask
                dq = dy * mask
                dpp = (dq @ W) * c[:, None]
                return {"dW": dq.T @ p, "db": dq.sum(0), "dx": oracle.dense_times_csc(dpp, A, transposed=True) * c[:, None]}
            res = {"s": s, "t": t, "x": x, "W": W, "b": b, "dy": dy, "y": y, "pre": pre, "pullback": pullback}
        else:
            del A, p, pre
        del xs, dpre, dp, dxs
    return min(times), oracle, res


def dist_parity(args, dg, layer, samples=320, max_deg=20000):
    """Parity of the node-partitioned path at the run's FULL size (every rank calls this; it runs collectives).

    Inputs are a pure function of the GLOBAL node id, so any rank can restate any row.  (1) A sample of this rank's rows
    (the high-degree head of its deal and random ones; rows whose in+out degree exceeds `max_deg` are dropped so that the
    CPU side stays small): their in- and out-edges are found by scanning the generated edge list again with torch ops,
    the in-degrees by a histogram of the same scan, and the ORACLE (gather -> scatter with the reference's c .* (A (c .* x))
    order, conv.jl:52-67) evaluates those rows of propagate, of the layer's forward and of the transposed propagate that
    the backward pass runs.  (2) The adjoint identity <A z, r> = <z, A' r> over ALL rows of all ranks ties the two shards
    (forward, transposed) of every rank together.  Normwise relative errors, max over ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import gnnb200 as gnn
    from gnnb200 import partition
    oracle = oracle_module()
    n, E, D = args.nodes, args.edges, args.dim
    dev, nl, rank = dg.device, dg.n_local, dg.rank
    g_local = dg.local_nodes().long()

    def feat(ids, salt):
        j = torch.arange(D, device=ids.device, dtype=torch.int64)
        v = (ids[:, None] * 1000003 + j[None, :] * 7919 + salt) % 65521
        return (v.double() / 65521.0 - 0.5).float()

    def fill(salt):
        out = torch.empty(nl, D, device=dev)
        for i in range(0, nl, 1 << 20):
            out[i:i + (1 << 20)] = feat(g_local[i:i + (1 << 20)], salt)
        return out

    gen = torch.Generator(device="cpu").manual_seed(99 + rank)
    # the deal is by decreasing degree: rows 0.. are the hubs (millions of edges at config 5; the degree cap would drop them
    # after their edges had been collected), so the high-degree part of the sample starts a little further down
    head = torch.arange(2048, 2048 + 64) if nl > 8192 else torch.arange(min(64, nl))
    idx = torch.unique(torch.cat([head, torch.randint(0, nl, (samples,), generator=gen)])).to(dev)
    tg = g_local[idx]

    c, cf, cb = dg.gcn_c()
    z, r = fill(1), fill(2)
    p = dg.propagate(dg.fwd, z, cf, c)
    q = dg.propagate(dg.bwd, r, cb, c)
    dots = torch.stack([(p * r).sum(dtype=torch.float64), (z * q).sum(dtype=torch.float64)])
    dist.all_reduce(dots)
    adjoint = abs(float(dots[0] - dots[1])) / max(abs(float(dots[0])), 1e-300)
    p_s, q_s = p[idx].cpu().numpy(), q[idx].cpu().numpy()
    del p, q, r
    with torch.no_grad():
        y = partition.dist_gcn_conv(layer, dg, gnn.unrows(z))
    y_s = gnn.rows(y)[idx].cpu().numpy()
    del y, z
    torch.cuda.empty_cache()

    # the sampled rows' edges and every node's in-degree, from the edge list itself
    deg = torch.zeros(n, dtype=torch.int32, device=dev)
    mark = torch.zeros(n, dtype=torch.bool, device=dev)
    mark[tg] = True
    ones = torch.ones(min(1 << 26, max(E, 1)), dtype=torch.int32, device=dev)
    ks, kt = [], []
    for s1, t1 in partition.rmat_chunks(n, E, SEED, dev, 1 << 26):
        s, t = s1 - 1, t1 - 1                                # the generated list is 1-based (Julia's convention)
        deg.index_add_(0, t, ones[:t.numel()])
        m = mark[s] | mark[t]
        ks.append(s[m])
        kt.append(t[m])
    ks, kt = torch.cat(ks), torch.cat(kt)
    del ones
    tgs, perm = torch.sort(tg)
    din = deg[tgs].long()
    ms = mark[ks]
    dout = torch.bincount(torch.searchsorted(tgs, ks[ms]), minlength=tgs.numel())
    ok = (din + dout) <= max_deg
    mark[tgs[~ok]] = False
    V = tgs[ok]
    rows_of_V = perm[ok].cpu().numpy()                       # positions in idx / p_s / y_s / q_s

    def restate(src, dst, salt):
        """rows V of c .* scatter(+, gather(c .* x, src), dst) on the graph with self loops, by the oracle"""
        keep = mark[dst]
        src, dst = torch.cat([src[keep], V]), torch.cat([dst[keep], V])          # + the self loops of V (conv.jl:26-27)
        U = torch.unique(torch.cat([src, V]))
        sc, dc = torch.searchsorted(U, src).cpu().numpy(), torch.searchsorted(U, dst).cpu().numpy()
        cU = (1.0 / np.sqrt((deg[U] + 1).cpu().numpy().astype(np.float32))).astype(np.float32)   # in-degree incl. self loop
        xs = feat(U, salt).cpu().numpy() * cU[:, None]
        out = oracle.propagate_unfused("+", sc + 1, dc + 1, int(U.numel()), xs, None) * cU[:, None]   # the oracle is 1-based, like Julia
        return out[torch.searchsorted(U, V).cpu().numpy()]

    e_p = e_y = e_q = 0.0
    if V.numel():
        p_ref = restate(ks, kt, 1)
        W = layer.weight.detach().cpu().numpy()
        b = layer.bias.detach().cpu().numpy() if layer.bias is not None else 0.0
        y_ref = np.maximum(p_ref @ W.T + b, 0)
        q_ref = restate(kt, ks, 2)
        e_p, e_y, e_q = relerr(p_s[rows_of_V], p_ref), relerr(y_s[rows_of_V], y_ref), relerr(q_s[rows_of_V], q_ref)
    st = torch.tensor([e_p, e_y, e_q, float(V.numel()), float((~ok).sum()), float(din[ok].sum() + dout[ok].sum())],
                      device=dev, dtype=torch.float64)
    mx, sm = st.clone(), st.clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    dist.all_reduce(sm)
    return {"propagate_rows": float(mx[0]), "layer_forward_rows": float(mx[1]), "transposed_propagate_rows": float(mx[2]),
            "adjoint_identity_all_rows": adjoint, "rows_checked": int(sm[3]), "rows_dropped_for_degree": int(sm[4]),
            "edges_restated": int(sm[5]),
            "method": "full-size graph; oracle restatement (gather/scatter, conv.jl:52-67 order) of sampled rows of every "
                      "rank from the regenerated edge list + <Az,r> = <z,A'r> over all rows; normwise, max over ranks"}


def cpu_leg_gcn(args, gpu_replay=None):
    """cpu_baseline (+ parity) of configs 2 / 5: the port on the bounded sample; the GPU replays the same sample."""
    import numpy as np
    n, E, D = args.cpu_nodes, args.cpu_edges, args.dim
    dt, oracle, res = cpu_gcn_step_port(n, E, D, steps=1, keep=gpu_replay is not None)
    parity = gpu_replay(res) if gpu_replay is not None else None
    # generous all-cores variant: prebuilt CSR + OpenMP over rows (fwd and transposed), same GEMMs
    s, t = oracle.rmat(n, E, SEED)
    s2, t2 = oracle.add_self_loops(s, t, n)
    rp, col, _ = oracle.csr(t2, s2, n)
    rpT, colT, _ = oracle.csr(s2, t2, n)
    rng = np.random.default_rng(0)
    x = rng.standard_normal((n, D), dtype=np.float32)
    W = (rng.standard_normal((D, D), dtype=np.float32) / np.sqrt(D)).astype(np.float32)
    dy = rng.standard_normal((n, D), dtype=np.float32)
    c = (1.0 / np.sqrt(np.diff(rp))).astype(np.float32)
    t0 = time.perf_counter()
    p = oracle.spmm_csr_omp(rp, col, n, x, None, c, c)
    pre = p @ W.T
    dpre = dy * (pre > 0)
    dW = dpre.T @ p
    dp = dpre @ W
    dx = oracle.spmm_csr_omp(rpT, colT, n, dp, None, c, c)
    dt_omp = time.perf_counter() - t0
    del dW, dx
    cpu = {"value": E / dt, "unit": "edges/s", "cores": blas_threads(), "kind": "port",
           "sample": f"RMAT N={n} E={E} D={D} seed {SEED}, 1 fwd+bwd GCNConv step: serial CSC rebuild + serial dense x CSC as "
                     f"the reference (1 thread), BLAS GEMMs on {blas_threads()} threads as Julia's OpenBLAS would; scaled by edges",
           "seconds": dt,
           "all_cores_openmp": {"value": E / dt_omp, "cores": oracle.num_threads(), "seconds": dt_omp,
                                "note": "generous variant, NOT the reference's algorithm: prebuilt CSR, OpenMP rows"}}
    return cpu, parity


# ================================================================================================= helpers for the GPU arm
def timed_region(torch, step, steps, dev, sampler_index, flush=None):
    """K steps between two events (synchronised on both sides); with `flush`, every step is timed by its own event pair and
    the L2 flush sits outside the pairs."""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(sampler_index) as clocks:
        torch.cuda.synchronize()
        if flush is None:
            ev0.record()
            for _ in range(steps):
                step()
            ev1.record()
            torch.cuda.synchronize()
            ms = ev0.elapsed_time(ev1) / steps
        else:
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for a, b in evs:
                flush()
                a.record(); step(); b.record()
            torch.cuda.synchronize()
            ms = sum(a.elapsed_time(b) for a, b in evs) / steps
    return ms, clocks.summary()


def time_kernel(torch, fn, reps, flush=None):
    for _ in range(3):
        fn()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    torch.cuda.synchronize()
    for a, b in evs:
        if flush is not None:
            flush()
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs) / len(evs)


def capture_step(torch, step, dev):
    """the whole step as ONE CUDA graph (removes the per-launch CPU latency of small workloads); None if capture fails"""
    try:
        side = torch.cuda.Stream(dev)
        with torch.cuda.stream(side):
            for _ in range(3):
                step()
        torch.cuda.synchronize()
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            step()
        cg.replay()
        torch.cuda.synchronize()
        return cg, None
    except Exception as e:
        torch.cuda.synchronize()
        return None, f"CUDA graph capture failed: {type(e).__name__}: {str(e)[:160]}"


def make_flush(torch, dev):
    buf = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)      # 256 MB > the 126 MB L2
    return lambda: buf.zero_()


def dump_outputs(out_dir, rows, whole, n):
    """Write `whole` (name -> tensor) in full and `rows` (name -> tensor with n rows) on one fixed, seeded sample of rows,
    listed in row_ids.npy, as out_dir/<name>.npy in float32; all rows when they fit DUMP_BYTES."""
    import numpy as np
    import torch
    room = DUMP_BYTES - sum(4 * v.numel() for v in whole.values())
    k = min(n, room // (8 + sum(4 * v[0].numel() for v in rows.values())))
    if k < 1:
        raise SystemExit(f"--dump-outputs: the outputs do not fit {DUMP_BYTES} bytes")
    ids = np.arange(n) if k == n else np.sort(np.random.default_rng(SEED).choice(n, k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "row_ids.npy"), ids.astype(np.float64))
    for name, v in rows.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), v[torch.as_tensor(ids, device=v.device)].float().cpu().numpy())
    for name, v in whole.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), v.float().cpu().numpy())


def base_line(args, value, ms, n_gpus, workload, extra_cfg, clocks, e2e, launches, roof, cpu, parity, dtype="f32"):
    cfg = {"workload": workload}
    cfg.update(extra_cfg)
    return {"metric": "edges/sec fwd+bwd GCNConv 128-dim on 100M-edge graph" if args.config == 2 else
            f"edges/sec fwd+bwd, BASELINE {CFG[args.config]['name']}",
            "value": value, "unit": "edges/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dtype,
            "data": "synthetic", "config": cfg, "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof,
            "cpu_baseline": cpu, "parity_rel_err": parity}


# ============================================================================================================= config 2
def run_config2(args, torch, gnn, dev):
    import ctypes as C
    lib = gnn._lib.lib
    n, E, D = args.nodes, args.edges, args.dim
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    g = gnn.rmat_graph(n, E, SEED, device=dev)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0
    t0 = time.perf_counter()
    g.plan()
    g2 = gnn.add_self_loops(g)
    gnn._lib.check(lib.gnnb_graph_csr(g2.plan().h, 1, None, None, None, None))   # transposed plan
    torch.cuda.synchronize()
    t_plan = time.perf_counter() - t0

    gen = torch.Generator(device=dev).manual_seed(0)
    torch.manual_seed(0)                    # the weights: torch seeds its CUDA generators differently in every process
    layer = gnn.GCNConv(D, D, torch.relu, device=dev)
    x = gnn.unrows(torch.randn(n, D, device=dev, generator=gen)).requires_grad_(True)
    dy = gnn.unrows(torch.randn(n, D, device=dev, generator=gen))
    last = {}

    def step():
        x.grad = None
        layer.weight.grad = None
        layer.bias.grad = None
        y = layer(g, x)
        y.backward(dy)
        if args.dump_outputs:
            last["y"] = y
        return y

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    l0 = gnn.launch_count()
    ms, clocks = timed_region(torch, step, args.steps, dev, dev.index or 0)
    launches = gnn.launch_count() - l0
    value = E / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"y": gnn.rows(last.pop("y").detach()), "dx": gnn.rows(x.grad)},
                     {"dW": layer.weight.grad, "db": layer.bias.grad}, n)

    # ---- the dominant kernel alone: fused GCN propagate (both directions), CUDA events on the launch stream
    xr = gnn.rows(x.detach())
    out = torch.empty_like(xr)
    p2 = g2.plan()
    st = torch.cuda.current_stream(dev).cuda_stream
    kt = {tr: time_kernel(torch, lambda tr=tr: gnn._lib.check(lib.gnnb_gcn_propagate(p2.h, tr, xr.data_ptr(), None, None, D,
                                                                                      out.data_ptr(), st)), args.steps)
          for tr in (0, 1)}
    E2 = E + n
    alg_bytes = E2 * (4 * D + 4) + 4 * (n + 1) + 4 * D * n          # SURVEY.md §8d gather model, per launch
    compulsory = 4 * D * n * 2 + 4 * E2 + 4 * (n + 1)
    kms = 0.5 * (kt[0] + kt[1])
    peak, peak_src = measured_peaks()
    achieved = alg_bytes / (kms * 1e-3) / 1e9
    default_wl = (n, E, D) == (CFG[2]["nodes"], CFG[2]["edges"], CFG[2]["dim"])
    traffic = ncu_traffic("r2_seg_lean_v0_ncu_raw.csv") if default_wl else None
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_GBps": (traffic / (kms * 1e-3) / 1e9) if traffic else None,
            "traffic_frac_of_peak": (traffic / (kms * 1e-3) / 1e9 / peak) if traffic else None,
            "traffic_source": "profiles/r2_seg_lean_v0_ncu_raw.csv (ncu --set full, same kernel, same workload)",
            "kernel": "gnnb::seg_lean_kernel<1,1,false,0,SUM> (fused GCN propagate, D=128, per-edge scale stream)",
            "kernel_ms": {"forward": kt[0], "transposed": kt[1]}, "algorithmic_bytes_per_launch": alg_bytes,
            "compulsory_bytes_per_launch": compulsory, "peak_source": peak_src, "share_of_step": 2 * kms / ms}
    del out

    # ---- e2e: the C ABI's host-buffer entry (one call = forward + backward, copies inside)
    e2e = None
    if not args.no_e2e:
        xh = torch.empty(n, D, pin_memory=True).normal_()
        dyh = torch.empty(n, D, pin_memory=True).normal_()
        yh = torch.empty(n, D, pin_memory=True)
        dxh = torch.empty(n, D, pin_memory=True)
        Wh = layer.weight.detach().cpu().contiguous()
        bh = layer.bias.detach().cpu().contiguous()
        dWh, dbh = torch.empty_like(Wh), torch.empty_like(bh)

        def step_host():
            gnn._lib.check(lib.gnnb_gcn_conv_step_host(p2.h, xh.data_ptr(), Wh.data_ptr(), bh.data_ptr(), 1, D, D,
                                                       dyh.data_ptr(), yh.data_ptr(), dxh.data_ptr(), dWh.data_ptr(),
                                                       dbh.data_ptr()))

        ke = max(2, min(args.steps, 5))
        step_host()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(ke):
            step_host()                                   # synchronous: returns when the results are in host memory
        torch.cuda.synchronize()
        ems = (time.perf_counter() - t0) * 1e3 / ke
        e2e = {"value": E / (ems * 1e-3), "unit": "edges/s", "ms_per_step": ems, "steps": ke,
               "h2d_bytes_per_step": 2 * 4 * n * D + 4 * D * D + 4 * D, "d2h_bytes_per_step": 2 * 4 * n * D + 4 * D * D + 4 * D,
               "api": "C ABI gnnb_gcn_conv_step_host on pinned host arrays (x, dy, W, b up; y, dx, dW, db down, all inside "
                      "the call); wall clock around synchronous calls"}
        del xh, dyh, yh, dxh

    # ---- cpu_baseline + parity: the oracle port on the bounded sample, replayed by the GPU
    cpu = parity = None
    if not args.no_cpu:
        def gpu_replay(r):
            ns = r["x"].shape[0]
            gs = gnn.GNNGraph(torch.as_tensor(r["s"]), torch.as_tensor(r["t"]), num_nodes=ns).to(dev)
            ls = gnn.GCNConv(D, D, torch.relu, device=dev)
            with torch.no_grad():
                ls.weight.copy_(torch.as_tensor(r["W"]))
                ls.bias.copy_(torch.as_tensor(r["b"]))
            xs = gnn.unrows(torch.as_tensor(r["x"]).to(dev)).requires_grad_(True)
            ys = ls(gs, xs)
            ys.backward(gnn.unrows(torch.as_tensor(r["dy"]).to(dev)))
            torch.cuda.synchronize()
            yg = gnn.rows(ys.detach()).cpu().numpy()
            ref = r["pullback"](yg > 0)                    # relu' is discontinuous at 0: the pullback is compared on the mask
            return {"y": relerr(yg, r["y"]), "dx": relerr(gnn.rows(xs.grad).cpu().numpy(), ref["dx"]),       # of its forward
                    "dW": relerr(ls.weight.grad.cpu().numpy(), ref["dW"]), "db": relerr(ls.bias.grad.cpu().numpy(), ref["db"]),
                    "relu_mask_disagreements": int(((yg > 0) != (r["pre"] > 0)).sum()), "elements": int(yg.size),
                    "against": f"oracle port (fp32, the reference's operation order) on RMAT N={ns} E={len(r['s'])}; "
                               "normwise relative error, bar 1e-5; backward on the GPU forward's relu mask"}
        cpu, parity = cpu_leg_gcn(args, gpu_replay)

    workload = (f"GCNConv {D}->{D} (add_self_loops, relu, bias) fwd+bwd on RMAT N={n} E={E} seed {SEED} (BASELINE configs[1]); "
                f"edges counted = graph edges E (the {n} self loops are extra work)")
    return base_line(args, value, ms, 1, workload,
                     {"l2": "inputs (5.1 GB features) are far larger than the 126 MB L2; no flush needed",
                      "plan_build_ms": t_plan * 1e3, "graph_gen_ms": t_gen * 1e3, "chunk_edges": 128},
                     clocks, e2e, launches, roof, cpu, parity)


# ============================================================================================================= config 1
def cora_like(torch, dev):
    n, E = CFG[1]["nodes"], CFG[1]["edges"]
    gen = torch.Generator(device="cpu").manual_seed(SEED)
    u = torch.randint(1, n + 1, (E // 2,), generator=gen)
    v = torch.randint(1, n + 1, (E // 2,), generator=gen)
    X = (torch.rand(n, 1433, generator=gen) < 0.0127).float()
    return n, E, torch.cat([u, v]), torch.cat([v, u]), X


def run_config1(args, torch, gnn, dev):
    import numpy as np
    n, E, s, t, X = cora_like(torch, dev)
    g = gnn.GNNGraph(s.to(dev), t.to(dev), num_nodes=n)
    torch.manual_seed(0)
    l1 = gnn.GCNConv(1433, 16, torch.relu, device=dev)
    l2 = gnn.GCNConv(16, 7, device=dev)
    params = list(l1.parameters()) + list(l2.parameters())
    x = gnn.unrows(X.to(dev))
    gen = torch.Generator(device="cpu").manual_seed(1)
    dy_h = torch.randn(n, 7, generator=gen)
    dy = gnn.unrows(dy_h.to(dev))

    def step():
        for p in params:
            p.grad = None
        y = l2(g, l1(g, x))
        y.backward(dy)
        return y

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    flush = make_flush(torch, dev)
    l0 = gnn.launch_count()
    ms_eager, clocks = timed_region(torch, step, args.steps, dev, dev.index or 0, flush)
    launches = gnn.launch_count() - l0
    # the whole step as ONE CUDA graph launch (launch-latency bound otherwise: ~40 kernels of a few microseconds)
    graph_ms = None
    cg, graph_note = capture_step(torch, step, dev)
    if cg is not None:
        graph_ms, _ = timed_region(torch, cg.replay, args.steps, dev, dev.index or 0, flush)
    ms = graph_ms if graph_ms is not None else ms_eager
    peak, peak_src = measured_peaks()
    bytes_step = 4 * (2 * n * 1433 + 4 * n * 16 + 4 * n * 7 + 3 * 1433 * 16) + 2 * 2 * (E + n) * (4 * 16 + 12)
    roof = {"bound": "hbm", "achieved": bytes_step / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": bytes_step / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
            "kernel": "whole step (no dominant kernel: ~40 launches of 2-10 us each; the 15.5 MB feature matrix is the only "
                      "array above 1 MB)", "algorithmic_bytes_per_launch": bytes_step,
            "launch_bound": {"eager_ms": ms_eager, "cuda_graph_ms": graph_ms, "launches_per_step": launches / args.steps,
                             "note": graph_note or "one cudaGraphLaunch per step removes the per-launch CPU latency"}}
    e2e = None
    if not args.no_e2e:
        Xh = X.pin_memory()
        yh = torch.empty(n, 7, pin_memory=True)

        def step_host():
            xd = gnn.unrows(Xh.to(dev, non_blocking=True))
            for p in params:
                p.grad = None
            y = l2(g, l1(g, xd))
            y.backward(dy)
            yh.copy_(gnn.rows(y.detach()), non_blocking=True)
            return l1.weight.grad.cpu()

        step_host()
        ems, _ = timed_region(torch, step_host, max(2, min(args.steps, 10)), dev, dev.index or 0)
        e2e = {"value": E / (ems * 1e-3), "unit": "edges/s", "ms_per_step": ems, "h2d_bytes_per_step": 4 * n * 1433,
               "d2h_bytes_per_step": 4 * n * 7 + 4 * 1433 * 16, "api": "gnnb200.GCNConv x2 on a pinned host feature matrix"}
    cpu = parity = None
    if not args.no_cpu:
        oracle = oracle_module()
        sn, tn = s.numpy().astype(np.int64), t.numpy().astype(np.int64)
        Xn = X.numpy()
        W1, b1 = l1.weight.detach().cpu().numpy(), l1.bias.detach().cpu().numpy()
        W2, b2 = l2.weight.detach().cpu().numpy(), l2.bias.detach().cpu().numpy()
        best = None
        for _ in range(5):
            t0 = time.perf_counter()
            s2, t2 = oracle.add_self_loops(sn, tn, n)
            h = Xn @ W1.T                                               # Dout < Din: multiply first (conv.jl:36-40)
            p1, c = oracle.gcn_propagate(s2, t2, n, h)
            pre1 = p1 + b1
            h1 = np.maximum(pre1, 0)
            h2 = h1 @ W2.T
            p2, _ = oracle.gcn_propagate(s2, t2, n, h2)
            y = p2 + b2
            dyn = dy_h.numpy()
            dh2 = oracle.propagate_unfused("+", t2, s2, n, dyn * c[:, None]) * c[:, None]
            dW2 = dh2.T @ h1
            dh1 = (dh2 @ W2) * (pre1 > 0)
            dh = oracle.propagate_unfused("+", t2, s2, n, dh1 * c[:, None]) * c[:, None]
            dW1 = dh.T @ Xn
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        yg = step()
        torch.cuda.synchronize()
        parity = {"y": relerr(gnn.rows(yg.detach()).cpu().numpy(), y), "dW1": relerr(l1.weight.grad.cpu().numpy(), dW1),
                  "dW2": relerr(l2.weight.grad.cpu().numpy(), dW2), "against": "oracle port, full size; bar 1e-5"}
        cpu = {"value": E / best, "unit": "edges/s", "cores": blas_threads(), "kind": "port", "seconds": best,
               "sample": "the whole config (N=2708, E=10556): serial gather/scatter path of the reference, BLAS GEMMs"}
    workload = (f"2-layer GCNConv 1433->16->7 (relu between, self loops) fwd+bwd on a Cora-shaped graph N={n} E={E} (bidirected "
                "random pairs, 1.27 % binary features; BASELINE configs[0]); edges counted once per step")
    return base_line(args, E / (ms * 1e-3), ms, 1, workload,
                     {"l2": "inputs fit L2: 256 MB written between timed iterations (outside the event pairs)",
                      "timed": "CUDA graph replay of the step" if graph_ms is not None else "eager"},
                     clocks, e2e, launches, roof, cpu, parity)


# ============================================================================================================= config 3
def run_config3(args, torch, gnn, dev):
    import numpy as np
    lib = gnn._lib.lib
    n, E, H, Cc = args.nodes, args.edges, 8, 64
    D = H * Cc
    g = gnn.rmat_graph(n, E, SEED, device=dev)
    torch.manual_seed(0)
    layer = gnn.GATConv(D, Cc, torch.relu, heads=H, device=dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    x = gnn.unrows(torch.randn(n, D, device=dev, generator=gen)).requires_grad_(True)
    dy = gnn.unrows(torch.randn(n, D, device=dev, generator=gen))

    def step():
        x.grad = None
        for p_ in layer.parameters():
            p_.grad = None
        y = layer(g, x)
        y.backward(dy)
        return y

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    l0 = gnn.launch_count()
    ms, clocks = timed_region(torch, step, args.steps, dev, dev.index or 0)
    launches = gnn.launch_count() - l0
    # dominant kernels alone
    g2 = gnn.add_self_loops(g)
    p = g2.plan()
    Wx = torch.randn(n, H, Cc, device=dev, generator=gen)
    el = torch.randn(n, H, device=dev, generator=gen); er = torch.randn(n, H, device=dev, generator=gen)
    out = torch.empty_like(Wx); smax = torch.empty(n, H, device=dev); ssum = torch.empty(n, H, device=dev)
    kf = time_kernel(torch, lambda: gnn._lib.check(lib.gnnb_gat_aggregate(p.h, Wx.data_ptr(), el.data_ptr(), er.data_ptr(), Cc, H, 0.2,
                                                                         out.data_ptr(), None, smax.data_ptr(), ssum.data_ptr(), None)), 5)
    dWx = torch.empty_like(Wx); del_ = torch.empty(n, H, device=dev); der = torch.empty(n, H, device=dev)
    do = torch.randn(n, H, Cc, device=dev, generator=gen)
    kb = time_kernel(torch, lambda: gnn._lib.check(lib.gnnb_gat_aggregate_bwd(p.h, Wx.data_ptr(), el.data_ptr(), er.data_ptr(),
                                                                             smax.data_ptr(), ssum.data_ptr(), out.data_ptr(),
                                                                             do.data_ptr(), Cc, H, 0.2, dWx.data_ptr(),
                                                                             del_.data_ptr(), der.data_ptr(), None)), 5)
    E2 = E + n
    alg_f = E2 * (4 * D + 4 + 4 * H) + 4 * (n + 1) + 4 * D * n + 3 * 4 * H * n
    alg_b = E2 * (2 * 4 * D + 4 + 8 * H) + 4 * (n + 1) + 2 * 4 * D * n
    peak, peak_src = measured_peaks()
    roof = {"bound": "hbm", "achieved": alg_b / (kb * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg_b / (kb * 1e-3) / 1e9 / peak,
            "traffic": ncu_traffic("r2_gat_lean_ncu_raw.csv", "gat_bwd_lean_kernel"), "peak_source": peak_src,
            "kernel": "gnnb::gat_bwd_lean_kernel<4> (attention backward over the work items of the CSR-by-source plan: dout and Wx rows gathered per edge)",
            "kernel_ms": {"gat_fwd": kf, "gat_bwd_total": kb}, "algorithmic_bytes_per_launch": alg_b,
            "forward": {"achieved": alg_f / (kf * 1e-3) / 1e9, "frac": alg_f / (kf * 1e-3) / 1e9 / peak, "algorithmic_bytes": alg_f},
            "share_of_step": (kf + kb) / ms}
    del Wx, el, er, out, smax, ssum, dWx, del_, der, do
    torch.cuda.empty_cache()
    e2e = None
    if not args.no_e2e:
        xh = torch.empty(n, D, pin_memory=True).normal_()
        dyh = torch.empty(n, D, pin_memory=True).normal_()
        yh = torch.empty(n, D, pin_memory=True); dxh = torch.empty(n, D, pin_memory=True)

        def step_host():
            xd = gnn.unrows(xh.to(dev, non_blocking=True)).requires_grad_(True)
            dyd = gnn.unrows(dyh.to(dev, non_blocking=True))
            for p_ in layer.parameters():
                p_.grad = None
            y = layer(g, xd)
            y.backward(dyd)
            yh.copy_(gnn.rows(y.detach()), non_blocking=True)
            dxh.copy_(gnn.rows(xd.grad), non_blocking=True)
            return layer.a.grad.cpu()

        step_host()
        ems, _ = timed_region(torch, step_host, 2, dev, dev.index or 0)
        e2e = {"value": E / (ems * 1e-3), "unit": "edges/s", "ms_per_step": ems, "h2d_bytes_per_step": 2 * 4 * n * D,
               "d2h_bytes_per_step": 2 * 4 * n * D + 4 * 2 * Cc * H, "api": "gnnb200.GATConv on pinned host arrays"}
        del xh, dyh, yh, dxh
    cpu = parity = None
    if not args.no_cpu:
        oracle = oracle_module()
        ns, Es = args.cpu_nodes, args.cpu_edges
        s, t = oracle.rmat(ns, Es, SEED)
        rng = np.random.default_rng(0)
        xs = rng.standard_normal((ns, D), dtype=np.float32)
        Wd = layer.dense_x.weight.detach().cpu().numpy()
        a = layer.a.detach().cpu().numpy()                              # (2C, H)
        bias = layer.bias.detach().cpu().numpy()
        t0 = time.perf_counter()
        s2, t2 = oracle.add_self_loops(s, t, ns)
        Wxs = (xs @ Wd.T).reshape(ns, H, Cc)
        o, _ = oracle.gat_aggregate(s2, t2, ns, Wxs, np.ascontiguousarray(a.T))
        ys = np.maximum(o.reshape(ns, D) + bias, 0)
        dt = time.perf_counter() - t0
        gs = gnn.GNNGraph(torch.as_tensor(s), torch.as_tensor(t), num_nodes=ns).to(dev)
        with torch.no_grad():
            yg = layer(gs, gnn.unrows(torch.as_tensor(xs).to(dev)))
        parity = {"y": relerr(gnn.rows(yg).cpu().numpy(), ys),
                  "against": f"oracle port (gather, vcat, logits, leakyrelu, softmax_edge_neighbors, weighted scatter) on RMAT N={ns} E={Es}, forward; bar 1e-5"}
        cpu = {"value": Es / (2.5 * dt), "unit": "edges/s", "cores": blas_threads(), "kind": "port", "seconds_forward": dt,
               "sample": f"RMAT N={ns} E={Es}, GATConv forward through the reference's unfused path (the (2C,H,E) tensors "
                         f"materialised), fwd+bwd estimated as 2.5 x forward (Zygote's pullback re-traverses every edge tensor)"}
    workload = (f"GATConv {D} -> {Cc} x {H} heads (concat, self loops, relu, slope 0.2) fwd+bwd on RMAT N={n} E={E} seed {SEED} "
                "(BASELINE configs[2]; N is this project's choice)")
    return base_line(args, E / (ms * 1e-3), ms, 1, workload, {"l2": "inputs (10 GB features) far larger than L2"},
                     clocks, e2e, launches, roof, cpu, parity)


# ============================================================================================================= config 4
def batched_er(torch, G, n1, e1, dev, seed=SEED):
    gen = torch.Generator(device="cpu").manual_seed(seed)
    off = (torch.arange(G) * n1).repeat_interleave(e1)
    s = torch.randint(0, n1, (G * e1,), generator=gen) + off + 1
    t = torch.randint(0, n1, (G * e1,), generator=gen) + off + 1
    return s, t


def run_config4(args, torch, gnn, dev):
    import numpy as np
    lib = gnn._lib.lib
    G, n1, e1, D = 1024, 1000, 5000, args.dim
    n, E = G * n1, G * e1
    s, t = batched_er(torch, G, n1, e1, dev)
    gi = torch.arange(1, G + 1).repeat_interleave(n1)
    g = gnn.GNNGraph(s.to(dev), t.to(dev), num_nodes=n, num_graphs=G, graph_indicator=gi.to(dev))
    torch.manual_seed(0)
    layer = gnn.SAGEConv(D, D, torch.relu, device=dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    x = gnn.unrows(torch.randn(n, D, device=dev, generator=gen)).requires_grad_(True)
    dy = gnn.unrows(torch.randn(n, D, device=dev, generator=gen))

    def step():
        x.grad = None
        layer.weight.grad = None
        layer.bias.grad = None
        y = layer(g, x)
        y.backward(dy)
        return y

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    flush = make_flush(torch, dev)
    l0 = gnn.launch_count()
    ms_eager, clocks = timed_region(torch, step, args.steps, dev, dev.index or 0, flush)
    launches = gnn.launch_count() - l0
    cg, graph_note = capture_step(torch, step, dev)      # ~45 launches of 0.02-0.3 ms: CPU launch latency otherwise dominates
    graph_ms = None
    if cg is not None:
        graph_ms, _ = timed_region(torch, cg.replay, args.steps, dev, dev.index or 0, flush)
    ms = graph_ms if graph_ms is not None else ms_eager
    xr = gnn.rows(x.detach()); out = torch.empty_like(xr); p = g.plan()
    gnn._lib.check(lib.gnnb_graph_csr(p.h, 1, None, None, None, None))
    kms = time_kernel(torch, lambda: gnn._lib.check(lib.gnnb_propagate(p.h, 0, 0, gnn._lib.MEAN, xr.data_ptr(), None, None, None, D,
                                                                       out.data_ptr(), None)), 10, flush)
    alg = E * (4 * D + 4) + 4 * (n + 1) + 4 * D * n
    peak, peak_src = measured_peaks()
    roof = {"bound": "hbm", "achieved": alg / (kms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (kms * 1e-3) / 1e9 / peak,
            "traffic": ncu_traffic("r2_seg_lean_mean_c4_ncu_raw.csv"), "peak_source": peak_src,
            "kernel": "gnnb::seg_lean_kernel<1,0,false,0,MEAN> (fused mean propagate, D=128) after an L2 flush",
            "kernel_ms": kms, "algorithmic_bytes_per_launch": alg, "compulsory_bytes_per_launch": 2 * 4 * D * n + 4 * E + 4 * (n + 1),
            "share_of_step": 2 * kms / ms,
            "launch_bound": {"eager_ms": ms_eager, "cuda_graph_ms": graph_ms, "launches_per_step": launches / args.steps,
                             "note": graph_note or "one cudaGraphLaunch per step"},
            "note": "components of 1000 nodes (512 KB of features) fit L2: the gather-model fraction can exceed 1"}
    e2e = None
    if not args.no_e2e:
        xh = torch.empty(n, D, pin_memory=True).normal_()
        dyh = torch.empty(n, D, pin_memory=True).normal_()
        yh = torch.empty(n, D, pin_memory=True); dxh = torch.empty(n, D, pin_memory=True)

        def step_host():
            xd = gnn.unrows(xh.to(dev, non_blocking=True)).requires_grad_(True)
            dyd = gnn.unrows(dyh.to(dev, non_blocking=True))
            layer.weight.grad = None
            layer.bias.grad = None
            y = layer(g, xd)
            y.backward(dyd)
            yh.copy_(gnn.rows(y.detach()), non_blocking=True)
            dxh.copy_(gnn.rows(xd.grad), non_blocking=True)
            return layer.weight.grad.cpu()

        step_host()
        ems, _ = timed_region(torch, step_host, max(2, min(args.steps, 5)), dev, dev.index or 0)
        e2e = {"value": E / (ems * 1e-3), "unit": "edges/s", "ms_per_step": ems, "h2d_bytes_per_step": 2 * 4 * n * D,
               "d2h_bytes_per_step": 2 * 4 * n * D + 4 * 2 * D * D, "api": "gnnb200.SAGEConv on pinned host arrays"}
    cpu = parity = None
    if not args.no_cpu:
        oracle = oracle_module()
        Gs = args.cpu_nodes or 64
        ss, ts = batched_er(torch, Gs, n1, e1, dev, seed=SEED + 1)
        ns, Es = Gs * n1, Gs * e1
        sn, tn = ss.numpy().astype(np.int64), ts.numpy().astype(np.int64)
        rng = np.random.default_rng(0)
        xs = rng.standard_normal((ns, D), dtype=np.float32)
        dys = rng.standard_normal((ns, D), dtype=np.float32)
        W, b = layer.weight.detach().cpu().numpy(), layer.bias.detach().cpu().numpy()
        t0 = time.perf_counter()
        m = oracle.propagate_unfused("mean", sn, tn, ns, xs)              # gather + sequential scatter, the reference's path
        cat = np.concatenate([xs, m], axis=1)                             # vcat(xi, m), conv.jl:281
        pre = cat @ W.T + b
        ys = np.maximum(pre, 0)
        deg = np.maximum(np.bincount(tn - 1, minlength=ns), 1).astype(np.float32)

        def pullback(mask):
            dq = dys * mask
            dc = dq @ W
            return dq.T @ cat, dc[:, :D] + oracle.propagate_unfused("+", tn, sn, ns, dc[:, D:] / deg[:, None])
        dW, dxs = pullback(pre > 0)
        dt = time.perf_counter() - t0
        gs = gnn.GNNGraph(ss.to(dev), ts.to(dev), num_nodes=ns)
        xg = gnn.unrows(torch.as_tensor(xs).to(dev)).requires_grad_(True)
        layer.weight.grad = None
        yg = layer(gs, xg)
        yg.backward(gnn.unrows(torch.as_tensor(dys).to(dev)))
        ygn = gnn.rows(yg.detach()).cpu().numpy()
        dW, dxs = pullback(ygn > 0)                        # relu' is discontinuous at 0: same mask as the GPU forward
        parity = {"y": relerr(ygn, ys), "dx": relerr(gnn.rows(xg.grad).cpu().numpy(), dxs),
                  "dW": relerr(layer.weight.grad.cpu().numpy(), dW),
                  "relu_mask_disagreements": int(((ygn > 0) != (pre > 0)).sum()), "elements": int(ygn.size),
                  "against": f"oracle port on {Gs} batched graphs (N={ns} E={Es}), fwd+bwd; bar 1e-5; backward on the GPU "
                             "forward's relu mask"}
        cpu = {"value": Es / dt, "unit": "edges/s", "cores": blas_threads(), "kind": "port", "seconds": dt,
               "sample": f"{Gs} of the 1024 graphs: unfused gather + serial scatter(mean) as the reference, vcat, BLAS GEMMs; scaled by edges"}
    workload = (f"SAGEConv {D}->{D} mean (relu, bias) fwd+bwd on {G} batched ER graphs ({n1} nodes, {e1} edges each): N={n} E={E} "
                "(BASELINE configs[3]; D is this project's choice)")
    return base_line(args, E / (ms * 1e-3), ms, 1, workload,
                     {"l2": "256 MB written between timed iterations (outside the event pairs): the 524 MB of features are "
                            "only 4x the L2", "timed": "CUDA graph replay of the step" if graph_ms is not None else "eager"},
                     clocks, e2e, launches, roof, cpu, parity)


# ============================================================================================================= reference arm
def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; Julia is not installed) on the host cores, rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = args.config if args.config in (2, 5) else 2
    n_full, E_full, D = CFG[cfg]["nodes"], CFG[cfg]["edges"], CFG[cfg]["dim"]
    if args.nodes != CFG[args.config]["nodes"] or args.edges != CFG[args.config]["edges"]:
        n_full, E_full, D = args.nodes, args.edges, args.dim
    need_gb = (10 * n_full * D * 4 + 4 * 8 * E_full + 16 * (E_full + n_full)) / 1e9
    try:
        import psutil
        avail_gb = psutil.virtual_memory().available / 1e9
    except Exception:
        avail_gb = 0.0
    full = (not args.ref_sample) and cfg == 2 and avail_gb > 1.3 * need_gb
    n, E = (n_full, E_full) if full else (args.cpu_nodes or 1_000_000, args.cpu_edges or 10_000_000)
    nwarm, nstep = (1, max(1, min(args.steps, 2))) if full else (1, max(1, min(args.steps, 3)))
    t_all = []
    for _ in range(nwarm + nstep):
        dt, _, _ = cpu_gcn_step_port(n, E, D, steps=1)
        t_all.append(dt)
    timed = t_all[nwarm:]
    dt = sum(timed) / len(timed)
    val = E / dt
    sample = (f"the full config: RMAT N={n} E={E} D={D}" if full else
              f"bounded sample RMAT N={n} E={E} D={D} of RMAT N={n_full} E={E_full} (host has {avail_gb:.0f} GB free, full size "
              f"needs {need_gb:.0f} GB)" if cfg == 2 else
              f"bounded sample RMAT N={n} E={E} D={D}; config {cfg} itself (102 GB of features) is not run on the CPU")
    line = {
        "impl": "reference", "metric": "edges/sec fwd+bwd GCNConv 128-dim on 100M-edge graph", "value": val, "unit": "edges/s",
        "n_gpus": args.gpus, "steps": len(timed), "warmup": nwarm, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"GCNConv {D}->{D} (add_self_loops, relu, bias) fwd+bwd on RMAT N={n_full} E={E_full} seed {SEED} "
                               f"(BASELINE configs[{cfg - 1}]); this arm ran {sample}", "same_size_as_repo_arm": bool(full)},
        "cpu_baseline": {"value": val, "unit": "edges/s", "cores": blas_threads(), "kind": "port",
                         "sample": f"{sample}; serial CSC rebuild + serial dense x CSC per call (the reference's CPU algorithm for "
                                   f"copy_xj/+; Julia unavailable, so the oracle port is timed) on 1 thread, BLAS GEMMs on "
                                   f"{blas_threads()} threads"},
        "e2e": {"value": val, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ============================================================================================================= GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import gnnb200 as gnn

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    torch.backends.cuda.matmul.allow_tf32 = False   # fp32 GEMM like the reference (cuBLAS sgemm)
    torch.backends.cudnn.allow_tf32 = False
    if world > 1 or os.environ.get("GNNB_BENCH_PARTITIONED"):   # the env switch: the partitioned path on one rank (debug)
        if args.dump_outputs:
            raise SystemExit("--dump-outputs is written by the single-GPU path")
        dist.init_process_group("nccl", device_id=dev)
        if args.config not in (2, 5):
            raise SystemExit("configs 1, 3, 4 are single-GPU workloads")
        from gnnb200 import partition
        if args.config == 5 and "GNNB_HALO_BUFFERS" not in os.environ:
            os.environ["GNNB_HALO_BUFFERS"] = "1"    # 1 KB rows: one halo buffer per shard (forward and backward alternate)
        return partition.bench_multi(args, world, int(os.environ.get("RANK", "0")), dev, SEED, ClockSampler, measured_peaks,
                                     cpu_leg=None if args.no_cpu else (lambda: cpu_leg_gcn(args)[0]),
                                     parity=None if args.no_parity else (lambda dg, layer: dist_parity(args, dg, layer)))
    if args.config == 5:
        raise SystemExit("config 5 (1 B edges, 256-wide rows) needs the 8 GPUs of a box: launch with torchrun --nproc-per-node 8")
    fn = {1: run_config1, 2: run_config2, 3: run_config3, 4: run_config4}[args.config]
    print(json.dumps(fn(args, torch, gnn, dev)), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
