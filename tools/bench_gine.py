"""GINE model throughput on the layerwise path, next to the C2 GIN model on the same batch.

Builds GINE 3x128 (C2's shape with bond features) on 1M QM9-shaped graphs, device-resident, and
times forwards with CUDA events on the model handle's stream after warm-up.  On the same batch it
also times C2's GIN model forced to the layerwise path and on AUTO (the fused tcgen05 kernel), so the
cost of the edge features reads against both.  Repeated at edge_dim 4 and 16.  A separate profiled
pass gives the per-class split (tables, aggregate, GEMM, pool) and the GINE aggregation's
algorithmic bytes over its measured time.  Then one C5-shaped power-law graph (2M nodes, edge_dim 8),
whose hub rows run unbucketed (one sub-warp per row).  Prints one JSON line; needs a CUDA device.

    python tools/bench_gine.py [--steps 10] [--warmup 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def card_info(torch):
    name = torch.cuda.get_device_name(0)
    power = None
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                            "-i", "0"], capture_output=True, text=True, timeout=30)
        power = float(r.stdout.strip().splitlines()[0]) if r.returncode == 0 else None
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        power = None
    return name, power


def gine_model(gnnb, in_dim, hidden, layers, edge_dim, out_dim, pools, seed=0):
    import torch
    import torch.nn as nn

    torch.manual_seed(seed)
    head = gnnb.MLP(hidden * len(pools), out_dim, hidden_dim=64, hidden_layers=2,
                    activation=nn.ReLU)
    return gnnb.GNNModel(in_dim, edge_dim, hidden, layers, hidden, gnnb.GINEConv_GNNB, nn.ReLU,
                         True, gnnb.GlobalPooling(list(pools)), head, None)


def to_device(torch, batch):
    d = {k: torch.from_numpy(np.ascontiguousarray(getattr(batch, k))).cuda()
         for k in ("x", "coo", "node_ptr", "edge_ptr")}
    d["edge_attr"] = (torch.from_numpy(np.ascontiguousarray(batch.edge_attr)).cuda()
                      if batch.edge_attr is not None else None)
    return d


def time_forward(torch, eng, dev, batch, steps, warmup):
    """ms per forward: CUDA events on the handle's stream around `steps` enqueued forwards"""
    out = torch.empty((batch.n_graphs, eng.out_dim), dtype=torch.float32, device="cuda")
    stream = torch.cuda.ExternalStream(eng.stream)

    def fwd():
        eng.run_device(dev["x"], dev["coo"], dev["node_ptr"], dev["edge_ptr"], out, batch.n_graphs,
                       batch.total_nodes, batch.total_edges, edge_attr=dev["edge_attr"])

    for _ in range(warmup):
        fwd()
    eng.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(steps):
        fwd()
    b.record(stream)
    eng.synchronize()
    b.synchronize()
    return a.elapsed_time(b) / steps, fwd


def profile(eng, fwd, reps):
    eng.set_profile(True)
    eng.read_profile()
    for _ in range(reps):
        fwd()
    eng.synchronize()
    p = eng.read_profile()
    eng.set_profile(False)
    return {k: round(v["ms"] / reps, 3) for k, v in p.items() if k != "fused"}


def gine_agg_bytes(batch, layer_in_dims, edge_dim):
    E, N = batch.total_edges, batch.total_nodes
    return sum(E * (4 * f + 4 * edge_dim + 8) + N * (4 * f * 2 + 8) for f in layer_in_dims)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--graphs", type=int, default=1_000_000)
    ap.add_argument("--large-nodes", type=int, default=2_000_000)
    ap.add_argument("--out", type=str, default=None)
    args = ap.parse_args(argv)
    if args.steps < 10:
        ap.error("--steps must be >= 10")
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_gine.py needs a CUDA device")
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.configs import C2, C5

    card, power = card_info(torch)
    res = dict(bench="gine_layerwise", card=card, power_limit_w=power, graphs=args.graphs,
               steps=args.steps, warmup=args.warmup, model="GINE 3x128 (C2 shape)", runs=[])
    gin = gnnb.build_model(C2, seed=0)
    for ed in (4, 16):
        batch = gnnb.make_molecular_batch(args.graphs, C2.mu_nodes, C2.mu_edges, C2.in_dim,
                                          seed=C2.seed, edge_dim=ed)
        dev = to_device(torch, batch)
        run = dict(edge_dim=ed, nodes=batch.total_nodes, edges=batch.total_edges)
        model = gine_model(gnnb, C2.in_dim, C2.hidden_dim, C2.num_layers, ed, C2.out_dim, C2.pools)
        with gnnb.Engine(model) as eng:
            ms, fwd = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
            assert eng.last_kernel == "layerwise"
            run["gine_ms"] = round(ms, 3)
            run["gine_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
            prof = profile(eng, fwd, args.steps)
            run["gine_profile_ms"] = prof
            fins = [C2.in_dim] + [C2.hidden_dim] * (C2.num_layers - 1)
            nbytes = gine_agg_bytes(batch, fins, ed)
            run["gine_agg_bytes"] = nbytes
            run["gine_agg_gb_per_s"] = round(nbytes / (prof["aggregate"] * 1e-3) / 1e9, 1)
        plain = dict(dev, edge_attr=None)
        # the device entry point picks its kernel from the capacity hints alone: give it the
        # batch's real maxima (as bench.py does), or AUTO cannot choose the fused kernel
        max_n = int(np.diff(batch.node_ptr).max())
        max_e = int(np.diff(batch.edge_ptr).max())
        with gnnb.Engine(gin, max_nodes=max_n, max_edges=max_e, path=gnnb.PATH_LAYERWISE) as eng:
            ms, _ = time_forward(torch, eng, plain, batch, args.steps, args.warmup)
            run["gin_layerwise_ms"] = round(ms, 3)
            run["gin_layerwise_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
        with gnnb.Engine(gin, max_nodes=max_n, max_edges=max_e) as eng:
            ms, _ = time_forward(torch, eng, plain, batch, args.steps, args.warmup)
            run["gin_auto_kernel"] = eng.last_kernel
            assert eng.last_kernel == "fused-tcgen05", eng.last_kernel
            run["gin_auto_ms"] = round(ms, 3)
            run["gin_auto_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
        res["runs"].append(run)
        print(json.dumps(run), file=sys.stderr, flush=True)
        del dev, batch
        torch.cuda.empty_cache()

    # C5-shaped power-law graph with edge features: hub rows are one sub-warp's serial work
    x, coo = gnnb.make_powerlaw_graph(args.large_nodes, C5.large_avg_degree, C5.in_dim, seed=C5.seed)
    rng = np.random.default_rng(C5.seed)
    ea = rng.random((coo.shape[0], 8), dtype=np.float32) * 2 - 1
    batch = gnnb.GraphBatch.from_graphs([(x, coo, ea)])
    dev = to_device(torch, batch)
    model = gine_model(gnnb, C5.in_dim, C5.hidden_dim, C5.num_layers, 8, C5.out_dim, C5.pools)
    with gnnb.Engine(model) as eng:
        ms, fwd = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
        res["large"] = dict(shape="C5 power-law", nodes=batch.total_nodes, edges=batch.total_edges,
                            edge_dim=8, layers=C5.num_layers, ms_per_forward=round(ms, 3),
                            max_in_degree=int(np.bincount(coo[:, 1]).max()),
                            hub_rows="unbucketed (one sub-warp per row)",
                            in_degrees="run lengths of the sorted destination keys",
                            profile_ms=profile(eng, fwd, args.steps))
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
