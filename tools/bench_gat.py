"""GAT model throughput on the layerwise path, next to the C2 GIN model on the same batch.

Builds GAT 3x128 with 4 heads (C2's shape) on 1M QM9-shaped graphs, device-resident, and times
forwards with CUDA events on the model handle's stream after warm-up.  On the same batch it also
times C2's GIN model forced to the layerwise path and on AUTO (the fused tcgen05 kernel).  A separate
profiled pass gives the per-class split (tables, aggregate, GEMM, pool) and the attention
aggregation's algorithmic bytes over its measured time.  Then, at edge_dim 4 and 16 on the same
graphs with bond features, GAT with edge attention (GATConv's edge_dim) beside plain GAT and the
C2-shaped GINE model, with the edge-logit pass's algorithmic bytes over its measured time.  Then GAT
2x128 with 4 heads on the C5-shaped power-law graph (2M nodes), whose hub rows are bucketed, with
the C5 GCN model's aggregation on the same graph beside it, and GAT with edge attention at edge_dim
8 on that graph.  Reads the card name and power limit in the same run.  Prints one JSON line; needs
a CUDA device.

    python tools/bench_gat.py [--steps 10] [--warmup 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import functools
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_gine import (card_info, gine_agg_bytes, gine_model, profile, time_forward,  # noqa: E402
                        to_device)

HEADS = 4


def gat_model(gnnb, in_dim, hidden, layers, out_dim, pools, seed=0, edge_dim=None):
    import torch
    import torch.nn as nn

    torch.manual_seed(seed)
    head = gnnb.MLP(hidden * len(pools), out_dim, hidden_dim=64, hidden_layers=2,
                    activation=nn.ReLU)
    conv = functools.partial(gnnb.GATConv_GNNB, heads=HEADS)
    if edge_dim is not None:
        conv = functools.partial(gnnb.GATConv_GNNB, heads=HEADS, edge_dim=edge_dim)
    return gnnb.GNNModel(in_dim, edge_dim, hidden, layers, hidden, conv, nn.ReLU, True,
                         gnnb.GlobalPooling(list(pools)), head, None)


def gat_agg_bytes(batch, layers, width, heads):
    """per edge: the neighbor index, the source's H logits and its H*C row; per node: offset and
    degree, the H destination logits, the output row, and the skip row on interior layers"""
    E, N = batch.total_edges, batch.total_nodes
    total = 0
    for k in range(layers):
        skip = 0 < k < layers - 1
        total += E * (4 + 4 * width + 4 * heads)
        total += N * (8 + 4 * heads + 4 * width + (4 * width if skip else 0))
    return total


def gat_edge_logits_bytes(batch, layers, heads, edge_dim):
    """the once-per-run edge-logit pass: per edge the edge index, the neighbor index, the edge_attr
    row and the L*H logits written; per node offset and degree and the L*H self-loop logits"""
    E, N, LH = batch.total_edges, batch.total_nodes, layers * heads
    return E * (4 + 4 + 4 * edge_dim + 4 * LH) + N * (8 + 4 * LH)


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
        raise SystemExit("bench_gat.py needs a CUDA device")
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.configs import C2, C5

    card, power = card_info(torch)
    res = dict(bench="gat_layerwise", card=card, power_limit_w=power, graphs=args.graphs,
               steps=args.steps, warmup=args.warmup, model=f"GAT 3x128, {HEADS} heads (C2 shape)")

    batch = gnnb.make_molecular_batch(args.graphs, C2.mu_nodes, C2.mu_edges, C2.in_dim,
                                      seed=C2.seed)
    dev = to_device(torch, batch)
    run = dict(nodes=batch.total_nodes, edges=batch.total_edges)
    model = gat_model(gnnb, C2.in_dim, C2.hidden_dim, C2.num_layers, C2.out_dim, C2.pools)
    with gnnb.Engine(model) as eng:
        ms, fwd = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
        assert eng.last_kernel == "layerwise"
        run["gat_ms"] = round(ms, 3)
        run["gat_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
        prof = profile(eng, fwd, args.steps)
        run["gat_profile_ms"] = prof
        nbytes = gat_agg_bytes(batch, C2.num_layers, C2.hidden_dim, HEADS)
        run["gat_agg_bytes"] = nbytes
        run["gat_agg_gb_per_s"] = round(nbytes / (prof["aggregate"] * 1e-3) / 1e9, 1)
    gin = gnnb.build_model(C2, seed=0)
    # the device entry point picks its kernel from the capacity hints alone: give it the batch's
    # real maxima (as bench.py does), or AUTO cannot choose the fused kernel
    max_n = int(np.diff(batch.node_ptr).max())
    max_e = int(np.diff(batch.edge_ptr).max())
    with gnnb.Engine(gin, max_nodes=max_n, max_edges=max_e, path=gnnb.PATH_LAYERWISE) as eng:
        ms, _ = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
        run["gin_layerwise_ms"] = round(ms, 3)
        run["gin_layerwise_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
    with gnnb.Engine(gin, max_nodes=max_n, max_edges=max_e) as eng:
        ms, _ = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
        run["gin_auto_kernel"] = eng.last_kernel
        assert eng.last_kernel == "fused-tcgen05", eng.last_kernel
        run["gin_auto_ms"] = round(ms, 3)
        run["gin_auto_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
    res["batch"] = run
    print(json.dumps(run), file=sys.stderr, flush=True)
    del dev, batch
    torch.cuda.empty_cache()

    # edge attention at edge_dim 4 and 16: the same graphs with bond features (x and coo do not
    # depend on edge_dim), beside plain GAT and the C2-shaped GINE model on the same batch
    res["edge_runs"] = []
    L = C2.num_layers
    for ed in (4, 16):
        batch = gnnb.make_molecular_batch(args.graphs, C2.mu_nodes, C2.mu_edges, C2.in_dim,
                                          seed=C2.seed, edge_dim=ed)
        dev = to_device(torch, batch)
        run = dict(edge_dim=ed, nodes=batch.total_nodes, edges=batch.total_edges)
        model = gat_model(gnnb, C2.in_dim, C2.hidden_dim, L, C2.out_dim, C2.pools, edge_dim=ed)
        with gnnb.Engine(model) as eng:
            ms, fwd = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
            assert eng.last_kernel == "layerwise"
            run["gat_edges_ms"] = round(ms, 3)
            run["gat_edges_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
            prof = profile(eng, fwd, args.steps)
            run["gat_edges_profile_ms"] = prof
            lb = gat_edge_logits_bytes(batch, L, HEADS, ed)
            run["edge_logits_bytes"] = lb
            run["edge_logits_gb_per_s"] = round(lb / (prof["edge_logits"] * 1e-3) / 1e9, 1)
            ab = gat_agg_bytes(batch, L, C2.hidden_dim, HEADS) + L * (
                batch.total_edges + batch.total_nodes) * 4 * HEADS
            run["gat_edges_agg_bytes"] = ab
            run["gat_edges_agg_gb_per_s"] = round(ab / (prof["aggregate"] * 1e-3) / 1e9, 1)
        plain = dict(dev, edge_attr=None)
        with gnnb.Engine(gat_model(gnnb, C2.in_dim, C2.hidden_dim, L, C2.out_dim, C2.pools)) as eng:
            ms, _ = time_forward(torch, eng, plain, batch, args.steps, args.warmup)
            run["gat_ms"] = round(ms, 3)
            run["gat_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
        gine = gine_model(gnnb, C2.in_dim, C2.hidden_dim, L, ed, C2.out_dim, C2.pools)
        with gnnb.Engine(gine) as eng:
            ms, fwd = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
            run["gine_ms"] = round(ms, 3)
            run["gine_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
            prof = profile(eng, fwd, args.steps)
            run["gine_profile_ms"] = prof
            nbytes = gine_agg_bytes(batch, [C2.in_dim] + [C2.hidden_dim] * (L - 1), ed)
            run["gine_agg_bytes"] = nbytes
            run["gine_agg_gb_per_s"] = round(nbytes / (prof["aggregate"] * 1e-3) / 1e9, 1)
        res["edge_runs"].append(run)
        print(json.dumps(run), file=sys.stderr, flush=True)
        del dev, batch, plain
        torch.cuda.empty_cache()

    # C5-shaped power-law graph: GAT with bucketed hub rows, and the C5 GCN model beside it
    x, coo = gnnb.make_powerlaw_graph(args.large_nodes, C5.large_avg_degree, C5.in_dim, seed=C5.seed)
    batch = gnnb.GraphBatch.from_graphs([(x, coo)])
    dev = to_device(torch, batch)
    model = gat_model(gnnb, C5.in_dim, C5.hidden_dim, C5.num_layers, C5.out_dim, C5.pools)
    large = dict(shape="C5 power-law", nodes=batch.total_nodes, edges=batch.total_edges,
                 layers=C5.num_layers, max_in_degree=int(np.bincount(coo[:, 1]).max()))
    with gnnb.Engine(model) as eng:
        ms, fwd = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
        large["gat_ms_per_forward"] = round(ms, 3)
        prof = profile(eng, fwd, args.steps)
        large["gat_profile_ms"] = prof
        large["gat_agg_ms_per_layer"] = round(prof["aggregate"] / C5.num_layers, 3)
    with gnnb.Engine(gnnb.build_model(C5, seed=0)) as eng:
        ms, fwd = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
        large["gcn_ms_per_forward"] = round(ms, 3)
        prof = profile(eng, fwd, args.steps)
        large["gcn_profile_ms"] = prof
        large["gcn_agg_ms_per_layer"] = round(prof["aggregate"] / C5.num_layers, 3)
    rng = np.random.default_rng(C5.seed)
    ea = rng.random((coo.shape[0], 8), dtype=np.float32) * 2 - 1
    dev["edge_attr"] = torch.from_numpy(ea).cuda()
    batch = gnnb.GraphBatch(batch.x, batch.coo, batch.node_ptr, batch.edge_ptr, ea)
    model = gat_model(gnnb, C5.in_dim, C5.hidden_dim, C5.num_layers, C5.out_dim, C5.pools,
                      edge_dim=8)
    with gnnb.Engine(model) as eng:
        ms, fwd = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
        large["gat_edges8_ms_per_forward"] = round(ms, 3)
        prof = profile(eng, fwd, args.steps)
        large["gat_edges8_profile_ms"] = prof
        lb = gat_edge_logits_bytes(batch, C5.num_layers, HEADS, 8)
        large["edge_logits_gb_per_s"] = round(lb / (prof["edge_logits"] * 1e-3) / 1e9, 1)
    res["large"] = large
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
