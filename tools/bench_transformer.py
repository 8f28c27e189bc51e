"""TransformerConv model throughput on the layerwise path, next to GAT and GATv2 on the same batch.

Builds TransformerConv 3x128 with 4 heads (C2's shape) on 1M QM9-shaped graphs, device-resident,
and times forwards with CUDA events on the model handle's stream after warm-up, beside GAT and GATv2
3x128 with 4 heads on the same batch.  At edge_dim 4 and 16, on the same graphs with bond features,
each conv with ``edge_dim``.  Then TransformerConv 2x128 with 4 heads on the C5-shaped power-law
graph (2M nodes), whose hub rows are bucketed, beside GAT and GATv2.  Separate profiled passes give
the per-class split (tables, aggregate, GEMM, pool) and the TransformerConv aggregation's algorithmic
bytes over its measured time.  Reads the card name and power limit in the same run.  Prints one JSON
line; needs a CUDA device.

    python tools/bench_transformer.py [--steps 10] [--warmup 3] [--out result.json]
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

from bench_gat import HEADS, gat_model  # noqa: E402
from bench_gatv2 import gatv2_model  # noqa: E402
from bench_gine import card_info, profile, time_forward, to_device  # noqa: E402


def transformer_model(gnnb, in_dim, hidden, layers, out_dim, pools, seed=0, edge_dim=None):
    import torch
    import torch.nn as nn

    torch.manual_seed(seed)
    head = gnnb.MLP(hidden * len(pools), out_dim, hidden_dim=64, hidden_layers=2,
                    activation=nn.ReLU)
    kw = dict(heads=HEADS) if edge_dim is None else dict(heads=HEADS, edge_dim=edge_dim)
    conv = functools.partial(gnnb.TransformerConv_GNNB, **kw)
    return gnnb.GNNModel(in_dim, edge_dim, hidden, layers, hidden, conv, nn.ReLU, True,
                         gnnb.GlobalPooling(list(pools)), head, None)


def transformer_agg_bytes(batch, layers, width, edge_dim=None):
    """per edge: the neighbor index and the source's k and v rows (2 H*C), with edge features its
    ef_sorted row (lde floats); per node: offset and degree, its q row, its root row r (which already
    holds the model's skip) and the output row"""
    E, N = batch.total_edges, batch.total_nodes
    lde = 0 if edge_dim is None else (edge_dim + 3) // 4 * 4
    per_layer = E * (4 + 8 * width + 4 * lde) + N * (8 + 12 * width)
    return layers * per_layer


def _timed(gnnb, torch, model, dev, batch, args, prefix, run, agg_bytes=None):
    with gnnb.Engine(model) as eng:
        ms, fwd = time_forward(torch, eng, dev, batch, args.steps, args.warmup)
        assert eng.last_kernel == "layerwise"
        run[f"{prefix}_ms"] = round(ms, 3)
        run[f"{prefix}_graphs_per_s"] = round(batch.n_graphs / ms * 1e3)
        prof = profile(eng, fwd, args.steps)
        run[f"{prefix}_profile_ms"] = prof
        if agg_bytes is not None:
            run[f"{prefix}_agg_bytes"] = agg_bytes
            run[f"{prefix}_agg_tb_per_s"] = round(agg_bytes / (prof["aggregate"] * 1e-3) / 1e12, 3)


def _three(gnnb, torch, dev, batch, args, run, in_dim, width, layers, out_dim, pools, ed=None):
    _timed(gnnb, torch, transformer_model(gnnb, in_dim, width, layers, out_dim, pools, edge_dim=ed),
           dev, batch, args, "transformer", run, transformer_agg_bytes(batch, layers, width, ed))
    _timed(gnnb, torch, gat_model(gnnb, in_dim, width, layers, out_dim, pools, edge_dim=ed),
           dev, batch, args, "gat", run)
    _timed(gnnb, torch, gatv2_model(gnnb, in_dim, width, layers, out_dim, pools, edge_dim=ed),
           dev, batch, args, "gatv2", run)


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
        raise SystemExit("bench_transformer.py needs a CUDA device")
    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.configs import C2, C5

    card, power = card_info(torch)
    res = dict(bench="transformer_layerwise", card=card, power_limit_w=power, graphs=args.graphs,
               steps=args.steps, warmup=args.warmup,
               model=f"TransformerConv 3x128, {HEADS} heads (C2 shape), beside GAT and GATv2")
    L, W = C2.num_layers, C2.hidden_dim

    # plain, then edge_dim 4 and 16: the same graphs (x and coo do not depend on edge_dim)
    res["runs"] = []
    for ed in (None, 4, 16):
        batch = gnnb.make_molecular_batch(args.graphs, C2.mu_nodes, C2.mu_edges, C2.in_dim,
                                          seed=C2.seed, edge_dim=ed or 0)
        dev = to_device(torch, batch)
        run = dict(edge_dim=ed, nodes=batch.total_nodes, edges=batch.total_edges)
        _three(gnnb, torch, dev, batch, args, run, C2.in_dim, W, L, C2.out_dim, C2.pools, ed)
        res["runs"].append(run)
        print(json.dumps(run), file=sys.stderr, flush=True)
        del dev, batch
        torch.cuda.empty_cache()

    # C5-shaped power-law graph: bucketed hub rows
    x, coo = gnnb.make_powerlaw_graph(args.large_nodes, C5.large_avg_degree, C5.in_dim, seed=C5.seed)
    batch = gnnb.GraphBatch.from_graphs([(x, coo)])
    dev = to_device(torch, batch)
    large = dict(shape="C5 power-law", nodes=batch.total_nodes, edges=batch.total_edges,
                 layers=C5.num_layers, max_in_degree=int(np.bincount(coo[:, 1]).max()))
    _three(gnnb, torch, dev, batch, args, large, C5.in_dim, C5.hidden_dim, C5.num_layers,
           C5.out_dim, C5.pools)
    res["large"] = large
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
