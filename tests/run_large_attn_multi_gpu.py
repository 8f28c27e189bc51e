#!/usr/bin/env python
"""Row-partitioned GAT or GATv2 model (C5's widths: 2 x 128 convs, --heads heads) over N GPUs
(LargeGraphAttentionModel: per-layer exchange of the layer GEMM's output, transport p2p or nccl);
the attention counterpart of tests/run_large_model_multi_gpu.py (GIN / SAGE / PNA).  Up to 200 000
nodes rank 0 checks against the float64 restatements of tests/test_gat_model_cpu.py /
test_gatv2_model_cpu.py; above that, rank 0 checks its rows and the pooled output against the
single-GPU model handle on the full graph, so full-size parity holds at every GPU count.
tests/test_gpu_multi_attn.py launches it under torchrun; by hand on a multi-GPU box:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29511 tests/run_large_attn_multi_gpu.py --conv gat [--nodes 2000000] [--bench]

With --bench it times the forward, times the per-layer exchanges alone (on more than one GPU),
reports the halo rows and bytes every layer moves over all ranks, on one process also times the
single-GPU model handle (layerwise path) on the same graph, and reports the card's name and power
limit.
"""
import argparse
import dataclasses
import functools
import json
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=80000)
    ap.add_argument("--bench", action="store_true")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--transport", default="auto", choices=["auto", "p2p", "nccl"])
    ap.add_argument("--conv", required=True, choices=["gat", "gatv2"])
    ap.add_argument("--heads", type=int, default=4)
    args = ap.parse_args()

    import torch
    import torch.distributed as dist

    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.configs import C5
    from gnn_builder_b200.distributed import LargeGraphAttentionModel, RowPartition
    from run_large_model_multi_gpu import _time_model_handle

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.nodes - args.nodes % world
    w = dataclasses.replace(C5, out_dim=16)
    x, coo = gnnb.make_powerlaw_graph(n, 16, w.in_dim, seed=5, max_degree=5000)
    model = _model(gnnb, w, args.conv, args.heads)
    part = RowPartition(n, world)
    r0, r1 = part.rows(rank)
    runner = LargeGraphAttentionModel(model, n, rank, world, dist=dist if world > 1 else None,
                                      transport=args.transport)
    runner.setup(part.local_edges(coo, rank))
    x_local = torch.from_numpy(x[r0:r1]).cuda()
    out, emb = runner.forward(x_local, return_embeddings=True)
    torch.cuda.synchronize()
    runner.check_transport()
    # run-to-run: the same input again gives the same bits (fixed reduction order everywhere)
    out_b, emb_b = runner.forward(x_local, return_embeddings=True)
    torch.cuda.synchronize()
    same = bool(torch.equal(out, out_b) and torch.equal(emb, emb_b))
    result = {"rank": rank, "world": world, "conv": args.conv, "heads": args.heads, "nodes": n,
              "edges": int(coo.shape[0]), "stats": runner.stats, "bit_identical_rerun": same}
    if rank == 0:
        if n <= 200000:
            ref, ref_emb = _float64_reference(args.conv, model, x, coo)
            result.update(reference="float64")
        else:
            ref, ref_emb = _handle_forward(gnnb, model, x, coo)
            result.update(reference="model handle")
        err_out = float(np.abs(out.cpu().numpy() - ref).max() / max(1.0, np.abs(ref).max()))
        err_emb = float(np.abs(emb.cpu().numpy() - ref_emb[r0:r1]).max()
                        / max(1.0, np.abs(ref_emb).max()))
        result.update(err_out=err_out, err_emb=err_emb,
                      ok=bool(err_out < 1e-4 and err_emb < 1e-4 and same))
    if args.bench:
        for _ in range(2):
            runner.forward(x_local)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.steps):
            runner.forward(x_local)
        ev1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([ev0.elapsed_time(ev1) / args.steps], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        result.update(ms_per_forward=float(ms.item()),
                      edges_per_sec=float(coo.shape[0] * w.num_layers / (ms.item() * 1e-3)))
        result.update(_exchange_stats(runner, dist, world, args.steps))
        if world == 1:
            result.update(handle_ms_per_forward=_time_model_handle(gnnb, model, x, coo, args.steps))
        if rank == 0:
            import subprocess

            q = subprocess.run(["nvidia-smi", f"--id={local}", "--query-gpu=name,power.limit",
                                "--format=csv,noheader"], capture_output=True, text=True)
            result.update(gpu=q.stdout.strip())
    runner.check_transport()
    if rank == 0:
        print(json.dumps(result), flush=True)
    runner.close()
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and result.get("ok") is False:
        sys.exit(1)


def _model(gnnb, w, conv, heads):
    """GAT / GATv2 with C5's widths: 2 x 128 convs, ReLU, skip, C5's pools, head out w.out_dim"""
    import torch
    import torch.nn as nn

    torch.manual_seed(1)
    cls = gnnb.GATConv_GNNB if conv == "gat" else gnnb.GATv2Conv_GNNB
    head = gnnb.MLP(w.hidden_dim * len(w.pools), w.out_dim, hidden_dim=64, hidden_layers=2,
                    activation=nn.ReLU)
    return gnnb.GNNModel(w.in_dim, None, w.hidden_dim, w.num_layers, w.hidden_dim,
                         functools.partial(cls, heads=heads), nn.ReLU, True,
                         gnnb.GlobalPooling(list(w.pools)), head, None)


def _float64_reference(conv, model, x, coo):
    """float64 restatement of the GAT / GATv2 model: (output [out], node embeddings)"""
    from gnn_builder_b200.data import GraphBatch
    from test_gat_model_cpu import np_gat_forward
    from test_gatv2_model_cpu import np_gatv2_forward

    fwd = np_gat_forward if conv == "gat" else np_gatv2_forward
    out, emb, _ = fwd(model, GraphBatch.from_graphs([(x, coo)]))
    return out[0], emb


def _handle_forward(gnnb, model, x, coo):
    """the single-GPU model handle on the full graph: (output [out], node embeddings)"""
    from gnn_builder_b200.data import GraphBatch

    with gnnb.Engine(model) as eng:
        out = eng.run(GraphBatch.from_graphs([(x, coo)]))
        return out[0], eng.node_embeddings(x.shape[0])


def _exchange_stats(runner, dist, world, steps):
    """the forward's exchanges timed alone (device time, max over ranks) and what every layer moves
    over all ranks"""
    import torch

    L = runner.desc["num_layers"]
    widths = runner.stats["exchanged_floats_per_halo_row"]
    rows = torch.tensor([runner.stats["halo_rows"]], dtype=torch.int64, device="cuda")
    res = {}
    if world > 1:
        dist.all_reduce(rows)

        def exchanges():
            for k in range(L):
                runner._exchange(k, widths[k])
                runner._arrived()

        exchanges()
        torch.cuda.synchronize()
        dist.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            exchanges()
        ev1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([ev0.elapsed_time(ev1) / steps], device="cuda")
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        res["exchange_ms_per_forward"] = float(ms.item())
    res["halo_rows_per_layer_all_ranks"] = int(rows.item())
    res["halo_bytes_per_layer_all_ranks"] = [int(rows.item()) * 4 * wd for wd in widths]
    return res


if __name__ == "__main__":
    main()
