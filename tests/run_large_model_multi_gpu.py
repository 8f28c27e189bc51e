#!/usr/bin/env python
"""Row-partitioned GIN, SAGE or PNA model (C5's shape) over N GPUs (per-layer halo exchange,
transport p2p or nccl), checked -- at a size the CPU oracle finishes in seconds -- against the
oracle; the GIN / SAGE / PNA counterpart of tests/run_large_multi_gpu.py (GCN).
tests/test_gpu_multi_convs.py launches it under torchrun; by hand on a multi-GPU box:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29511 tests/run_large_model_multi_gpu.py --conv pna [--nodes 200000] [--bench]

With --bench on one process it also times the single-GPU model handle (layerwise path) on the same
graph, and it reports the card's name and power limit.
"""
import argparse
import dataclasses
import json
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=80000)
    ap.add_argument("--bench", action="store_true")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--transport", default="auto", choices=["auto", "p2p", "nccl"])
    ap.add_argument("--conv", required=True, choices=["gin", "sage", "pna"])
    args = ap.parse_args()

    import torch
    import torch.distributed as dist

    import gnn_builder_b200 as gnnb
    from gnn_builder_b200.configs import C5
    from gnn_builder_b200.data import pna_delta_from_histogram
    from gnn_builder_b200.distributed import LargeGraphModel, RowPartition

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.nodes - args.nodes % world
    w = dataclasses.replace(C5, conv=args.conv, out_dim=16)
    x, coo = gnnb.make_powerlaw_graph(n, 16, w.in_dim, seed=5, max_degree=5000)
    delta = (pna_delta_from_histogram(np.bincount(np.bincount(coo[:, 1], minlength=n)))
             if args.conv == "pna" else 1.0)
    model = gnnb.build_model(w, pna_delta=delta, seed=1)
    part = RowPartition(n, world)
    r0, r1 = part.rows(rank)
    runner = LargeGraphModel(model, n, rank, world, dist=dist if world > 1 else None,
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
    result = {"rank": rank, "world": world, "conv": args.conv, "nodes": n, "edges": int(coo.shape[0]),
              "stats": runner.stats, "bit_identical_rerun": same}
    if rank == 0 and n <= 200000:
        from oracle import Oracle

        orc = Oracle()
        ref, ref_emb = orc.model_forward(model.describe(),
                                         list(model.named_parameter_arrays().values()), x, coo,
                                         return_node_emb=True)
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


def _time_model_handle(gnnb, model, x, coo, steps):
    """ms per forward of the same model and graph through the single-GPU model handle (layerwise
    path, inputs already on the device)"""
    import torch

    n, E = x.shape[0], coo.shape[0]
    dx, dcoo = torch.from_numpy(x).cuda(), torch.from_numpy(coo).cuda()
    dn = torch.tensor([0, n], dtype=torch.int64, device="cuda")
    de = torch.tensor([0, E], dtype=torch.int64, device="cuda")
    dout = torch.empty((1, model.describe()["mlp_out"]), device="cuda")
    with gnnb.Engine(model, path=gnnb.PATH_LAYERWISE) as eng:
        stream = torch.cuda.ExternalStream(eng.stream)
        for _ in range(2):
            eng.run_device(dx, dcoo, dn, de, dout, 1, n, E)
        eng.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(steps):
            eng.run_device(dx, dcoo, dn, de, dout, 1, n, E)
        ev1.record(stream)
        eng.synchronize()
        return ev0.elapsed_time(ev1) / steps


if __name__ == "__main__":
    main()
