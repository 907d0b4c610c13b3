"""Cost of the sharded epoch loop on B200s: ms/step of train_on_arrays_sharded's step (device batch selection +
padded batch, ShardedTrainStep.step_selected) against bare ShardedTrainStep.step replays of full local batches on
the same partition, alternated in blocks; and (--epoch) one timed C2 epoch plus evaluation.

    torchrun --nproc-per-node 2 profiles/sharded_epoch.py --workload C4 --out out/sharded_epoch_c4x2.json
    torchrun --nproc-per-node 8 profiles/sharded_epoch.py --workload C5 --out out/sharded_epoch_c5x8.json
    torchrun --nproc-per-node 2 profiles/sharded_epoch.py --workload C2 --epoch --out out/epoch_c2x2.json

Prints (and writes) one JSON object from rank 0 with the card's name and power limit read in the same run."""
import argparse
import json
import os
import pathlib
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="C4", choices=["C2", "C4", "C5"])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--blocks", type=int, default=6)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--epoch", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    from credgcn import config, synth
    from credgcn.sharded import (ShardedTrainStep, build_local_graph, partition_users, shard_edges,
                                 train_on_arrays_sharded)
    shp = synth.SHAPES[a.workload]
    res = {"workload": a.workload, "world": world, "card": card(), "batch": a.batch}
    if a.epoch:
        sg = synth.make_graph(a.workload)
        cfg = config.CFG(variant=shp["variant"], epochs=1, batch_size=a.batch, emb_dim=shp["emb_dim"],
                         num_layers=shp["num_layers"], eval_mode="full", device=str(dev))
        config.cfg = cfg
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        train_on_arrays_sharded(sg.train_edges, sg.val_edges, sg.test_edges, sg.num_users, sg.num_items, sg.cred,
                                None, cfg)
        torch.cuda.synchronize()
        res["epoch_plus_val_and_test_eval_s"] = time.perf_counter() - t0
    else:
        full = synth.make_graph_device(a.workload, dev)
        U, I = full.num_users, full.num_items
        deg = torch.bincount(full.train_edges[0].to(torch.int64), minlength=U).cpu().numpy()
        bounds = partition_users(deg, world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        edges = shard_edges(full.train_edges.cpu().numpy(), bounds, rank)
        cred = full.cred[lo:hi].contiguous()
        del full
        gl = build_local_graph(edges, hi - lo, I, cred, shp["variant"], dev)
        torch.manual_seed(0)
        d = shp["emb_dim"]
        step = ShardedTrainStep(gl, torch.nn.init.xavier_uniform_(torch.empty(hi - lo, d, device=dev)),
                                torch.nn.init.xavier_uniform_(torch.empty(I, d, device=dev)), shp["num_layers"],
                                shp["order"], mix_pop=None if shp["variant"] == "cu" else 0.7, exchange="auto",
                                max_batch=a.batch)
        train_users = np.flatnonzero(deg > 0)
        rng = np.random.default_rng(0)
        rng.shuffle(train_users)
        step.plan_epochs(len(train_users), lo, hi)
        step.begin_epoch(train_users)
        mine = train_users[(train_users >= lo) & (train_users < hi)][: a.batch // world] - lo
        users = torch.as_tensor(np.resize(mine, a.batch // world), device=dev)
        # two graphs of one step object: the bare step over a full local batch, and the epoch step
        step.capture(users.numel())
        g_bare, l_bare, u_bare = step._graph, step._g_loss, step._g_users   # (kept alive: the graph reads them)
        u_bare.copy_(users)
        step.capture(a.batch, selected=True)
        g_sel = step._graph
        times = {"bare_step": [], "epoch_step": []}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for b in range(2 * a.blocks):
            kind = "bare_step" if b % 2 == 0 else "epoch_step"
            g = g_bare if kind == "bare_step" else g_sel
            step.begin_epoch(train_users)
            dist.barrier()
            ev[0].record()
            for _ in range(a.steps):
                g.replay()
            ev[1].record()
            torch.cuda.synchronize()
            t = torch.tensor([ev[0].elapsed_time(ev[1]) / a.steps], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            times[kind].append(float(t.item()))
        del l_bare, u_bare
        step.check()
        res.update({k + "_ms": {"median": float(np.median(v)), "min": min(v), "max": max(v), "blocks": v}
                    for k, v in times.items()})
        step.close()
    if rank == 0:
        print(json.dumps(res))
        if a.out:
            pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
            pathlib.Path(a.out).write_text(json.dumps(res, indent=1))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
