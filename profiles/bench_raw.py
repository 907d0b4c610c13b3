"""profiles/bench_raw.py -- ms per training step of the plain LightGCN baseline (RAW, lightgcn.py) on one GPU.

    python profiles/bench_raw.py OUT.json [--workloads C2,C4] [--steps 20] [--warmup 5] [--rounds 3]   (GPU)

One step is bench.py's: 4096 batch users, uniform negatives from a TripleSampler on the NormAdj graph (credibility 1,
build_norm_adj), K = 3 layers in Jacobi order, BPR + L2 (1e-4), Adam (lr 1e-3).  It is taken three ways:

    raw_trainstep   TrainStep(RawLightGCN), replaying its captured CUDA graph
    cu_trainstep    TrainStep(CredLightGCN) on the same graph: the two-table model, the same kernels (reference point)
    raw_autograd    the route a user of RawLightGCN has without TrainStep: get_user_item_emb + bpr_loss + backward
                    through the autograd wrappers + torch.optim.Adam over emb.weight, eager, sampler as above

C2 (d = 64) keeps its tables in L2; C4 (10 M x 2 M x 160 M train edges, d = 128) is HBM-bound and its TrainSteps
take the item frontier and the deferred last layer.  Each step is timed by CUDA events around it, with L2 overwritten
(a 256 MiB fill) before it, as bench.py's `value`.  The two TrainSteps are built, captured, timed and freed in turn,
`rounds` times (at C4 two of them side by side leave too little room); the autograd route runs once, after them.
The card's name and power limit are read in the same process.
"""
import argparse
import json
import pathlib
import subprocess
import sys

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

BATCH, K, REG, LR = 4096, 3, 1e-4, 1e-3


def card(index):
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                          "-i", str(index)], capture_output=True, text=True).stdout.strip()
    f = [x.strip() for x in out.split(",")]
    return {"torch_name": torch.cuda.get_device_name(index), "name": f[0] if f[0] else None,
            "power_limit": f[1] if len(f) > 1 else None, "clocks_max_sm": f[2] if len(f) > 2 else None}


def setup(name, dev):
    from credgcn import graph, synth
    big = name in ("C4", "C5")
    sg = synth.make_graph_device(name, dev) if big else synth.make_graph(name)
    U, I, E = sg.num_users, sg.num_items, int(sg.train_edges.shape[1])
    adj = graph.build_norm_adj(sg.train_edges, U, I, dev)
    sg.train_edges = sg.val_edges = sg.test_edges = None
    torch.cuda.empty_cache()
    train_users = torch.nonzero(adj.graph.deg_u > 0).reshape(-1).cpu().numpy()
    np.random.default_rng(42).shuffle(train_users)                    # bench.py run_single: same batches
    n_batches = min(max(len(train_users) // BATCH, 1), 64)
    batches = [torch.from_numpy(train_users[s * BATCH:(s + 1) * BATCH]).to(dev) for s in range(n_batches)]
    return dict(adj=adj, d=synth.SHAPES[name]["emb_dim"], batches=batches, U=U, I=I, E=E, nnz=adj.graph.nnz)


def timed(step_fn, batches, steps, warmup, flush):
    for s in range(warmup):
        step_fn(batches[s % len(batches)])
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s, (a, b) in enumerate(ev):
        flush.fill_(s & 0xff)
        a.record()
        step_fn(batches[s % len(batches)])
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def net_of(kind, adj, d, dev):
    from credgcn import model
    g = adj.graph
    torch.manual_seed(42)
    if kind == "cu":
        return model.CredLightGCN(g.num_users, g.num_items, d, K, g.operator("C"), g.operator("A")).to(dev)
    return model.RawLightGCN(g.num_users, g.num_items, d, K, adj).to(dev)


def trainstep_ms(kind, w, dev, args, flush):
    from credgcn import model, sampler
    net = net_of(kind, w["adj"], w["d"], dev)
    st = model.TrainStep(net, lr=LR, reg_weight=REG, sampler=sampler.TripleSampler(w["adj"].graph, None, seed=42))
    st.capture(BATCH, preserve_state=False)
    ms = timed(st.step, w["batches"], args.steps, args.warmup, flush)
    info = {"deferred_last_layer": bool(st._defer_final), "loss_finite": bool(torch.isfinite(st.step(w["batches"][0])))}
    del st, net
    torch.cuda.empty_cache()
    return ms, info


def autograd_ms(w, dev, args, flush):
    from credgcn import sampler
    net = net_of("raw", w["adj"], w["d"], dev)
    samp = sampler.TripleSampler(w["adj"].graph, None, seed=42)
    opt = torch.optim.Adam(net.parameters(), lr=LR)

    def step(users):
        pos, neg = samp.sample(users)
        opt.zero_grad()
        ue, ie = net.get_user_item_emb()
        loss = net.bpr_loss(users, pos, neg, ue, ie, REG)
        loss.backward()
        opt.step()
        return loss
    ms = timed(step, w["batches"], args.steps, args.warmup, flush)
    del opt, net
    torch.cuda.empty_cache()
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--workloads", default="C2,C4")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_raw.py needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    out = {"card": card(dev.index), "batch_users": BATCH, "num_layers": K, "steps": args.steps,
           "warmup": args.warmup, "rounds": args.rounds, "workloads": {}}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for name in args.workloads.split(","):
        w = setup(name, dev)
        res = {k: w[k] for k in ("U", "I", "E", "nnz", "d")}
        rounds = {"raw_trainstep": [], "cu_trainstep": []}
        for _ in range(args.rounds):
            for kind in ("raw", "cu"):
                ms, info = trainstep_ms(kind, w, dev, args, flush)
                rounds[f"{kind}_trainstep"].append(float(np.median(ms)))
                res[f"{kind}_trainstep_info"] = info
        for k, v in rounds.items():
            res[k] = {"median_ms_per_round": v, "ms_per_step": float(np.median(v))}
        ms = autograd_ms(w, dev, args, flush)
        res["raw_autograd"] = {"ms_per_step": float(np.median(ms)), "ms_all": ms}
        res["raw_over_cu"] = res["raw_trainstep"]["ms_per_step"] / res["cu_trainstep"]["ms_per_step"]
        res["autograd_over_raw_trainstep"] = res["raw_autograd"]["ms_per_step"] / res["raw_trainstep"]["ms_per_step"]
        out["workloads"][name] = res
        print(json.dumps({name: {k: v for k, v in res.items() if not k.endswith("_info")}}), flush=True)
        del w
        torch.cuda.empty_cache()
    pathlib.Path(args.out).write_text(json.dumps(out, indent=1))
    print(json.dumps(out["card"]))


if __name__ == "__main__":
    main()
