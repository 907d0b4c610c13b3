"""Deep full-rank top-K timing: the k = 128 fp32 kernel against the deep path (csrc/eval_deep.cu) at k in
{129, 500, 1000, 4096}, on C2 (all 31,668 users, propagated embeddings) and on a C4-shaped catalogue (2 M items,
d = 128, random tables, 4,096 users with 20 random train items each).

CUDA events around each call; every k is warmed up, then the repeats alternate over the k values in one process.
The card's name and power limit are read in the same run and written beside the numbers.
    python profiles/bench_topk_deep.py [--reps 7] [--out FILE]"""
import argparse
import json
import pathlib
import subprocess
import sys

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
import numpy as np
import torch

from credgcn import evaluate, graph, model, synth

KS = (128, 129, 500, 1000, 4096)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def c2_inputs(dev):
    sg = synth.make_graph("C2")
    shp = synth.SHAPES["C2"]
    gr = graph.build_graph(sg.train_edges, sg.num_users, sg.num_items, sg.cred, shp["variant"], dev)
    torch.manual_seed(0)
    eu = torch.nn.init.xavier_uniform_(torch.empty(sg.num_users, shp["emb_dim"])).to(dev)
    ei = torch.nn.init.xavier_uniform_(torch.empty(sg.num_items, shp["emb_dim"])).to(dev)
    fu, fi = model.propagate_forward(gr, eu, ei, shp["num_layers"], shp["order"])
    return fu, fi, torch.arange(sg.num_users, device=dev), (gr.samp_indptr, gr.samp_idx)


def c4_inputs(dev, U=4096, I=2_000_000, d=128):
    g = torch.Generator(device=dev).manual_seed(4)
    fu = torch.randn(U, d, device=dev, generator=g) * 0.1
    fi = torch.randn(I, d, device=dev, generator=g) * 0.1
    idx = torch.sort(torch.randint(0, I, (U, 20), device=dev, dtype=torch.int32, generator=g), dim=1).values
    csr = (torch.arange(0, 20 * U + 1, 20, device=dev, dtype=torch.int64), idx.reshape(-1).contiguous())
    return fu, fi, torch.arange(U, device=dev), csr


def run(name, fu, fi, users, csr, reps):
    out = {"workload": name, "users": int(users.numel()), "items": int(fi.shape[0]), "d": int(fi.shape[1]),
           "item_table_MB": round(fi.numel() * 4 / 2**20, 1), "fma_per_user": int(fi.shape[0]) * int(fi.shape[1])}
    ref = {}
    for K in KS:                                       # warm-up of every shape, and the prefix check
        for _ in range(2):
            ids, sc = evaluate.topk_device(fu, fi, users, csr, K)
        ref[K] = ids[:, :128].clone()
    torch.cuda.synchronize()
    prefix_ok = all(torch.equal(ref[K], ref[128]) for K in KS)
    times = {K: [] for K in KS}
    for _ in range(reps):                              # alternate the k values inside every repeat
        for K in KS:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            evaluate.topk_device(fu, fi, users, csr, K)
            b.record()
            torch.cuda.synchronize()
            times[K].append(a.elapsed_time(b))
    med = {K: float(np.median(t)) for K, t in times.items()}
    out["ms"] = {str(K): {"median": round(med[K], 3), "min": round(min(times[K]), 3), "max": round(max(times[K]), 3)}
                 for K in KS}
    out["ratio_to_k128"] = {str(K): round(med[K] / med[128], 3) for K in KS if K != 128}
    out["prefix_128_equal"] = prefix_ok
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_topk_deep.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"card": card(), "kernels": {"128": "k_eval_fp32", "others": "k_eval_deep + k_eval_deep_finish"},
           "note": "C2 item table fits L2 (126 MB); the C4-shaped table (1 GB) does not. Median of alternated repeats."}
    res["C2"] = run("C2", *c2_inputs(dev), args.reps)
    torch.cuda.empty_cache()
    res["C4_shape"] = run("C4-shaped random", *c4_inputs(dev), args.reps)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
