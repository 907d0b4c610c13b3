"""profiles/frontier.py -- the item frontier of bench.py's C4 batches and what it does to the first adjoint hop.

    python profiles/frontier.py stats OUT.json [--batches N]        (GPU)  |F|, its edges and its hot-set share
    python profiles/frontier.py kernels OUT.json [--tree DIR]       (GPU)  torch.profiler times of one eager C4 step
    python profiles/frontier.py reads OUT.json                      (GPU)  what reading TrainStep.f_u costs; C2 deferral
    python profiles/frontier.py traffic STATS.json                  (CPU)  rewrite launches 5 - 8 of r2_traffic.json

The frontier F of a batch is pos + neg + the train items of the batch users (cgx_batch_frontier): the only rows where
the first item-side adjoint bi' = g_i + A^T g_u can be non-zero.  `stats` builds the C4 graph and the sampler exactly
as bench.py does and measures F over bench's first batches.  `kernels` runs eager training steps (no CUDA graph) of
the package found in --tree (default: this repository) under torch.profiler and lists the SpMM launches of the last
step in launch order.  `reads` times, with CUDA events and under torch.profiler, the first read of f_u after an eager
C4 step (the last layer's products on the rows the step left out), and C2 graph replays with the deferred last layer
forced on and off.  `traffic` replaces the last forward hop (launches 5 and 6, restricted to F and the batch users)
and the two launches of the Gauss-Seidel adjoint at k = 0 in profiles/r2_traffic.json (which bench.py divides by the
propagation time for roofline.frac) with bytes computed from the measured frontier: the ncu capture of those four
launches predates the frontier and no longer describes them.
"""
import argparse
import json
import pathlib
import sys

HERE = pathlib.Path(__file__).resolve().parent
BATCH = 4096


def c4_setup(tree, with_step):
    sys.path.insert(0, str(tree))
    import numpy as np
    import torch
    from credgcn import graph, model, sampler, synth
    dev = torch.device("cuda")
    shp = synth.SHAPES["C4"]
    sg = synth.make_graph_device("C4", dev)
    U, I = sg.num_users, sg.num_items
    gr = graph.build_graph(sg.train_edges, U, I, sg.cred, shp["variant"], dev)
    sg.train_edges = sg.val_edges = sg.test_edges = None
    torch.cuda.empty_cache()
    # bench.py run_single: same seeds, same sampler, same batches
    torch.manual_seed(42)
    samp = sampler.TripleSampler(gr, 0.7, 0.75, 50, seed=42)
    train_users = torch.nonzero(gr.deg_u > 0).reshape(-1).cpu().numpy()
    np.random.default_rng(42).shuffle(train_users)
    n_batches = min(max(len(train_users) // BATCH, 1), 64)
    batches = [torch.from_numpy(train_users[s * BATCH:(s + 1) * BATCH]).to(dev) for s in range(n_batches)]
    step = None
    if with_step:
        net = model.LightGCN(U, I, shp["emb_dim"], shp["num_layers"], gr.operator("A"), gr.operator("C")).to(dev)
        step = model.TrainStep(net, lr=1e-3, reg_weight=1e-4, sampler=samp)
    return dict(torch=torch, np=np, model=model, gr=gr, samp=samp, batches=batches, shp=shp, step=step)


def stats(args):
    e = c4_setup(HERE.parent, False)
    torch, model, gr = e["torch"], e["model"], e["gr"]
    d = e["shp"]["emb_dim"]
    deg_i = (gr.by_item.indptr[1:] - gr.by_item.indptr[:-1]).to(torch.int64)
    n_hot = min((48 << 20) // (4 * d), gr.num_items)             # CredGraph.HOT_BYTES worth of item rows
    hot = torch.zeros(gr.num_items, dtype=torch.bool, device=deg_i.device)
    hot[gr.by_item.perm[:n_hot].long()] = True
    rows = []
    for s, users in enumerate(e["batches"][:args.batches]):
        pos, neg = e["samp"].sample(users, offset=s)
        f = model.batch_frontier(gr, users, pos, neg).bool()
        rows.append(dict(batch=s, front_items=int(f.sum()), front_edges=int(deg_i[f].sum()),
                         front_edges_hot=int(deg_i[f & hot].sum())))
    mean = {k: sum(r[k] for r in rows) / len(rows) for k in rows[0] if k != "batch"}
    by_user, by_item = gr.by_user, gr.by_item
    out = dict(workload="C4", batch_users=BATCH, emb_dim=d, num_users=gr.num_users, num_items=gr.num_items,
               nnz=int(gr.nnz), item_rows_long=by_item.n_long, item_chunks=by_item.n_chunks,
               user_rows_long=by_user.n_long, user_chunks=by_user.n_chunks, hot_item_rows=n_hot,
               gpu=torch.cuda.get_device_name(), mean=mean, batches=rows)
    pathlib.Path(args.out).write_text(json.dumps(out, indent=1))
    print(json.dumps(dict(mean=mean, nnz=out["nnz"], items=out["num_items"])))


def kernels(args):
    e = c4_setup(pathlib.Path(args.tree).resolve(), True)
    torch, step, batches = e["torch"], e["step"], e["batches"]
    for s in range(3):
        step.step(batches[s])
    torch.cuda.synchronize()
    steps = []
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for s in range(3, 3 + args.steps):
            step.step(batches[s])
            torch.cuda.synchronize()
    ev = sorted((k for k in prof.events() if k.device_type == torch.autograd.DeviceType.CUDA),
                key=lambda k: k.time_range.start)
    spmm = [k for k in ev if "k_spmm" in k.name]
    per = len(spmm) // args.steps
    for s in range(args.steps):
        steps.append([dict(kernel=k.name.split("(")[0].replace("void ", "").replace("cgx::", ""),
                           ms=round(k.time_range.elapsed_us() / 1e3, 3)) for k in spmm[s * per:(s + 1) * per]])
    other = [dict(kernel=k.name.split("(")[0].replace("void ", "").replace("cgx::", ""),
                  ms=round(k.time_range.elapsed_us() / 1e3, 3)) for k in ev if "frontier" in k.name]
    out = dict(tree=str(args.tree), gpu=torch.cuda.get_device_name(), spmm_launches_per_step=per, steps=steps,
               frontier_launches=other)
    pathlib.Path(args.out).write_text(json.dumps(out, indent=1))
    for s in steps:
        print(" ".join(f"{l['ms']:.2f}" for l in s))


def _kname(k):
    return k.name.split("(")[0].replace("void ", "").replace("cgx::", "")


def reads(args):
    e = c4_setup(HERE.parent, True)
    torch, step, batches, np = e["torch"], e["step"], e["batches"], e["np"]
    for s in range(3):
        step.step(batches[s])
        step.f_u
    torch.cuda.synchronize()
    assert step._defer_final, "C4 should defer the last layer"
    read_ms = []
    for s in range(3, 3 + args.steps):
        step.step(batches[s])
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step.f_u
        b.record()
        torch.cuda.synchronize()
        read_ms.append(a.elapsed_time(b))
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        step.step(batches[0])
        torch.cuda.synchronize()
        step.f_i
        torch.cuda.synchronize()
    ev = sorted((k for k in prof.events() if k.device_type == torch.autograd.DeviceType.CUDA),
                key=lambda k: k.time_range.start)
    lst = [dict(kernel=_kname(k), ms=round(k.time_range.elapsed_us() / 1e3, 3)) for k in ev]
    # the read starts with the two torch kernels that invert the masks
    n_step = next(j for j, x in enumerate(lst) if "elementwise" in x["kernel"])
    out = dict(gpu=torch.cuda.get_device_name(), first_read_ms_events=read_ms,
               first_read_ms_median=float(np.median(read_ms)),
               step_kernels=[x for x in lst[:n_step] if "spmm" in x["kernel"] or "frontier" in x["kernel"]],
               read_kernels=lst[n_step:])
    del step, e
    torch.cuda.empty_cache()
    # C2 (tables inside L2): graph replays with the deferred last layer forced on / off, alternated
    from credgcn import graph, model, sampler, synth
    shp = synth.SHAPES["C2"]
    sg = synth.make_graph("C2")
    gr = graph.build_graph(sg.train_edges, sg.num_users, sg.num_items, sg.cred, shp["variant"], "cuda")
    users = torch.nonzero(gr.deg_u > 0).reshape(-1)[:4096].cuda()
    sts = {}
    for defer in (False, True):
        torch.manual_seed(42)
        net = model.LightGCN(sg.num_users, sg.num_items, shp["emb_dim"], shp["num_layers"], gr.operator("A"),
                             gr.operator("C")).cuda()
        st = model.TrainStep(net, lr=1e-3, reg_weight=1e-4, sampler=sampler.TripleSampler(gr, 0.7, 0.75, 50, seed=42))
        st._defer_final = defer
        sts[defer] = st.capture(users.numel())
    c2 = {False: [], True: []}
    for rep in range(5):
        for defer, st in sts.items():
            for _ in range(20):
                st.step(users)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(200):
                st.step(users)
            b.record()
            torch.cuda.synchronize()
            c2[defer].append(a.elapsed_time(b) / 200)
    out["c2_ms_per_step"] = {"eager_last_layer": c2[False], "deferred_last_layer": c2[True],
                             "median_eager": float(np.median(c2[False])), "median_deferred": float(np.median(c2[True]))}
    pathlib.Path(args.out).write_text(json.dumps(out, indent=1))
    print(json.dumps({k: v for k, v in out.items() if k not in ("step_kernels", "read_kernels")}))
    for x in out["read_kernels"]:
        print(x)


def traffic(args):
    """Compulsory DRAM bytes of the two launches of the first adjoint hop under the frontier, from measured |F|.
    Launch 7 (item rows, masked by F): work descriptors of every item row; idx + val of the rows in F; the first
    batch of column ids / values that every group loads before it reads its flag (one 32-byte sector each for the
    rows outside F); the written rows of F; the gathered g_u rows and the g_i seed rows.  Launch 8 (user rows,
    gathers bi' where F is flagged): work descriptors, idx + val of every row, every output row, the rows of F once
    (27 MB: they stay in L2), the g_u seed rows.  Flag arrays (1 byte per row) count once."""
    st = json.loads(pathlib.Path(args.stats).read_text())
    m, d, B = st["mean"], st["emb_dim"], st["batch_users"]
    U, I, E = st["num_users"], st["num_items"], st["nnz"]
    row = 4 * d
    out_items = I - m["front_items"]
    l7 = (16 * (st["item_chunks"] + I - st["item_rows_long"]) + 8 * m["front_edges"] + 64 * out_items
          + row * m["front_items"] + row * B + row * 2 * B + I + U)
    l8 = (16 * (st["user_chunks"] + U - st["user_rows_long"]) + 8 * E + row * U + row * m["front_items"]
          + row * B + I + U)
    path = HERE / "r2_traffic.json"
    data = json.loads(path.read_text())
    c4 = data["C4"]
    src = f"profiles/{pathlib.Path(args.stats).name} (frontier.py traffic)"
    # Launches 5 and 6, the last forward hop restricted to F (item rows) and the batch users (user rows).  Launch 5
    # gathers u_{K-1} along the edges of F's rows: it is charged the captured launch's DRAM bytes per edge net of its
    # streams (descriptors, three d-wide row streams), times the edges of F; plus every descriptor, the first batch of
    # column ids / values of the rows outside F, F's three row streams, and the flag arrays (all-ones gather flags
    # over users, the mask over items).  Launch 6: every descriptor, the first batch of every row outside the batch,
    # the batch rows' idx + val, gathered rows and two row streams (ACC_IN, ACC_OUT), and the flag arrays.
    l5_cap = c4["launches"][4].get("captured_before_frontier", c4["launches"][4])
    desc_i = 16 * (st["item_chunks"] + I - st["item_rows_long"])
    desc_u = 16 * (st["user_chunks"] + U - st["user_rows_long"])
    per_edge = (l5_cap["gb"] * 1e9 - desc_i - 3 * row * I) / E
    l5 = desc_i + 64 * out_items + per_edge * m["front_edges"] + 3 * row * m["front_items"] + U + I
    bu_edges = B * E / U
    l6 = desc_u + 64 * (U - B) + (8 + row) * bu_edges + 2 * row * B + U + I
    for i, gb, kind in ((4, l5, "last forward hop: item rows masked by the batch's item frontier F"),
                        (5, l6, "last forward hop: user rows masked by the batch users"),
                        (6, l7, "item rows masked by the batch's item frontier F"),
                        (7, l8, "user rows gathering only the rows of F")):
        old = c4["launches"][i]
        c4["launches"][i] = dict(kernel=old.get("captured_kernel", old["kernel"]), gb=round(gb / 1e9, 3),
                                 computed=True, what=kind, source=src,
                                 captured_before_frontier=dict(ms=old.get("ms"), gb=old.get("gb"),
                                                               l2_hit_pct=old.get("l2_hit_pct"))
                                 if "captured_before_frontier" not in old else old["captured_before_frontier"])
    for i in range(4, 8):
        c4["launches"][i]["kernel"] = "k_spmm<16, 2, 4, 4, 1, 0, 0>"
    c4["bytes_per_step"] = sum(l["gb"] for l in c4["launches"]) * 1e9
    c4["source"] = ("computed: ncu --set full of bench.py's eager step (profiles/r2_ncu_spmm_c4.txt) for launches "
                    f"1-4 and 9-12, bytes computed from the measured item frontier ({src}) for launches 5-8")
    c4["note"] = ("launches 5 and 6 (the last forward hop) and 7 and 8 (the Gauss-Seidel adjoint at k = 0) are "
                  "computed, not captured: they now touch only the batch's item frontier (and, launch 6, the batch "
                  "users); their capture before that change is kept under captured_before_frontier")
    path.write_text(json.dumps(data, indent=1))
    print(f"launch 5: {l5 / 1e9:.3f} GB, launch 6: {l6 / 1e9:.3f} GB, launch 7: {l7 / 1e9:.3f} GB, "
          f"launch 8: {l8 / 1e9:.3f} GB, step: {c4['bytes_per_step'] / 1e9:.1f} GB")


def main():
    ap = argparse.ArgumentParser()
    sub = ap.add_subparsers(dest="cmd", required=True)
    a = sub.add_parser("stats")
    a.add_argument("out")
    a.add_argument("--batches", type=int, default=16)
    a = sub.add_parser("kernels")
    a.add_argument("out")
    a.add_argument("--tree", default=str(HERE.parent))
    a.add_argument("--steps", type=int, default=2)
    a = sub.add_parser("reads")
    a.add_argument("out")
    a.add_argument("--steps", type=int, default=5)
    a = sub.add_parser("traffic")
    a.add_argument("stats")
    args = ap.parse_args()
    dict(stats=stats, kernels=kernels, reads=reads, traffic=traffic)[args.cmd](args)


if __name__ == "__main__":
    main()
