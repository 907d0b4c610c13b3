#!/usr/bin/env python
"""bench.py -- edges/sec of the K-layer credibility-weighted LightGCN training step on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C4] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one full training step of the reference loop (lightgcn_cu.py:608-654 /
Version-2/lighgcn_cu_pop.py:826-866) on one batch of 4096 users: on-device triple sampling, K-layer forward, fused
BPR+L2 loss, adjoint propagation, dense Adam.  metric = train edges / step time.

Default workload: C4 (10M users x 2M items x 200M edges, d = 128, K = 3) -- the largest BASELINE configuration that
fits one GPU and the HBM-bound one; with --gpus N every rank owns one C4-shaped user shard (weak scaling).  Without
--workload the N = 1 line also carries a `c2` object: the same measurement on BASELINE configs[1] (L2-resident).
Prints ONE JSON line (rank 0).  DESIGN.md section 5 explains every key.
"""
import argparse
import json
import os
import pathlib
import subprocess
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "edges/sec (3-layer cred-weighted LightGCN fwd+bwd)"
DEFAULT_WORKLOAD = "C4"
REG = 1e-4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=["C1", "C2", "C3", "C4", "C5"])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the C2 leg of the default run")
    ap.add_argument("--cpu-steps", type=int, default=3)
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--hot-mb", type=float, default=None,
                    help="MiB of hot (high-degree) rows the SpMM keeps L2-resident (default: CredGraph.HOT_BYTES)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (one GPU only)")
    return ap.parse_args()


def ceil_div(a, b):
    return (a + b - 1) // b


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def gather_model_bytes(U, I, nnz, d, K):
    """SURVEY.md section 8d, fwd+bwd: r = 4d bytes per row; one SpMM moves nnz (4 + 4 + r) + n_dst r; a layer adds the
    running-sum epilogue 2 (U + I) r.  Every gathered row counts as a fresh read (an upper bound once L2 helps)."""
    r = 4 * d
    return 2 * (K * (2 * nnz * (8 + r) + (U + I) * r) + 2 * K * (U + I) * r)


def compulsory_bytes(U, I, nnz, d, K):
    """SURVEY.md section 8d (i): every source row read once per product instead of once per edge."""
    r = 4 * d
    return 2 * (K * (2 * nnz * 8 + 2 * (U + I) * r) + 2 * K * (U + I) * r)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md recipe): one background `nvidia-smi -lms 20`;
    `with` marks a timed region and `summary()` reports the samples whose timestamps fall inside one."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.windows = []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None

    def __enter__(self):
        self._t0 = time.time()
        return self

    def __exit__(self, *a):
        self.windows.append((self._t0, time.time()))

    def summary(self):
        rows = []
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                out = ""
            import datetime
            for line in out.splitlines():
                f = [x.strip() for x in line.split(",")]
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(f[1]), float(f[2]), [v.lower().startswith("active") for v in f[4:8]]))
                except Exception:
                    continue
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        first = self.windows[:1]          # the headline workload's timed region
        inside = [r for r in rows if any(t0 - 0.02 <= r[0] <= t1 + 0.02 for t0, t1 in first)]
        if not inside and rows and first:                 # region shorter than the sampling period: nearest samples
            mid = 0.5 * (first[0][0] + first[0][1])
            inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
        reasons = sorted({n for r in inside for n, v in zip(names, r[3]) if v})
        return {"sm_mhz": float(np.median([r[1] for r in inside])) if inside else None,
                "sm_max_mhz": max([r[2] for r in inside]) if inside else None,
                "reasons": reasons, "samples": len(inside), "samples_total": len(rows)}


def workload_config(name, batch, gpus=1):
    """The `config` object: a function of the workload only, so that both arms print the same one."""
    from credgcn import synth
    shp = synth.SHAPES[name]
    U, I, E = shp["num_users"], shp["num_items"], shp["num_edges"]
    table_mb = (U + I) * shp["emb_dim"] * 4 / 1e6
    per = " per GPU (one user shard each, items replicated)" if gpus > 1 and name != "C5" else ""
    return {
        "workload": f"{name}: {U:,} users x {I:,} items x {E:,} edges{per}, 80 % of them train edges "
                    f"({shp['variant']} operator, {shp['order']} order), synthetic power law + 5 % fake-user clusters",
        "emb_dim": shp["emb_dim"], "num_layers": shp["num_layers"], "batch_users": batch * gpus,
        "step": "sample+fwd+loss+bwd+adam", "fake_user_frac": 0.05,
        "parallelism": "single GPU" if gpus == 1 else f"user-shard x{gpus}",
        "l2": (f"embedding tables {table_mb:,.0f} MB >> 126 MB L2" if table_mb > 500 else
               f"embedding tables {table_mb:,.0f} MB fit L2") + "; 256 MiB L2 flush between timed steps",
    }


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (oracle/_ref, staged by oracle/make_ref.py), else the port
# ------------------------------------------------------------------------------------------------------------------
def reference_sample(name, fraction):
    """A bounded sample of workload `name` for the CPU arm: the same generator law at `fraction` of the users, items
    AND edges, so that edges per table row -- what sets the reference's cost per edge -- stay those of the
    workload; fraction = 1 is the workload itself."""
    from credgcn import synth
    shp = synth.SHAPES[name]
    if fraction >= 1.0:
        return synth.make_graph(name), shp
    U = max(int(shp["num_users"] * fraction), 1024)
    I = max(int(shp["num_items"] * fraction), 1024)
    E = max(int(shp["num_edges"] * fraction), 16384)
    return synth.make_graph(name, num_users=U, num_items=I, num_edges=E), shp


def _cheap_triples(sg, users, rng, as_numpy=False):
    """pos from the user's row, neg uniform (rejection skipped: it does not change the arithmetic being timed)."""
    if not hasattr(sg, "_csr"):
        u_all, i_all = sg.train_edges[0].astype(np.int64), sg.train_edges[1].astype(np.int64)
        order = np.argsort(u_all, kind="stable")
        indptr = np.zeros(sg.num_users + 1, np.int64)
        np.cumsum(np.bincount(u_all, minlength=sg.num_users), out=indptr[1:])
        sg._csr = (indptr, i_all[order])
    indptr, items = sg._csr
    users = np.asarray(users, dtype=np.int64)
    deg = indptr[users + 1] - indptr[users]
    pos = items[np.minimum(indptr[users] + (rng.random(users.size) * deg).astype(np.int64), items.size - 1)]
    neg = rng.integers(0, sg.num_items, size=users.size)
    if as_numpy:
        return users, pos, neg
    return torch.tensor(users), torch.tensor(pos), torch.tensor(neg)


class CpuArm:
    """One CPU training step of the reference: `kind` = "reference" (the unmodified scripts under oracle/_ref) or
    "port" (oracle.TorchCpuBaseline, when the scripts did not travel)."""

    def __init__(self, sg, shp, batch):
        sys.path.insert(0, str(ROOT / "oracle"))
        import ref_runner
        torch.set_num_threads(os.cpu_count() or 1)
        self.E = int(sg.train_edges.shape[1])
        rng = np.random.default_rng(11)
        if ref_runner.available():
            self.kind = "reference"
            self.arm = ref_runner.ReferenceArm(shp["variant"], sg.train_edges, sg.num_users, sg.num_items, sg.cred,
                                               shp["emb_dim"], shp["num_layers"])
            users = self.arm.batches(batch)
            t0 = time.perf_counter()
            first = self.arm.sample_batch(users[0])          # the reference's per-user Python sampler, one batch
            self.sampler_ms = 1e3 * (time.perf_counter() - t0)
            # the other batches take cheap triples: the sampler is reported on its own, not inside the timed steps
            self.triples = [first] + [_cheap_triples(sg, b, rng) for b in users[1:8] if len(b) == len(users[0])]
            self.build_ms = {"build_mats": 1e3 * self.arm.build_mats_s, "edges_to_user_csr": 1e3 * self.arm.build_csr_s}
        else:
            import credgcn_oracle as orc
            self.kind = "port"
            ops = orc.Operators(sg.train_edges, sg.num_users, sg.num_items, sg.cred, shp["variant"])
            torch.manual_seed(42)
            e0_u = torch.nn.init.xavier_uniform_(torch.empty(sg.num_users, shp["emb_dim"])).numpy()
            e0_i = torch.nn.init.xavier_uniform_(torch.empty(sg.num_items, shp["emb_dim"])).numpy()
            self.arm = orc.TorchCpuBaseline(ops, e0_u, e0_i, shp["num_layers"], shp["order"])
            train_users = np.flatnonzero(np.bincount(sg.train_edges[0], minlength=sg.num_users) > 0)
            rng.shuffle(train_users)
            self.triples = [_cheap_triples(sg, train_users[s:s + batch], rng, as_numpy=True)
                            for s in range(0, min(len(train_users), 8 * batch), batch)]
            self.sampler_ms, self.build_ms = None, None

    def step(self, s):
        t = self.triples[s % len(self.triples)]
        return self.arm.step(*t) if self.kind == "reference" else self.arm.step(*t, REG)

    def time_steps(self, steps, warmup):
        for s in range(warmup):
            self.step(s)
        ts = []
        for s in range(steps):
            t0 = time.perf_counter()
            self.step(warmup + s)            # ends with loss.item(): complete when it returns
            ts.append(time.perf_counter() - t0)
        return 1e3 * float(np.mean(ts))


def cpu_baseline_object(name, batch, steps, warmup, budget_s):
    """Time the CPU arm on a bounded sample of `name`: the largest power-of-two user fraction whose
    (warmup + steps) steps fit `budget_s` (probed with one step on a small fraction)."""
    from credgcn import synth
    shp = synth.SHAPES[name]
    frac = 1.0 if shp["num_edges"] <= 4_000_000 else 1.0 / 64
    sg, _ = reference_sample(name, frac)
    arm = CpuArm(sg, shp, batch)
    if frac < 1.0:
        probe_ms = arm.time_steps(1, 1)
        want = frac
        while want < 1.0 and (steps + warmup) * probe_ms * (2 * want / frac) / 1e3 < budget_s:
            want *= 2
        if want > frac * 1.5:
            frac = min(want, 1.0)
            sg, _ = reference_sample(name, frac)
            arm = CpuArm(sg, shp, batch)
    ms = arm.time_steps(steps, warmup)
    what = ("the reference's own scripts (oracle/_ref: build_*_mats, LightGCN / CredLightGCN, bpr_loss, "
            "torch.optim.Adam)" if arm.kind == "reference" else
            "oracle port of the reference's COO torch.sparse.mm + autograd + Adam path")
    sample = (f"{steps} training steps (final embeddings + loss + backward + Adam; the reference's per-user Python "
              f"sampler is timed separately) of {what} on "
              + (f"all of {name}" if frac >= 1.0 else f"a {frac:.4g}-scale sample of {name} (users, items and edges)")
              + f": {sg.num_users:,} users x {sg.num_items:,} items x {arm.E:,} train edges, "
              f"d={shp['emb_dim']}, K={shp['num_layers']}")
    obj = {"value": arm.E / (ms / 1e3), "unit": "edges/s", "cores": torch.get_num_threads(), "kind": arm.kind,
           "sample": sample, "ms_per_step": ms, "sample_fraction": frac}
    if arm.sampler_ms is not None:
        obj["reference_sampler_ms_per_batch"] = arm.sampler_ms
        obj["reference_graph_build_ms"] = arm.build_ms
    return obj


def run_reference(args):
    """--impl reference: the reference's CPU implementation on the same config / metric / unit (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    name = args.workload or DEFAULT_WORKLOAD
    obj = cpu_baseline_object(name, args.batch, args.steps, args.warmup, budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": obj["value"], "unit": "edges/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": obj["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, args.batch, args.gpus),
        "cpu_baseline": obj,
        "e2e": {"value": obj["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# our arm, one GPU
# ------------------------------------------------------------------------------------------------------------------
def traffic_per_step(name):
    """DRAM bytes per training step of the SpMM launches, from the committed ncu --set full capture of this round
    (profiles/r2_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum summed over the 4K launches of a step)."""
    p = ROOT / "profiles" / "r2_traffic.json"
    if not p.exists():
        return None, None
    j = json.loads(p.read_text()).get(name)
    if not j:
        return None, None
    return float(j["bytes_per_step"]), j.get("source")


DUMP_ROWS = 8192        # rows kept of each table: 6 tables x 8192 rows x d = 128 x 4 B = 25 MB per workload at most


def dump_last_step(out_dir, prefix, loss, step):
    """--dump-outputs: what the last timed TrainStep.step() computed, as float32 .npy files that two builds can be
    compared by -- the loss it returned, the embedding tables Adam updated in place, and the final embeddings and
    gradients it leaves on the step and the parameters.  Tables longer than DUMP_ROWS rows are cut to the same seeded
    sample of rows in every run."""
    out = pathlib.Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / f"{prefix}loss.npy", loss.detach().float().reshape(1).cpu().numpy())
    m = step.model
    for side, emb, final in (("user", m.user_emb.weight, step.f_u), ("item", m.item_emb.weight, step.f_i)):
        n = emb.shape[0]
        rows = None
        if n > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
            rows = torch.from_numpy(rows).to(emb.device)
        for what, t in (("emb", emb), ("final", final), ("grad", emb.grad)):
            t = t.detach() if rows is None else t.detach().index_select(0, rows)
            np.save(out / f"{prefix}{side}_{what}.npy", t.float().cpu().numpy())


def run_single(args, name, dev, steps, warmup, clocks, with_cpu, with_extras, dump_prefix=None):
    from credgcn import _lib, graph, model, sampler, synth
    shp = synth.SHAPES[name]
    t0 = time.time()
    big = name in ("C4", "C5")
    sg = synth.make_graph_device(name, dev) if big else synth.make_graph(name)
    t_gen = time.time() - t0
    U, I, E = sg.num_users, sg.num_items, int(sg.train_edges.shape[1])
    d, K = shp["emb_dim"], shp["num_layers"]

    # ---- graph build (device-resident edges; for host-generated workloads also end to end from host edges) ----
    t_build_e2e = None
    if not big:
        graph.build_graph(sg.train_edges[:, :1000], U, I, sg.cred, shp["variant"], dev)   # module load / first launch
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gr = graph.build_graph(sg.train_edges, U, I, sg.cred, shp["variant"], dev)
        torch.cuda.synchronize()
        t_build_e2e = time.perf_counter() - t0
        del gr
    edges_dev = sg.train_edges if big else torch.from_numpy(sg.train_edges).to(dev)
    cred_dev = sg.cred if big else torch.from_numpy(sg.cred).to(dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gr = graph.build_graph(edges_dev, U, I, cred_dev, shp["variant"], dev)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    del edges_dev
    if big:
        sg.train_edges = sg.val_edges = sg.test_edges = None      # free the generator's copies
        torch.cuda.empty_cache()

    torch.manual_seed(42)
    Net = model.CredLightGCN if shp["variant"] == "cu" else model.LightGCN
    ops = (gr.operator("C"), gr.operator("A")) if shp["variant"] == "cu" else (gr.operator("A"), gr.operator("C"))
    net = Net(U, I, d, K, *ops).to(dev)
    samp = sampler.TripleSampler(gr, None if shp["variant"] == "cu" else 0.7, 0.75, 50, seed=42)
    step = model.TrainStep(net, lr=1e-3, reg_weight=REG, sampler=samp)

    train_users = torch.nonzero(gr.deg_u > 0).reshape(-1).cpu().numpy()
    np.random.default_rng(42).shuffle(train_users)
    steps_per_epoch = ceil_div(len(train_users), args.batch)
    n_batches = min(max(len(train_users) // args.batch, 1), 64)
    host_batches = [train_users[s * args.batch:(s + 1) * args.batch] for s in range(n_batches)]
    dev_batches = [torch.from_numpy(b).to(dev) for b in host_batches]
    pinned = [torch.from_numpy(b).pin_memory() for b in host_batches]
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    B = int(host_batches[0].size)

    # ---- ONE code path for `value` and `e2e`: the public TrainStep.step() replaying the captured CUDA graph ----
    step.capture(B, preserve_state=name != "C5")
    for s in range(max(warmup, 3)):
        step.step(dev_batches[s % n_batches])
    torch.cuda.synchronize()

    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    with clocks:
        torch.cuda.synchronize()
        # (a) `value`: inputs already resident in HBM, CUDA events around the replay, L2 flushed between steps
        for s in range(steps):
            if not args.no_flush:
                flush_buf.fill_(s & 0xff)
            starts[s].record()
            loss_dev = step.step(dev_batches[s % n_batches])
            ends[s].record()
        torch.cuda.synchronize()
        step_ms = [a.elapsed_time(b) for a, b in zip(starts, ends)]
        if dump_prefix is not None:
            dump_last_step(args.dump_outputs, dump_prefix, loss_dev, step)
        # (b) `e2e`: the same call with PINNED HOST batches -- H2D of the batch, replay, D2H of the loss, every step
        for s in range(2):
            float(step.step(pinned[s % n_batches]).item())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss_host = 0.0
        for s in range(steps):
            loss_host = float(step.step(pinned[s % n_batches]).item())
        torch.cuda.synchronize()
        e2e_ms = 1e3 * (time.perf_counter() - t0) / steps
        # (c) phase split + launch count: the same kernels launched eagerly with events between the phases
        #     (events cannot sit inside a replayed graph); `ncu --profile-from-start off` sees exactly these steps
        n_phase = min(steps, 5)
        step.phase_events = []
        step.step(dev_batches[0])                 # first eager launch after the capture: one-time lazy work
        step.phase_events = []
        eager_ends = [torch.cuda.Event(enable_timing=True) for _ in range(n_phase)]
        launches0 = _lib.lib().cgx_launch_count()
        torch.cuda.profiler.start()
        for s in range(n_phase):
            if not args.no_flush:
                flush_buf.fill_(s & 0xff)
            step.step(dev_batches[s % n_batches])
            eager_ends[s].record()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        launches_per_step = (_lib.lib().cgx_launch_count() - launches0) // n_phase
        phases = step.phase_events
        step.phase_events = None
        # (d) epoch: a real one when it is short, else extrapolated from the timed steps
        epoch_ms, epoch_kind = None, None
        if steps_per_epoch <= 256:
            ep_users = train_users.copy()
            np.random.default_rng(7).shuffle(ep_users)
            ep_batches = [torch.from_numpy(ep_users[s:s + args.batch]).to(dev)
                          for s in range(0, len(ep_users), args.batch)]
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for ub in ep_batches:                 # full batches replay the graph, the ragged tail launches eagerly
                step.step(ub)
            b.record()
            torch.cuda.synchronize()
            epoch_ms, epoch_kind = a.elapsed_time(b), f"timed: {len(ep_batches)} steps, every train user once"
    ms = float(np.mean(step_ms))
    if epoch_ms is None:
        epoch_ms, epoch_kind = ms * steps_per_epoch, f"extrapolated: {steps_per_epoch} steps x the timed mean step"

    fwd_ms = float(np.median([m[0].elapsed_time(m[1]) for m in phases]))
    loss_ms = float(np.median([m[1].elapsed_time(m[2]) for m in phases]))
    bwd_ms = float(np.median([m[2].elapsed_time(m[3]) for m in phases]))
    rest_ms = float(np.median([m[3].elapsed_time(e) for m, e in zip(phases, eager_ends)]))   # L2 term + Adam
    prop_ms = fwd_ms + bwd_ms
    hbm_peak, peak_src = peaks()
    n_spmm = 4 * K
    gather = gather_model_bytes(U, I, gr.nnz, d, K)
    comp = compulsory_bytes(U, I, gr.nnz, d, K)
    table_mb = (U + I) * d * 4 / 1e6
    traffic, traffic_src = traffic_per_step(name)
    hbm_bound = table_mb > 500
    # Tables beyond L2: the bytes that bound the kernel are the ones that cross the DRAM pins -- SURVEY 8d (ii), ncu
    # dram__bytes of the committed capture of these very launches; the gather model (every neighbour row a fresh
    # read) over-counts the hot rows L2 serves.  Tables inside L2: nothing is HBM-bound; lead with compulsory bytes.
    if hbm_bound and traffic:
        alg, alg_kind = traffic, "DRAM bytes of the 4K SpMM launches of a step (ncu capture, profiles/r2_traffic.json)"
    elif hbm_bound:
        alg, alg_kind = gather, "gather model (SURVEY 8d): no ncu capture committed for this workload"
    else:
        alg, alg_kind = comp, "compulsory bytes (SURVEY 8d i): tables are L2-resident, the kernel is latency-bound"
    achieved = alg / (prop_ms / 1e3) / 1e9
    roof = {
        "bound": "hbm", "kernel": "k_spmm (+ k_spmm_finish for rows > 16384 nnz), 4K launches per step",
        "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "peak_source": peak_src,
        "bytes": alg_kind, "traffic": (traffic / n_spmm) if traffic else None, "traffic_source": traffic_src,
        "avg_launch_ms": prop_ms / n_spmm, "launches_per_step": n_spmm,
        "frac_dram_bytes": (traffic / (prop_ms / 1e3) / 1e9 / hbm_peak) if traffic else None,
        "frac_gather_model": gather / (prop_ms / 1e3) / 1e9 / hbm_peak,
        "frac_compulsory": comp / (prop_ms / 1e3) / 1e9 / hbm_peak,
        "gather_model_bytes_per_step": gather, "compulsory_bytes_per_step": comp,
        "sparse_first_adjoint": _lib.get_option("SPARSE_FIRST_ADJOINT") != 0,
        "hot_rows": {"bytes": graph.CredGraph.HOT_BYTES, "items": gr.by_user.n_hot, "users": gr.by_item.n_hot},
    }
    line = {
        "metric": METRIC, "value": E / (ms / 1e3), "unit": "edges/s", "n_gpus": 1, "steps": steps,
        "warmup": max(warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, args.batch),
        "train_edges": E, "nnz": gr.nnz,
        "e2e": {"value": E / (e2e_ms / 1e3), "unit": "edges/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(host_batches[0].nbytes), "d2h_bytes_per_step": 4,
                "api": "TrainStep.step(pinned_host_users) [CUDA-graph replay] + loss.item()"},
        "value_api": "TrainStep.step(device_users) [the same CUDA-graph replay], CUDA events",
        "gpu_launches": int(launches_per_step * steps),
        "gpu_launches_note": f"{launches_per_step} kernels of libcredgcn.so per step (counted on eager launches of the "
                             "same step; a graph replay launches the same kernels)",
        "roofline": roof,
        "phases_ms": {"propagate_fwd": fwd_ms, "bpr_loss+grad_scatter": loss_ms, "propagate_bwd": bwd_ms,
                      "l2_term+adam": rest_ms,
                      "source": f"medians over {n_phase} eager launches of the step inside the timed region (the "
                                "sampler and the scatter plan run before / beside the forward)"},
        "fwd_bwd_edges_per_s": E / (prop_ms / 1e3),
        "graph_build_ms": {"device_resident": 1e3 * t_build,
                           "from_host_edges": None if t_build_e2e is None else 1e3 * t_build_e2e,
                           "edges_per_s": E / t_build, "synthetic_generation_s": t_gen},
        "steps_per_epoch": steps_per_epoch, "epoch_ms": epoch_ms, "epoch_ms_kind": epoch_kind,
        "loss": loss_host,
    }

    if with_extras and E <= 20_000_000:
        line.update(extras_small(args, sg, shp, gr, net, dev))
    del step, net, gr, samp, dev_batches, flush_buf
    torch.cuda.empty_cache()
    if with_cpu:
        line["cpu_baseline"] = cpu_baseline_object(name, args.batch, args.cpu_steps, 1, budget_s=25.0)
    return line


def extras_small(args, sg, shp, gr, net, dev):
    """C1-C3 only: the full-rank evaluation leg (north_star 4) and the reference's own GPU path (stock torch)."""
    from credgcn import evaluate, model
    out = {}
    U, I, d, K = sg.num_users, sg.num_items, shp["emb_dim"], shp["num_layers"]
    with torch.no_grad():
        f_u, f_i = model.propagate_forward(gr, net.user_emb.weight.detach(), net.item_emb.weight.detach(), K,
                                           shp["order"])
    all_users = torch.arange(U, device=dev)
    csr = (gr.samp_indptr, gr.samp_idx)
    ev = {"users": U, "items": I, "k": 20, "flops": 2.0 * U * I * d}
    ids_ref = None
    for prec in ("fp32", "bf16x3"):
        for _ in range(2):
            ids, _ = evaluate.topk_device(f_u, f_i, all_users, csr, 20, prec)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ids, _ = evaluate.topk_device(f_u, f_i, all_users, csr, 20, prec)
        b.record()
        torch.cuda.synchronize()
        t = a.elapsed_time(b)
        ev[prec] = {"ms": t, "useful_tflops": ev["flops"] / t / 1e9, "users_per_s": U / (t / 1e3)}
        if ids_ref is None:
            ids_ref = ids
        else:
            ev[prec]["ids_equal_fp32"] = bool(torch.equal(ids, ids_ref))
            ev[prec]["kernel"] = "tcgen05 selection + exact fp32 re-scoring + completeness proof"
    out["eval_full_rank"] = ev
    # the reference's own GPU path: its script-level code on stock ATen / cuSPARSE kernels (oracle port, device=cuda)
    sys.path.insert(0, str(ROOT / "oracle"))
    import credgcn_oracle as orc
    torch.cuda.empty_cache()
    ops = orc.Operators(sg.train_edges, U, I, sg.cred, shp["variant"])
    e0_u = net.user_emb.weight.detach().cpu().numpy().copy()
    e0_i = net.item_emb.weight.detach().cpu().numpy().copy()
    base = orc.TorchCpuBaseline(ops, e0_u, e0_i, K, shp["order"], device=str(dev))
    rng = np.random.default_rng(11)
    tu = np.flatnonzero(np.bincount(sg.train_edges[0], minlength=U) > 0)[:args.batch]
    tri = _cheap_triples(sg, tu, rng, as_numpy=True)
    ts = []
    for s in range(21):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        base.step(*tri, REG)
        ts.append(time.perf_counter() - t0)
    gms = 1e3 * float(np.mean(ts[1:]))
    E = int(sg.train_edges.shape[1])
    out["torch_gpu_baseline"] = {"value": E / (gms / 1e3), "unit": "edges/s", "ms_per_step": gms, "kind": "port",
                                 "sample": "20 training steps, stock torch CUDA sparse COO path (ATen/cuSPARSE) on "
                                           "this GPU, oracle port of the reference's script-level code"}
    fu_h, fi_h = f_u.cpu().numpy(), f_i.cpu().numpy()
    tr = (gr.samp_indptr.cpu().numpy(), gr.samp_idx.cpu().numpy().astype(np.int64))
    t0 = time.perf_counter()
    orc.full_rank_topk(fu_h, fi_h, np.arange(256), tr, 20)
    out["eval_full_rank"]["cpu_port_ms_per_user"] = 1e3 * (time.perf_counter() - t0) / 256
    return out


def main():
    args = parse()
    if args.dump_outputs is not None and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        raise SystemExit("--dump-outputs writes the training step of --impl ours on one GPU")
    if args.dump_outputs is not None and args.steps < 1:
        raise SystemExit("--dump-outputs writes the last timed step: it needs --steps 1 or more")
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from credgcn import graph
    if args.hot_mb is not None:
        graph.CredGraph.HOT_BYTES = int(args.hot_mb * (1 << 20))
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        from credgcn import sharded
        return sharded.bench_main(args, rank, world, dev)

    name = args.workload or DEFAULT_WORKLOAD
    if name == "C5":
        print("[bench] C5 on ONE GPU: 50M x 10M x 1B edges needs ~165 GB of the 180 GB", file=sys.stderr)
    clocks = ClockSampler(local)
    dump = args.dump_outputs is not None
    line = run_single(args, name, dev, args.steps, args.warmup, clocks, with_cpu=not args.no_cpu_baseline,
                      with_extras=True, dump_prefix="" if dump else None)
    if args.workload is None and not args.no_extra:
        # the L2-resident BASELINE config (configs[1]) measured the same way, as an extra object
        c2 = run_single(args, "C2", dev, args.steps, args.warmup, clocks, with_cpu=False, with_extras=True,
                        dump_prefix="c2_" if dump else None)
        line["c2"] = {k: c2[k] for k in ("value", "unit", "ms_per_step", "config", "e2e", "roofline", "phases_ms",
                                         "graph_build_ms", "steps_per_epoch", "epoch_ms", "epoch_ms_kind",
                                         "eval_full_rank", "torch_gpu_baseline", "train_edges") if k in c2}
    line["clocks"] = clocks.summary()
    print(json.dumps(line))


if __name__ == "__main__":
    main()
