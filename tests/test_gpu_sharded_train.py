"""train_on_arrays_sharded (the user-sharded epoch loop) against the single-GPU train_on_arrays on the same data,
config and seeds, for all six variants and both evaluation protocols: every step's triples, the per-epoch losses,
the validation / test metrics, the final tables, the checkpoint (loaded into the single-GPU class, it reproduces the
test metrics) and -- across ranks -- bit-identical item tables.

Bound on the tables: the sharded run adds the same terms as the single-GPU run, in another order (partial item
tables summed over ranks, the compact loss gradient added in rank order), so each step's tables differ in the last
bits (~1e-7 relative) and Adam carries such differences over a few steps; the bar is the project's 1e-4 relative.

One process with no process group runs the loop over a single shard (every user); 2 / 4 / 8 ranks are spawned as
tests/test_gpu_multi.py does and skipped on boxes with fewer GPUs."""
import contextlib
import io
import os
import pathlib
import re
import sys
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = pathlib.Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
pytestmark = pytest.mark.gpu

TABLE_BOUND = 1e-4
METRIC_TOL = 1e-6
# (variant, eval_mode, batch, device candidates): C1-shaped graph of ~900 users -> tails at 256 and B > n_train at 2048
CASES = [("cu", "sampled", 256, False), ("v2", "sampled", 256, False), ("v2", "full", 256, False),
         ("msg", "full", 256, False), ("me", "sampled", 256, True), ("da", "full", 256, False),
         ("raw", "sampled", 256, False), ("raw", "full", 2048, False), ("v2", "sampled", 2048, True)]


def _graph():
    from credgcn import synth
    return synth.make_graph("C1", num_users=900, num_items=600, num_edges=45_000, duplicate_edges=20)


def _cfg(variant, mode, batch, on_device, dev):
    from credgcn import config
    return config.CFG(variant=variant, eval_mode=mode, batch_size=batch, epochs=2, emb_dim=64, num_layers=3,
                      lambda_fair=0.5 if variant == "cu" else 0.0, sampled_eval_on_device=on_device, device=str(dev))


def _losses(text):
    return [float(x) for x in re.findall(r"Epoch \d+ \| loss=([-0-9.eE]+)", text)]


def _expected_triples(sg, cfg, dev):
    """What the single-GPU loop draws: per step m (1-based over the run), the batch of the epoch's shuffle and the
    TripleSampler triples at offset m."""
    from credgcn import graph, sampler
    from credgcn.train import _GRAPH_VARIANT, _POPMIX
    U, I = sg.num_users, sg.num_items
    gv = "cu" if cfg.variant == "raw" else _GRAPH_VARIANT[cfg.variant]
    cred = np.ones(U, np.float32) if cfg.variant == "raw" else sg.cred
    gr = graph.build_graph(sg.train_edges, U, I, cred, gv, dev)
    smp = (sampler.TripleSampler(gr, cfg.neg_mix_pop, cfg.neg_pop_gamma, cfg.neg_max_tries, cfg.seed)
           if cfg.variant in _POPMIX else sampler.TripleSampler(gr, None, seed=cfg.seed))
    users = np.flatnonzero(np.bincount(sg.train_edges[0], minlength=U) > 0)
    rng = np.random.default_rng(cfg.seed)
    out, m = [], 0
    for _ in range(cfg.epochs):
        rng.shuffle(users)
        for s in range(0, len(users), cfg.batch_size):
            m += 1
            b = torch.as_tensor(users[s:s + cfg.batch_size], device=dev)
            p, n = smp.sample(b, offset=m)
            out.append((b.cpu().numpy(), p.cpu().numpy(), n.cpu().numpy()))
    return out


def _run_case(rank, world, dev, case, group=None):
    """Both loops on one case; returns {name: error} on rank 0 (None elsewhere)."""
    from credgcn import evaluate, train
    from credgcn.sharded import train_on_arrays_sharded
    from credgcn import config
    variant, mode, batch, on_device = case
    sg = _graph()
    cfg = _cfg(variant, mode, batch, on_device, dev)
    keep = config.cfg
    config.cfg = cfg                # the evaluation functions read the module-global cfg, as in the reference
    try:
        return _run_case_cfg(rank, world, dev, case, sg, cfg, group)
    finally:
        config.cfg = keep


def _run_case_cfg(rank, world, dev, case, sg, cfg, group):
    from credgcn import evaluate, train
    from credgcn.sharded import train_on_arrays_sharded
    variant, mode, batch, on_device = case
    rec, steps = [], []

    def on_step(step, epoch, s):
        rec.append(step.last_batch())
        if not steps:
            steps.append(step)

    with tempfile.TemporaryDirectory() as tmp:
        out_dir = tmp if rank == 0 else None
        buf = io.StringIO()
        torch.manual_seed(7)
        with contextlib.redirect_stdout(buf):
            sd, res = train_on_arrays_sharded(sg.train_edges, sg.val_edges, sg.test_edges, sg.num_users, sg.num_items,
                                              sg.cred, out_dir, cfg, group, on_step)
        sh_text = buf.getvalue()
        ei = steps[0].ei.data
        recs = [rec]
        same_items = True
        if world > 1:
            recs = [None] * world
            dist.all_gather_object(recs, rec, group=group)
            parts = [torch.empty_like(ei) for _ in range(world)]
            dist.all_gather(parts, ei.contiguous(), group=group)
            same_items = all(torch.equal(p, parts[0]) for p in parts)
        if rank != 0:
            return None
        errs = {"items_identical_across_ranks": 0.0 if same_items else 1.0}
        # triples of every step: the union over ranks of (global user, slot, pos, neg) == the single-GPU batch
        want = _expected_triples(sg, cfg, dev)
        bad = 0
        for m, (users, pos, neg) in enumerate(want):
            got = np.full((3, len(users)), -1, np.int64)
            for r in range(world):
                gu, sl, p, n = recs[r][m]
                got[:, sl] = np.stack([gu, p, n])
            bad += int((got != np.stack([users, pos, neg])).sum())
        errs["triples_mismatch"] = float(bad)
        # the single-GPU loop
        buf = io.StringIO()
        torch.manual_seed(7)
        with contextlib.redirect_stdout(buf):
            model, want_res = train.train_on_arrays(sg.train_edges, sg.val_edges, sg.test_edges, sg.num_users,
                                                    sg.num_items, sg.cred, None, cfg)
        one_text = buf.getvalue()
        la, lb = _losses(sh_text), _losses(one_text)
        assert len(la) == len(lb) == cfg.epochs, (sh_text, one_text)
        errs["loss"] = max(abs(a - b) / max(abs(b), 1e-12) for a, b in zip(la, lb))

        def metric_err(a, b):
            e = 0.0
            for k in cfg.Ks:
                for key, v in b[k].items():
                    if isinstance(v, float):
                        e = max(e, abs(a[k][key] - v))
                    else:
                        assert a[k][key] == v, (k, key, a[k][key], v)
            return e
        errs["test_metrics_abs"] = metric_err(res, want_res)
        kl = lambda text: [ln for ln in text.splitlines() if ln.startswith("  K=")]   # noqa: E731  (VAL and TEST)
        errs["metric_lines_differ"] = float(kl(sh_text) != kl(one_text))
        wsd = model.state_dict()
        errs["tables"] = max(float((sd[k].to(dev) - wsd[k]).abs().max() / wsd[k].abs().max()) for k in wsd)
        # the checkpoint file loads into the single-GPU class and reproduces the test metrics
        name = "best_model_cred.pt" if variant == "cu" else "best_model.pt"
        model.load_state_dict(torch.load(pathlib.Path(tmp) / "model" / name, map_location=dev))
        tr = model.graph.user_csr_numpy()
        te = train.evaluate_csr(sg.test_edges, sg.num_users, sg.num_items, dev)
        rich = variant == "v2"
        pop, tot = evaluate.compute_item_popularity(sg.train_edges, sg.num_items) if rich else (None, 0)
        if mode == "full" and variant != "cu":
            again = evaluate.evaluate_full_ranking(model, tr, te, sg.num_items, dev, pop, tot, sg.cred if rich else None)
        else:
            again = evaluate.evaluate_sampled(model, tr, te, sg.num_items, dev, pop, tot, sg.cred if rich else None)
        errs["checkpoint_metrics_abs"] = metric_err(again, res)
        return errs


def _check(case, errs):
    print(case, {k: f"{v:.2e}" for k, v in errs.items()})
    assert errs["triples_mismatch"] == 0, (case, errs)
    assert errs["items_identical_across_ranks"] == 0, (case, errs)
    assert errs["loss"] < 1e-5, (case, errs)
    assert errs["test_metrics_abs"] <= METRIC_TOL, (case, errs)
    assert errs["metric_lines_differ"] == 0, (case, errs)
    assert errs["checkpoint_metrics_abs"] <= METRIC_TOL, (case, errs)
    assert errs["tables"] < TABLE_BOUND, (case, errs)


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-{c[1]}-B{c[2]}{'-devcand' if c[3] else ''}")
def test_one_shard_equals_single_gpu(case):
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    errs = _run_case(0, 1, dev, case)
    _check(case, errs)


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        res = {}
        for case in CASES:
            errs = _run_case(rank, world, dev, case)
            if rank == 0:
                res[case] = errs
            dist.barrier()
        if rank == 0:
            out[0] = res
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_loop_equals_single_gpu(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 31600 + (os.getpid() % 2000) + world
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
        res = dict(out)[0]
    for case, errs in res.items():
        _check(case, errs)
