"""Host-side logic that needs no GPU: the bench contract of the reference arm, the byte model of the roofline,
the synthetic generator, the metric assembly and the shard bookkeeping."""
import json
import pathlib
import subprocess
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]


def test_reference_arm_prints_the_contract_line():
    """bench.py --impl reference runs the reference's own scripts (oracle/_ref, staged by oracle/make_ref.py; the
    oracle port when they did not travel) on the host cores and prints ONE JSON line with the keys the driver reads
    (C1, the reference's own CPU-runnable configuration) -- and its `config` is the one our arm prints."""
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "C1", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    o = json.loads(lines[0])
    assert o["impl"] == "reference" and o["unit"] == "edges/s" and o["higher_is_better"] is True
    assert o["steps"] == 2 and o["warmup"] == 1 and o["n_gpus"] == 1 and o["value"] > 0 and o["ms_per_step"] > 0
    assert o["metric"].startswith("edges/sec") and "workload" in o["config"] and o["config"]["workload"].startswith("C1")
    have_ref = (ROOT / "oracle" / "_ref" / "lightgcn_cu.py").exists()
    assert o["cpu_baseline"]["kind"] == ("reference" if have_ref else "port") and o["cpu_baseline"]["cores"] >= 1
    sys.path.insert(0, str(ROOT))
    import bench
    assert o["config"] == bench.workload_config("C1", 4096, 1)          # same_config: both arms print this object
    if have_ref:
        assert o["cpu_baseline"]["reference_sampler_ms_per_batch"] > 0
    assert o["cpu_baseline"]["value"] == o["value"] == o["e2e"]["value"]
    assert o["e2e"]["h2d_bytes_per_step"] == 0 and o["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_exit_silently():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_algorithmic_bytes_reproduce_the_survey_figures():
    """SURVEY.md 8d, gather model at the nominal edge counts: C1 0.329 GB, C2 5.26 GB, C3 13.47 GB, C4 1358.6 GB,
    C5 3444.5 GB."""
    sys.path.insert(0, str(ROOT))
    import bench
    cases = [((943, 1682, 100_000, 64, 3), 0.329e9), ((31_668, 38_048, 1_560_000, 64, 3), 5.26e9),
             ((52_643, 91_599, 2_980_000, 64, 4), 13.47e9), ((10_000_000, 2_000_000, 200_000_000, 128, 3), 1358.6e9),
             ((50_000_000, 10_000_000, 1_000_000_000, 64, 3), 3444.5e9)]
    for args, want in cases:
        assert abs(bench.gather_model_bytes(*args) - want) / want < 2e-3, (args, bench.gather_model_bytes(*args))


def test_synthetic_generator_is_seeded_and_shaped():
    from credgcn import synth
    a, b = synth.make_graph("C1"), synth.make_graph("C1")
    shp = synth.SHAPES["C1"]
    assert a.num_users == shp["num_users"] == 943 and a.num_items == shp["num_items"] == 1682
    for k in ("train_edges", "val_edges", "test_edges", "cred", "is_fake"):
        np.testing.assert_array_equal(getattr(a, k), getattr(b, k))
    n = a.train_edges.shape[1] + a.val_edges.shape[1] + a.test_edges.shape[1]
    assert abs(n - shp["num_edges"]) <= 0.01 * shp["num_edges"]
    assert abs(a.train_edges.shape[1] / n - 0.8) < 0.01
    keys = a.train_edges[0].astype(np.int64) * a.num_items + a.train_edges[1]
    assert np.unique(keys).size == keys.size                              # unique pairs ...
    d = synth.make_graph("C1", duplicate_edges=300)
    kd = d.train_edges[0].astype(np.int64) * d.num_items + d.train_edges[1]
    assert np.unique(kd).size < kd.size                                   # ... unless duplicates are asked for
    assert a.cred.dtype == np.float32 and a.cred.min() == 0.0 and a.cred.max() == 1.0
    assert abs(a.is_fake.mean() - 0.05) < 0.01
    assert a.cred[a.is_fake].mean() < a.cred[~a.is_fake].mean()           # fake users are the low-credibility ones
    assert not np.array_equal(synth.make_graph("C1", seed=1).train_edges, a.train_edges)
    # the torch generator of the C4 / C5 shapes is seeded in the same way, credibilities included
    import torch
    da, db = (synth.make_graph_device("C4", "cpu", num_users=20_000, num_items=4_000, num_edges=100_000)
              for _ in range(2))
    for k in ("train_edges", "val_edges", "test_edges", "cred", "is_fake"):
        assert torch.equal(getattr(da, k), getattr(db, k)), k


def test_metric_assembly_from_device_sums_equals_host_metrics():
    """evaluate.metrics_result (what the GPU path and the sharded path finish with) fed with sums computed in NumPy
    reproduces metrics_from_ranked."""
    from credgcn import evaluate as ev
    rng = np.random.default_rng(3)
    U, I, n, Ks = 200, 400, 150, [10, 20]
    users = np.sort(rng.choice(U, n, replace=False)).astype(np.int64)
    rows = [np.sort(rng.choice(I, rng.integers(1, 15), replace=False)) for _ in range(U)]
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    idx = np.concatenate(rows).astype(np.int64)
    ranked = np.stack([rng.permutation(I)[:20] for _ in range(n)]).astype(np.int32)
    pop = rng.integers(0, 90, I).astype(np.int64)
    cred = rng.random(U)
    want = ev.metrics_from_ranked(ranked, users, (indptr, idx), I, Ks, "full", pop, int(pop.sum()), cred, 0.2)
    hits = ev._hits_matrix(ranked, users, (indptr, idx), I)
    n_gt = np.diff(indptr)[users]
    disc = 1.0 / np.log2(np.arange(20) + 2.0)
    idcg_tab = np.concatenate([[0.0], np.cumsum(disc)])
    hi, lo = ev.make_cred_groups(users, cred, 0.2)
    in_hi, in_lo = np.isin(users, hi), np.isin(users, lo)
    ks = sorted(Ks)
    sums, counts = np.zeros((len(ks), 7)), np.zeros(len(ks), np.int64)
    for ki, K in enumerate(ks):
        h = hits[:, :K]
        recall = h.sum(1) / np.maximum(n_gt, 1)
        idcg = idcg_tab[np.minimum(n_gt, K)]
        p = pop[ranked[:, :K].astype(np.int64)].astype(np.float64)
        sums[ki] = [(h.sum(1) / K).sum(), recall.sum(), ((h * disc[:K]).sum(1) / idcg).sum(),
                    np.log(p + 1.0).mean(1).sum(), (-np.log2((p + 1.0) / (pop.sum() + I))).mean(1).sum(),
                    recall[in_hi].sum(), recall[in_lo].sum()]
        counts[ki] = np.unique(ranked[:, :K]).size
    got = ev.metrics_result(Ks, ks, sums, counts, n, I, "full", (int(in_hi.sum()), int(in_lo.sum()), cred[users].mean()))
    for K in Ks:
        assert got[K].keys() == want[K].keys()
        for k, v in want[K].items():
            assert got[K][k] == (v if not isinstance(v, float) else __import__("pytest").approx(v, rel=1e-12)), (K, k)


def test_shard_edges_and_partition_cover_the_graph():
    from credgcn import sharded, synth
    sg = synth.make_graph("C1")
    for world in (1, 2, 3, 8):
        deg_u = np.bincount(sg.train_edges[0], minlength=sg.num_users)
        bounds = sharded.partition_users(deg_u, world)
        assert bounds[0] == 0 and bounds[-1] == sg.num_users and len(bounds) == world + 1
        assert all(b1 >= b0 for b0, b1 in zip(bounds, bounds[1:]))
        total = 0
        for r in range(world):
            e = sharded.shard_edges(sg.train_edges, bounds, r)
            total += e.shape[1]
            if e.shape[1]:
                assert e[0].min() >= 0 and e[0].max() < bounds[r + 1] - bounds[r]      # shard-local user ids
            sel = (sg.train_edges[0] >= bounds[r]) & (sg.train_edges[0] < bounds[r + 1])
            np.testing.assert_array_equal(e[1], sg.train_edges[1][sel])
        assert total == sg.train_edges.shape[1]
        nnz = [int(deg_u[bounds[r]:bounds[r + 1]].sum()) for r in range(world)]
        assert max(nnz) - min(nnz) <= 2 * int(deg_u.max())                  # balanced by non-zeros, not by users


def test_exchange_selection_rules():
    """Host-side policy of the multi-GPU exchange (DESIGN.md section 6), without a GPU: which form a table takes."""
    from types import SimpleNamespace
    from credgcn import sharded

    def ex(world, region_mb, mc=1):
        e = sharded.P2PExchange.__new__(sharded.P2PExchange)          # policy methods only: no buffers
        e.world, e.region, e.mc, e.force_push, e.use_nvls = world, region_mb << 20, mc, None, None
        return e

    # small tables: pull at 2 ranks, pushed above -- whatever the environment says (the classes read none; only the
    # benchmark command maps its experiment switches onto force_push / use_nvls / DEFAULT_BACKING)
    import os
    os.environ["CGX_P2P_PUSH"], os.environ["CGX_P2P_NVLS"] = "1", "1"
    try:
        assert not ex(2, 10).push_enabled(33) and ex(4, 10).push_enabled(33)
        assert not ex(2, 2560).nvls_enabled(2560 << 20)
    finally:
        del os.environ["CGX_P2P_PUSH"], os.environ["CGX_P2P_NVLS"]
    # large tables: pushed while the item rows are long (C4 shards: 80 per row), not for short rows (C5 shards: 10)
    assert ex(2, 1024).push_enabled(80) and ex(8, 1024).push_enabled(80) and not ex(8, 2560).push_enabled(10)
    assert ex(8, 2560).push_enabled(None)                              # unknown row length: the old default
    # NVLS form: needs the multicast mapping, 4+ ranks and a large table; forced on / off by use_nvls
    assert ex(8, 2560).nvls_enabled(2560 << 20) and not ex(2, 2560).nvls_enabled(2560 << 20)
    assert not ex(8, 2560, mc=0).nvls_enabled(2560 << 20) and not ex(8, 10).nvls_enabled(10 << 20)
    e = ex(2, 10)
    e.use_nvls = True
    assert e.nvls_enabled(1 << 20)
    e.force_push = True
    assert e.push_enabled(1)
    # whole-step choice: big table + short rows -> the configured exchange, everything else the peer-memory one
    g = SimpleNamespace(by_item=SimpleNamespace(nnz=100_000_000, n_rows=10_000_000))
    assert sharded.ShardedTrainStep.choose_exchange(g, 10_000_000, 64, 8) == sharded.ShardedTrainStep.BIG_SHORT_ROWS_EXCHANGE
    g4 = SimpleNamespace(by_item=SimpleNamespace(nnz=160_000_000, n_rows=2_000_000))
    assert sharded.ShardedTrainStep.choose_exchange(g4, 2_000_000, 128, 8) == "p2p"
    assert sharded.ShardedTrainStep.choose_exchange(g, 10_000_000, 64, 1) == "p2p"
    # compact loss-gradient block: rows | coefficients | row ids | loss, the same size on every rank
    assert sharded.ShardedTrainStep._block_floats(4096, 128) == 2 * 4096 * 130 + 4
