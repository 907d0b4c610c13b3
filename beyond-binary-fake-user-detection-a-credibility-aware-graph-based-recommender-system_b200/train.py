"""Training entry points with the reference's flow, prints and checkpoint keys.

    load_credibility_vector   lightgcn_cu.py:305-362 / Version-2/lighgcn_cu_pop.py:166-221
    train_lightgcn            lightgcn_cu.py:552-687 / lighgcn_cu_pop.py:758-934

`train_lightgcn()` reads `<cfg.out_dir>/npy/{train,val,test}_edges.npy` and
`<cfg.out_dir>/model/{user2idx,item2idx}.pkl` exactly like the reference (the JSONL ingest that
produces them is out of scope, SURVEY.md section 8f-3); `train_on_arrays` is the same loop for in-memory
edges.  `cfg.variant` selects which script is reproduced:
    "cu"  lightgcn_cu.py                 Jacobi order, uniform negatives, fairness term, sampled eval
    "msg" version_1/lightgcn_cu_message  Gauss-Seidel, uniform negatives
    "me"  version_1/..._method-e         Gauss-Seidel, popularity-mixture negatives
    "da"  version_1/..._Degree-Aware     Gauss-Seidel, uniform negatives, alpha_i damping
    "v2"  Version-2/lighgcn_cu_pop       Gauss-Seidel, popularity-mixture negatives, extra metrics
    "raw" lightgcn.py                    plain LightGCN: one table over users + items, the symmetric normalised
                                         adjacency (build_norm_adj, Jacobi order), uniform negatives, no credibility
                                         CSV, sampled or full eval, `best_model.pt` with the key `emb.weight`
RAW's L2 weight is cfg.reg (1e-4, as in every script).  lightgcn-1.py is the same script with cfg.epochs = 200.
"""
from __future__ import annotations

import csv
import pickle
from pathlib import Path

import numpy as np
import torch

from . import config, evaluate
from .graph import build_graph, build_norm_adj
from .model import CredLightGCN, LightGCN, RawLightGCN, TrainStep
from .sampler import TripleSampler

_GRAPH_VARIANT = {"cu": "cu", "v2": "v2", "msg": "v2", "me": "v2", "da": "da"}
_POPMIX = {"v2", "me"}


def set_seed(seed: int):
    np.random.seed(seed)
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)


def load_credibility_vector(arg, user2idx: dict) -> np.ndarray:
    """cred[num_users] float32 in [0, 1]; users missing from the CSV keep 1.0.  First argument is
    num_users (lightgcn_cu.py signature, path from cfg.cred_csv_path) or the CSV path
    (lighgcn_cu_pop.py signature).  Header `user_id,credibility` wins over `user_idx,credibility`."""
    if isinstance(arg, (int, np.integer)):
        num_users, path = int(arg), Path(config.cfg.cred_csv_path)
    else:
        num_users, path = len(user2idx), Path(arg)
    cred = np.ones((num_users,), dtype=np.float32)
    if not path.exists():
        print(f"[CRED] Cred CSV not found: {path}. Using all-ones credibility.")
        return cred
    with open(path, "r", encoding="utf-8") as f:
        reader = csv.DictReader(f)
        cols = {c.strip() for c in (reader.fieldnames or [])}
        used = skipped = 0
        if {"user_id", "credibility"} <= cols:
            for row in reader:
                uid = row.get("user_id")
                if not uid:
                    continue
                k = user2idx.get(uid)
                if k is None:
                    skipped += 1
                    continue
                try:
                    cred[k] = float(row["credibility"])
                    used += 1
                except Exception:
                    continue
            print(f"[CRED] Loaded by user_id. used={used:,} skipped_not_in_lightgcn={skipped:,}")
        elif {"user_idx", "credibility"} <= cols:
            for row in reader:
                try:
                    k = int(row["user_idx"])
                    if 0 <= k < num_users:
                        cred[k] = float(row["credibility"])
                        used += 1
                except Exception:
                    continue
            print(f"[CRED] Loaded by user_idx. used={used:,}")
        else:
            raise ValueError(f"[CRED] Unsupported cred CSV header: {sorted(cols)}. "
                             "Expected (user_id,credibility) OR (user_idx,credibility).")
    cred = np.clip(cred, 0.0, 1.0).astype(np.float32)
    p10, p50, p90 = np.percentile(cred, [10, 50, 90])
    print(f"[CRED] stats: min={cred.min():.4f} p10={p10:.4f} p50={p50:.4f} p90={p90:.4f} max={cred.max():.4f}")
    return cred


def _print_metrics(tag, res, Ks, rich):
    print(tag)
    for K in Ks:
        r = res[K]
        line = f"  K={K}: P={r['precision']:.4f} R={r['recall']:.4f} NDCG={r['ndcg']:.4f} "
        if rich and "item_coverage" in r:
            line += (f"COV={r['item_coverage']:.4f} LogPop={r['avg_log_popularity']:.4f} "
                     f"SI={r['avg_self_information']:.4f} CredU={r['cred_utility']:.4f} "
                     f"HighR={r['high_cred_recall']:.4f} LowR={r['low_cred_recall']:.4f} ")
        print(line + f"({r['mode']})")


def train_on_arrays(train_edges, val_edges, test_edges, num_users, num_items, cred_np, out_dir=None, cfg=None):
    """The reference's training loop on in-memory edges.  Returns (model, test_results).  cred_np is not read for
    cfg.variant == "raw" (None is fine)."""
    cfg = cfg or config.cfg
    variant = cfg.variant
    device = cfg.device
    print("Using device:", device)

    if variant == "raw":
        norm_adj = build_norm_adj(train_edges, num_users, num_items, device)
        graph = norm_adj.graph
    else:
        graph = build_graph(train_edges, num_users, num_items, cred_np, _GRAPH_VARIANT[variant], device)
    train_csr = graph.user_csr_numpy()
    val_csr = evaluate_csr(val_edges, num_users, num_items, device)
    test_csr = evaluate_csr(test_edges, num_users, num_items, device)

    rich = variant == "v2"
    item_pop, total_train = evaluate.compute_item_popularity(np.asarray(train_edges), num_items) if rich else (None, 0)
    pop_fair = None
    if variant == "cu":
        deg_i = graph.deg_i_float()
        pop_fair = (deg_i / max(float(deg_i.max()), 1.0)).astype(np.float32)      # lightgcn_cu.py:583
        model = CredLightGCN(num_users, num_items, cfg.emb_dim, cfg.num_layers, graph.operator("C"),
                             graph.operator("A")).to(device)
        reg = cfg.lambda_reg
    elif variant == "raw":
        model = RawLightGCN(num_users, num_items, cfg.emb_dim, cfg.num_layers, norm_adj).to(device)
        reg = cfg.reg
    else:
        model = LightGCN(num_users, num_items, cfg.emb_dim, cfg.num_layers, graph.operator("A"),
                         graph.operator("C")).to(device)
        reg = cfg.reg
    step = None

    rng = np.random.default_rng(cfg.seed)
    indptr_tr = train_csr[0]
    train_users = np.where((indptr_tr[1:] - indptr_tr[:-1]) > 0)[0]
    if len(train_users) == 0:
        raise RuntimeError("No train users with interactions. Check your threshold/split.")

    if variant in _POPMIX:
        item_deg = graph.deg_i.cpu().numpy().astype(np.float64)
        p10, p50, p90, p99 = np.percentile(item_deg, [10, 50, 90, 99])
        print(f"[NEG-E] item_deg percentiles: p10={p10:.0f} p50={p50:.0f} p90={p90:.0f} p99={p99:.0f} "
              f"max={item_deg.max():.0f}")
        print(f"[NEG-E] mix_pop={cfg.neg_mix_pop} gamma={cfg.neg_pop_gamma}")
        sampler = TripleSampler(graph, cfg.neg_mix_pop, cfg.neg_pop_gamma, cfg.neg_max_tries, cfg.seed)
    else:
        sampler = TripleSampler(graph, None, seed=cfg.seed)
    step = TrainStep(model, lr=cfg.lr, reg_weight=reg, fair_weight=cfg.lambda_fair if variant == "cu" else 0.0,
                     pop=pop_fair if (variant == "cu" and cfg.lambda_fair) else None, sampler=sampler)
    if len(train_users) >= cfg.batch_size:
        step.capture(cfg.batch_size)          # full batches replay one CUDA graph; the tail batch runs eagerly

    def run_eval(csr):
        if cfg.eval_mode == "full" and variant != "cu":
            return evaluate.evaluate_full_ranking(model, train_csr, csr, num_items, device, item_pop, total_train,
                                                  cred_np if rich else None)
        return evaluate.evaluate_sampled(model, train_csr, csr, num_items, device, item_pop, total_train,
                                         cred_np if rich else None)

    best_val, best_state = -1.0, None
    best_path = None
    if out_dir is not None:
        (Path(out_dir) / "model").mkdir(parents=True, exist_ok=True)
        best_path = Path(out_dir) / "model" / ("best_model_cred.pt" if variant == "cu" else "best_model.pt")

    for epoch in range(1, cfg.epochs + 1):
        model.train()
        rng.shuffle(train_users)
        users_dev = torch.from_numpy(train_users).to(device)
        losses = []
        for start in range(0, len(train_users), cfg.batch_size):
            losses.append(step.step(users_dev[start:start + cfg.batch_size]).clone())
        avg_loss = float(torch.stack(losses).mean().item()) if losses else 0.0
        print(f"Epoch {epoch:03d} | loss={avg_loss:.6f}" if variant == "cu" else f"Epoch {epoch:02d} | loss={avg_loss:.6f}")

        if epoch % cfg.eval_every == 0:
            model.eval()
            val_res = run_eval(val_csr)
            selK = max(cfg.Ks)
            _print_metrics("VAL metrics:", val_res, cfg.Ks, rich)
            if val_res[selK]["recall"] > best_val:
                best_val = val_res[selK]["recall"]
                best_state = {k: v.detach().clone() for k, v in model.state_dict().items()}
                if best_path is not None:
                    torch.save(model.state_dict(), best_path)
                    print(f"  ✅ Saved best model to {best_path} (val Recall@{selK}={best_val:.4f})")

    if best_state is not None:
        model.load_state_dict(best_state)
        model.eval()
    test_res = run_eval(test_csr)
    _print_metrics("\nTEST metrics:", test_res, cfg.Ks, rich)
    return model, test_res


def evaluate_csr(edges, num_users, num_items, device):
    from .graph import user_csr_device
    indptr, idx = user_csr_device(edges, num_users, num_items, device)
    return indptr.cpu().numpy(), idx.cpu().numpy().astype(np.int64)


def train_lightgcn():
    """Reference entry point: everything comes from the module-global cfg and cfg.out_dir."""
    cfg = config.cfg
    out = Path(cfg.out_dir)
    train_edges = np.load(out / "npy" / "train_edges.npy")
    val_edges = np.load(out / "npy" / "val_edges.npy")
    test_edges = np.load(out / "npy" / "test_edges.npy")
    with open(out / "model" / "user2idx.pkl", "rb") as f:
        user2idx = pickle.load(f)
    with open(out / "model" / "item2idx.pkl", "rb") as f:
        item2idx = pickle.load(f)
    num_users, num_items = len(user2idx), len(item2idx)
    print(f"Loaded edges. Users={num_users:,} Items={num_items:,} "
          f"Train={train_edges.shape[1]:,} Val={val_edges.shape[1]:,} Test={test_edges.shape[1]:,}")
    cred_np = None if cfg.variant == "raw" else load_credibility_vector(cfg.cred_csv_path, user2idx)
    _, test_res = train_on_arrays(train_edges, val_edges, test_edges, num_users, num_items, cred_np, out, cfg)
    return test_res


def main():
    """The reference's main() (lightgcn_cu.py:690-703): build the graph files if they are missing, then train.
    Unlike the reference, the raw JSONL is only required when the graph files do not exist yet."""
    from . import ingest
    set_seed(config.cfg.seed)
    if not (Path(config.cfg.out_dir) / "npy" / "train_edges.npy").exists():
        print("Graph files not found. Building graph first...")
        ingest.build_graph_from_jsonl()
    else:
        print("Graph files exist. Skipping construction.")
    train_lightgcn()
