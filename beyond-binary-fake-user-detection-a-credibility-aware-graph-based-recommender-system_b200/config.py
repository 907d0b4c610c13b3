"""CFG: field-for-field mirror of the reference's config dataclasses
(lightgcn_cu.py:30-74 united with Version-2/lighgcn_cu_pop.py:26-74).  As in the reference,
functions that take no explicit knobs read the module-global `cfg`; edit it in place."""
from __future__ import annotations

import pathlib
from dataclasses import dataclass

import torch

_HERE = pathlib.Path.cwd()


@dataclass
class CFG:
    jsonl_path: str = str(_HERE / "dataset" / "Clothing_Shoes_and_Jewelry.jsonl")
    out_dir: str = str(_HERE / "dataset" / "lightgcn_cu_pipeline_parent")
    cred_csv_path: str = str(_HERE / "dataset" / "graph_pyg_parent_asin" / "credibility_scores_minmax_with_user_id.csv")

    user_key: str = "user_id"
    item_key: str = "parent_asin"
    rating_key: str = "rating"
    pos_rating_threshold: float = 4.0

    train_p: float = 0.80
    val_p: float = 0.10
    test_p: float = 0.10

    seed: int = 42
    device: str = "cuda" if torch.cuda.is_available() else "cpu"
    emb_dim: int = 64
    num_layers: int = 3
    lr: float = 1e-3

    lambda_reg: float = 1e-4      # lightgcn_cu.py:58
    reg: float = 1e-4             # lighgcn_cu_pop.py:46 (same role)
    lambda_fair: float = 0.0      # lightgcn_cu.py:61

    epochs: int = 400
    batch_size: int = 4096

    Ks: tuple = (10, 20)
    eval_every: int = 1
    eval_mode: str = "sampled"    # "sampled" or "full"
    sampled_negatives: int = 99

    print_every: int = 1_000_000
    decode_errors: str = "replace"

    # Method E: popularity-aware negatives (lighgcn_cu_pop.py:67-69)
    neg_mix_pop: float = 0.7
    neg_pop_gamma: float = 0.75
    neg_max_tries: int = 50
    # credibility groups (lighgcn_cu_pop.py:74)
    cred_group_pct: float = 0.20

    # which script's behaviour train_lightgcn() follows: "cu" | "v2" | "da" | "msg" | "me" | "raw"
    variant: str = "v2"
    # full-rank eval: "bf16x3" = tcgen05 candidate selection + exact fp32 re-scoring + completeness proof (the
    # SAME ids and score bits as "fp32", 6-7x faster); "fp32" = CUDA-core kernel; "bf16" = one approximate pass
    score_precision: str = "bf16x3"
    # sampled eval: False = candidates from the reference's own PCG64 stream on the host (identical lists);
    # True = candidates drawn on device (same protocol, Philox streams; no per-user Python loop)
    sampled_eval_on_device: bool = False
    metrics_on_device: bool = True   # ranking metrics by cgx_eval_metrics (False: vectorised NumPy on the host)


cfg = CFG()
