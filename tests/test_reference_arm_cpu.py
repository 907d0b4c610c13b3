"""The reference arm of bench.py: oracle/ref_runner.py drives the UNMODIFIED reference scripts staged under oracle/_ref/
(oracle/make_ref.py).  These CPU tests hold one training step and the sampler loop of that arm to what the reference
itself computed -- its loss, gradients and sampled triples stored in tests/golden/*.npz (tests/golden/make_golden.py)
-- so they run on any checkout; where the scripts are staged, the staged scripts are run as well and held to the same
numbers.  Only the byte-identity check of the staged files needs them."""
import hashlib
import json
import pathlib
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "oracle"))
import credgcn_oracle as orc  # noqa: E402
import ref_runner  # noqa: E402
from conftest import load_golden, rel_err  # noqa: E402

CASES = ("tiny", "small")


@pytest.mark.skipif(not ref_runner.available(), reason="oracle/_ref is not staged (run oracle/make_ref.py)")
def test_staged_scripts_match_their_manifest():
    man = json.loads((ref_runner.REF_DIR / "MANIFEST.json").read_text())
    for name in ref_runner.MODULES.values():
        assert hashlib.md5((ref_runner.REF_DIR / name).read_bytes()).hexdigest() == man[name]["md5"], name
    assert not any(p.suffix == ".py" and p.name not in ref_runner.MODULES.values() for p in ref_runner.REF_DIR.iterdir())


def _adam_step(e0_u, e0_i, g_u, g_i, lr):
    """torch.optim.Adam(lr) stepped once on (e0_u, e0_i) with the given gradients, as the reference's loop does
    (CU:587,652 / V2:793,863)."""
    pu, pi = torch.nn.Parameter(torch.tensor(e0_u)), torch.nn.Parameter(torch.tensor(e0_i))
    pu.grad, pi.grad = torch.tensor(g_u), torch.tensor(g_i)
    torch.optim.Adam([pu, pi], lr=lr).step()
    return pu.detach().numpy(), pi.detach().numpy()


@pytest.mark.parametrize("variant,order", [("v2", "gs"), ("cu", "jacobi"), ("da", "gs")])
def test_reference_step_agrees_with_the_oracle(variant, order):
    """One training step -- final embeddings, loss, backward, Adam -- from the reference's initial weights on its
    triples: the oracle port that bench.py times when the scripts are not staged (TorchCpuBaseline) gives the
    reference's loss and the weights Adam makes of the reference's gradients."""
    from credgcn.config import CFG
    cfg = CFG()
    reg = cfg.lambda_reg if variant == "cu" else cfg.reg
    for case in CASES:
        g = load_golden(case, variant)
        U, I, K, d = int(g["num_users"]), int(g["num_items"]), int(g["num_layers"]), int(g["emb_dim"])
        want_loss = float(g["loss"])
        want_u, want_i = _adam_step(g["e0_u"], g["e0_i"], g["grad_u"], g["grad_i"], cfg.lr)
        ops = orc.Operators(g["train_edges"], U, I, g["cred"], variant)
        port = orc.TorchCpuBaseline(ops, g["e0_u"], g["e0_i"], K, order, lr=cfg.lr)
        arms = [("port", port.step(g["users"], g["pos"], g["neg"], reg), port.eu, port.ei)]
        if ref_runner.available():
            arm = ref_runner.ReferenceArm(variant, g["train_edges"], U, I, g["cred"], d, K)
            with torch.no_grad():
                arm.model.user_emb.weight.copy_(torch.tensor(g["e0_u"]))
                arm.model.item_emb.weight.copy_(torch.tensor(g["e0_i"]))
            loss = arm.step(*(torch.tensor(g[k]) for k in ("users", "pos", "neg")))
            arms.append(("reference", loss, arm.model.user_emb.weight, arm.model.item_emb.weight))
        for name, loss, eu, ei in arms:
            eu, ei = eu.detach().numpy(), ei.detach().numpy()
            assert abs(loss - want_loss) <= 1e-5 * abs(want_loss), (case, name, loss, want_loss)
            # Adam's first step moves a parameter by lr * g / (|g| + 1e-8): to lr against the gradient's sign where
            # |g| >> 1e-8, so the updated weights agree to a small fraction of lr
            assert np.abs(eu - want_u).max() < 1e-2 * cfg.lr and np.abs(ei - want_i).max() < 1e-2 * cfg.lr, (case, name)
            du = eu - g["e0_u"]
            moved = np.abs(g["grad_u"]) > 1e-5
            assert moved.any() and np.all(np.sign(du[moved]) == -np.sign(g["grad_u"][moved])), (case, name)
            assert np.allclose(np.abs(du[moved]), cfg.lr, rtol=2e-2), (case, name)
            assert rel_err(eu, want_u) < 1e-5 and rel_err(ei, want_i) < 1e-5, (case, name)


def test_reference_sampler_loop_returns_valid_triples():
    """ReferenceArm's sampler loop (seeded generator, shuffled train users, one batch, per-user draws) returns the
    triples the reference's own loop drew under cfg.seed.  Without the staged scripts the arm runs on the oracle's
    restatement of the reference's sampling functions (held to the same triples by test_oracle_golden)."""
    from credgcn.config import CFG
    for case in CASES:
        for variant in ("v2", "cu", "da"):
            g = load_golden(case, variant)
            U, I, K, d = int(g["num_users"]), int(g["num_items"]), int(g["num_layers"]), int(g["emb_dim"])
            if ref_runner.available():
                arm = ref_runner.ReferenceArm(variant, g["train_edges"], U, I, g["cred"], d, K)
            else:
                arm = ref_runner.ReferenceArm.__new__(ref_runner.ReferenceArm)
                arm.variant, arm.device, arm.num_users, arm.num_items = variant, "cpu", U, I
                arm.ref = SimpleNamespace(cfg=CFG(), sample_pos_item=orc.draw_positive,
                                          sample_neg_item=orc.draw_negative_uniform,
                                          sample_neg_item_popmix=orc.draw_negative_popmix)
                arm.train_csr = orc.edges_to_user_csr(g["train_edges"], U)
                arm.pop_prob = None
                if variant == "v2":
                    arm.pop_prob = orc.popularity_law(orc.degrees(g["train_edges"], U, I)[1], arm.ref.cfg.neg_pop_gamma)
                indptr = arm.train_csr[0]
                arm.train_users = np.where((indptr[1:] - indptr[:-1]) > 0)[0]
                arm.rng = np.random.default_rng(arm.ref.cfg.seed)
            batch = arm.batches(len(g["samp_users"]))[0]
            u, p, n = (t.numpy() for t in arm.sample_batch(batch))
            np.testing.assert_array_equal(u, g["samp_users"])
            np.testing.assert_array_equal(p, g["samp_pos"])
            np.testing.assert_array_equal(n, g["samp_neg"])
            indptr, indices = arm.train_csr
            assert len(u) == len(batch) and set(u) <= set(arm.train_users)
            for uu, pp, nn in zip(u, p, n):
                row = indices[indptr[uu]:indptr[uu + 1]]
                assert pp in row and nn not in row and 0 <= nn < I
