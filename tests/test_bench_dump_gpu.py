"""bench.py --dump-outputs: the last timed step's outputs as float32 .npy files, 64 MB at most, the same bits in two
runs with the same arguments (C2: its user and item tables are longer than bench.DUMP_ROWS, so both are sampled)."""
import json
import pathlib
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]
pytestmark = pytest.mark.gpu


def _bench(out_dir, steps=3):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "C2", "--steps", str(steps),
                          "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_are_reproducible(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    runs = [_bench(tmp_path / "a"), _bench(tmp_path / "b")]
    assert [r["steps"] for r in runs] == [3, 3]
    names = {p.name for p in (tmp_path / "a").iterdir()}
    assert names == {"loss.npy"} | {f"{s}_{w}.npy" for s in ("user", "item") for w in ("emb", "final", "grad")}
    assert names == {p.name for p in (tmp_path / "b").iterdir()}
    total = 0
    for n in sorted(names):
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float32 and np.isfinite(a).all(), n
        assert a.shape == ((1,) if n == "loss.npy" else (8192, 64)), (n, a.shape)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), n
        total += a.nbytes
    assert total <= 64e6
    assert np.abs(np.load(tmp_path / "a" / "user_grad.npy")).max() > 0
    # the dump follows --steps: one timed step fewer gives other tables, final embeddings and gradients (a dump of a
    # fixed step, such as the last warm-up step, would not)
    assert _bench(tmp_path / "c", steps=2)["steps"] == 2
    for n in ("user_emb.npy", "item_emb.npy", "user_final.npy", "item_final.npy", "user_grad.npy", "item_grad.npy"):
        a, c = np.load(tmp_path / "a" / n), np.load(tmp_path / "c" / n)
        assert not np.array_equal(a, c), n
