"""bench.py --dump-outputs (-m gpu): the arrays of the last timed step are complete, belong to one step, fit in 64 MB and are
bit-identical from run to run (seeded inputs, atomic-free kernels), so two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARAMS = ["entity_embeddings", "relation_embeddings", "W_entities", "sparse_gat_1.W",
          "sparse_gat_1.attention_0.a", "sparse_gat_1.attention_0.a_2", "sparse_gat_1.attention_1.a",
          "sparse_gat_1.attention_1.a_2", "sparse_gat_1.out_att.a", "sparse_gat_1.out_att.a_2"]


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", str(steps), "--warmup", "1",
           "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    p = subprocess.run(cmd, cwd=out_dir.parent, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    return line, {f[:-len(".npy")]: np.load(out_dir / f) for f in os.listdir(out_dir)}


def test_dump_outputs_complete_and_reproducible(tmp_path):
    line, a = _bench(tmp_path / "a", 3)
    assert line["steps"] == 3
    assert set(a) == {"sample_rows", "loss", "out_entity", "out_relation", "mask"} | {"grad." + k for k in PARAMS}
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 * 2 ** 20
    n, r, d = 10_000, 200, 200                                 # c1; fewer entities than the row sample: every row is kept
    assert np.array_equal(a["sample_rows"], np.arange(n))
    assert a["out_entity"].shape == (n, d) and a["out_relation"].shape == (r, d) and a["mask"].shape == (n,)
    assert a["grad.entity_embeddings"].shape == (n, 50)
    assert np.all(a["mask"] == 1)
    assert np.allclose(np.linalg.norm(a["out_entity"], axis=1), 1.0, atol=1e-5)   # ResidualNorm rows
    # the loss is <out_entity, G_e> + <out_relation, G_r> of the same step (G drawn like bench.SingleGPU does)
    g = torch.Generator().manual_seed(0)
    torch.randn(n, 50, generator=g), torch.randn(r, 50, generator=g)
    g_ent, g_rel = torch.randn(n, d, generator=g).double().numpy(), torch.randn(r, d, generator=g).double().numpy()
    want = (a["out_entity"] * g_ent).sum() + (a["out_relation"] * g_rel).sum()
    assert abs(a["loss"].item() - want) <= 1e-5 * max(1.0, abs(want))

    _, b = _bench(tmp_path / "b", 3)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
