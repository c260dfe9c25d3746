"""bench.py --dump-outputs on the GPU: the last timed step's loss terms and parameters land as float32 .npy files, and two runs
with the same arguments (same seeded inputs, weights and noise) give the same arrays up to rounding.  cfg4 is the workload
that splits the batch across CTAs, where the weight-gradient sums are reduce-added in no fixed order."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LR = 1e-3                # the Engine's default learning rate, which bench.py uses

pytestmark = pytest.mark.gpu


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg4", "--steps", str(steps), "--warmup", "3",
                        "--no-cpu-baseline", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_of_the_timed_step(tmp_path):
    import gmvae_b200
    from bench import WORKLOADS
    line, a = _bench(tmp_path / "a", 3)
    assert line["steps"] == 3
    w = WORKLOADS["cfg4"]
    eng = gmvae_b200.Engine(model=w["model"], latent_size=w["latent_size"], hidden_sizes=w["hidden_sizes"],
                            mixture_components=w["mixture_components"], max_batch=128, seed=1234)
    init = {"param." + n.replace("/", "."): v.cpu().numpy() for n, v in eng.parameters().items()}
    eng.close()
    assert {k: v.shape for k, v in a.items()} == {"loss_terms": (4,), **{k: v.shape for k, v in init.items()}}
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["loss_terms"].tolist() == line["config"]["loss_terms"]        # the step whose loss the JSON line reports
    # one Adam step from the seeded weights: no parameter moved by more than the learning rate, and most moved
    for k, p0 in init.items():
        d = np.abs(a[k] - p0)
        assert d.max() <= LR * (1 + 1e-3), k
    assert np.mean([np.mean(np.abs(a[k] - p0) > 0.5 * LR) for k, p0 in init.items()]) > 0.5
    _, b = _bench(tmp_path / "b", 3)
    np.testing.assert_allclose(b["loss_terms"], a["loss_terms"], rtol=1e-5)
    for k in init:
        d = np.abs(b[k] - a[k])
        assert d.max() <= 1e-2 * LR, (k, float(d.max()), int((d > 1e-4 * LR).sum()), d.size)
