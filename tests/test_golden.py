"""Committed golden vectors (tests/golden/*.json, written by tests/tools/make_golden.py from the oracle).
CPU: the oracle still reproduces them bit-for-bit-ish (regression pin).  GPU: the CUDA step in the
fp32 validation mode matches them to rel 1e-5 and in bf16 mode the loss terms to 2e-3."""
import glob
import json
import os

import pytest
import torch

from oracle import gmvae_oracle as O
from tests.helpers import make_spec, perturbed_params, rel

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.json")))


def _load(path):
    rec = json.load(open(path))
    cfg = rec["config"]
    spec = make_spec(cfg)
    params = perturbed_params(spec, seed=rec["params_seed"])
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"], rec["data_seed"], rec["noise_seed"])
    assert int(x.sum()) == rec["x_sum"] and abs(eps.double().sum().item() - rec["eps_sum"]) < 1e-9
    return rec, cfg, spec, params, x, eps, u


def test_golden_files_present():
    assert len(GOLDEN) >= 8


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-5] for p in GOLDEN])
def test_oracle_reproduces_golden(path):
    rec, cfg, spec, params, x, eps, u = _load(path)
    terms, grads = O.loss_and_grads(spec, params, x, eps, u)
    for k, v in rec["terms"].items():
        assert abs(terms[k].item() - v) <= 1e-11 * max(1.0, abs(v)), k
    for n, v in rec["grad_norms"].items():
        assert abs(grads[n].norm().item() - v) <= 1e-10 * max(1e-6, v), n
    for n, pts in rec["grad_samples"].items():
        flat = grads[n].reshape(-1)
        for i, v in pts:
            assert abs(flat[i].item() - v) <= 1e-12 + 1e-9 * abs(v)
    if "terms_marginal" in rec:                                       # objective M on the same inputs, eps [B, K, Z]
        eps_m = torch.randn(cfg["batch"], spec.mixture_components, spec.latent_size,
                            generator=torch.Generator().manual_seed(rec["noise_seed"]))
        tm, _ = O.loss_and_grads(spec, params, x, eps_m, u, "marginal")
        for k, v in rec["terms_marginal"].items():
            assert abs(tm[k].item() - v) <= 1e-11 * max(1.0, abs(v)), ("marginal", k)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-5] for p in GOLDEN])
def test_cuda_step_matches_golden(path, precision):
    from tests.helpers import make_engine
    rec, cfg, spec, params, x, eps, u = _load(path)
    eng = make_engine(cfg, precision)
    eng.set_parameters(params)
    t = eng.forward_backward(x, eps=eps, gumbel_u=u).cpu().tolist()
    tol = 1e-5 if precision == "fp32" else 2e-3
    for i, k in enumerate(("loss", "nll", "kl_div_z", "nent")):
        ref = rec["terms"][k]
        if ref == 0.0 and t[i] == 0.0:
            continue
        # true relative error; bf16 kl_div_z below one nat: absolute 2e-3 nats (tests/helpers.bf16_term_ok)
        floor = 1.0 if (precision == "bf16" and k == "kl_div_z") else 1e-30
        assert abs(t[i] - ref) / max(abs(ref), floor) < tol, (k, t[i], ref)
    if precision == "fp32":
        grads = eng.gradients()
        for n, v in rec["grad_norms"].items():
            assert rel(grads[n].norm().item(), v) < 1e-5, n
        for n, pts in rec["grad_samples"].items():
            flat = grads[n].reshape(-1).cpu()
            for i, v in pts:
                assert abs(flat[i].item() - v) <= 1e-5 * rec["grad_norms"][n], (n, i)
    eng.close()
