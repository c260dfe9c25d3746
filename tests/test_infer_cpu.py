"""The bounds of tests/test_infer_gpu.py, checked on the CPU: every fp32 bound is at least twice the oracle's own fp32 evaluation
error on its case (and the bf16 bound at least twice the rounding model's own fp32 evaluation error), and the element-wise
comparisons reject planted errors that the earlier max|got - ref| / max|ref| < 2e-2 bar accepts."""
import pytest
import torch

from oracle import gmvae_oracle as O
from tests import regimes
from tests.helpers import CONFIGS, make_spec, perturbed_params
from tests.test_infer_gpu import (OLD_BAR, TOL, TRAINED, InferRound, case_inputs, figure, old_bar, prior_case, prior_reference,
                                  reference, value)

CASES = [(n, None) for n in CONFIGS] + TRAINED


def _setup(name, regime):
    cfg = CONFIGS[name]
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    if regime:
        params = regimes.build(regime, spec, params)
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    return spec, params, x, eps, u


def _gaps(spec, params, x, eps, u, q, tol):
    """Worst figure, per output, of the reference evaluated in fp32 against the same reference in fp64."""
    z, y = case_inputs(spec, params, x, eps, u)
    r64 = reference(spec, params, x, eps, u, z, y, q)
    r32 = reference(spec, params, x, eps, u, z, y, q, dt=torch.float32)
    return {k: figure(r64[k], value(r32[k], spec.sigma_min), tol, spec.sigma_min) for k in r64 if k != "encode.y"}


@pytest.mark.parametrize("name,regime", CASES, ids=[n if r is None else f"{n}-{r}" for n, r in CASES])
def test_bounds_cover_the_oracles_own_fp32_error(name, regime):
    spec, params, x, eps, u = _setup(name, regime)
    g = _gaps(spec, params, x, eps, u, InferRound(False), TOL["fp32"])
    bad = {k: v for k, v in g.items() if not 2 * v <= TOL["fp32"]}
    assert not bad, (name, regime, "fp32 bound < 2x the fp32-vs-fp64 oracle gap", bad)
    g = _gaps(spec, params, x, eps, u, InferRound(True), TOL["bf16"])
    bad = {k: v for k, v in g.items() if not 2 * v <= TOL["bf16"]}
    assert not bad, (name, regime, "bf16 bound < 2x the rounding model's own fp32-vs-fp64 gap", bad)


@pytest.mark.parametrize("model,K,Z", [("gmvae", 128, 260), ("vae_gmp", 128, 260)])
def test_prior_bounds_cover_fp32(model, K, Z):
    _, spec, params = prior_case(model, K, Z)
    r64 = prior_reference(spec, {k: v.float() for k, v in params.items()})
    # the table evaluated in fp32, as the kernel does
    p32 = {k: v.float() for k, v in params.items()}
    if model == "gmvae":
        w, b = p32["prior_gmm_fcnet/linear_0/w"], p32["prior_gmm_fcnet/linear_0/b"]
        mu, raw = (w + b)[:, :Z], (w + b)[:, Z:]
        sg = O.softplus(raw + torch.tensor(spec.raw_sigma_bias, dtype=torch.float32)).clamp_min(spec.sigma_min)
    else:
        mu, sg = p32["loc"], O.softplus(p32["raw_scale_diag"])
    assert 2 * figure(r64["prior.mu"], mu, TOL["fp32"]) <= TOL["fp32"]
    assert 2 * figure(r64["prior.sigma"], sg, TOL["fp32"], spec.sigma_min) <= TOL["fp32"]


# --------------------------------------------------------------------------- planted errors
def _planted_case():
    """cfg3 with trained-like weights (scales down to 1e-4, saturated decoder, peaked q(y|x)) and a sigma_min of 1e-3 that holds
    the smallest scales: the exact oracle's outputs."""
    spec, params, x, eps, u = _setup("cfg3", "trained_like")
    spec.sigma_min = float(torch.tensor(1e-3, dtype=torch.float32))
    z, y = case_inputs(spec, params, x, eps, u)
    ref = reference(spec, params, x, eps, u, z, y)
    return spec, ref


def _assert_caught(rec, got, spec, what):
    old = old_bar(rec, got)
    new = figure(rec, got, TOL["fp32"], spec.sigma_min)
    assert old < OLD_BAR, (what, "the max-normalised bar should accept this planted error", old)
    assert new > TOL["fp32"], (what, "the element-wise bound should reject it", new)
    return old, new


def test_planted_row_swap():
    """One row of q(z|x,y)'s sigma replaced by its neighbour: of the rows that differ from the next one, the replacement the
    max-normalised bar sees least (small scales: the rows differ by about 1 % of the largest scale)."""
    spec, ref = _planted_case()
    rec = ref["condition.encoder.sigma"]
    v = value(rec, spec.sigma_min)
    d = (v[1:] - v[:-1]).abs().max(1).values
    d[d == 0] = float("inf")
    i = int(d.argmin())
    got = v.clone()
    got[i] = got[i + 1]
    _assert_caught(rec, got, spec, f"row {i}")


def test_planted_partial_tile():
    """The 16-column partial tile (columns 768-783 of 784: three 256-wide n-tiles and 16 columns) of the decoder's logits
    shifted by 1 %."""
    spec, ref = _planted_case()
    rec = ref["condition.decoder"]
    got = value(rec).clone()
    got[:, 768:784] *= 1.01
    _assert_caught(rec, got, spec, "partial tile")


def test_planted_decode_tail():
    """A decoded probability near 1e-6 returned as 1e-4."""
    spec, ref = _planted_case()
    rec = ref["decode"]
    got = value(rec).clone()
    i = int((got.log() - torch.log(torch.tensor(1e-6, dtype=torch.float64))).abs().argmin())
    assert abs(got.reshape(-1)[i].log10().item() + 6) < 1
    got.reshape(-1)[i] *= 100
    _assert_caught(rec, got, spec, "decode tail")


def test_planted_sigma_at_floor():
    """One sigma held at sigma_min returned as twice sigma_min."""
    spec, ref = _planted_case()
    rec = ref["condition.encoder.sigma"]
    got = value(rec, spec.sigma_min).clone()
    held = (rec[1] < spec.sigma_min * 0.5).nonzero()
    assert held.shape[0] > 0
    r, c = held[0].tolist()
    got[r, c] *= 2
    _assert_caught(rec, got, spec, "sigma at floor")
