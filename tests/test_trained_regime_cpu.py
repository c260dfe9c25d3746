"""The trained-model regimes of tests/regimes.py on the CPU: each builder reaches its targets in the fp64 oracle's forward pass,
the oracle stays finite, and every bound of tests/test_trained_regime_gpu.py is at least what the arithmetic itself allows:
  fp32 mode  the oracle evaluated in fp32 against the fp64 oracle, per loss term and per gradient tensor (and, where one decoder
             unit sits within fp32 reach of its ReLU's kink, what flipping that unit moves the decoder tensors by);
  bf16 mode  the oracle under the bf16 rounding model (helpers.Bf16Model) against the exact oracle, per loss term; and, for the
             gradient bounds listed, that oracle evaluated in fp32 against the same in fp64.
A bound that is not the suite's standard one is listed in the GPU file with this figure beside it."""
import pytest
import torch

from oracle import gmvae_oracle as O
from tests import regimes as R
from tests.helpers import Bf16Model, KL_ABS_FLOOR
from tests.test_trained_regime_gpu import (BF16_CASES, FP32_BOUND, FP32_CASES, FP32_MASK_FLIP, GRAD_BF16_BOUND, NENT_ABS_FLOOR,
                                           TERMS_BF16_BOUND, TOL, fp32_bound, terms_bf16_bound)

TERMS = ("loss", "nll", "kl_div_z", "nent")
_MEMO = {}


def _ref(c, q=O.EXACT, dtype=torch.float64):
    """(terms, grads) of the oracle on a case, in `dtype`, under rounding model `q` (memoised: the cases share them)."""
    key = (R.case_id(c), type(q).__name__, dtype)
    if key not in _MEMO:
        cfg, spec, params, x, eps, u = R.setup(c)
        params = {k: v.to(dtype) for k, v in params.items()}
        _MEMO[key] = O.loss_and_grads(spec, params, x.bool(), eps.to(dtype), None if u is None else u.to(dtype),
                                      objective=c["objective"], q=q)
    return _MEMO[key]


def _rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def mask_flip_figure(c, layer):
    """The decoder pre-activation of `layer` nearest zero, relative to the layer's rms, and what flipping that one ReLU moves each
    decoder gradient tensor by in the fp64 oracle."""
    cfg, spec, params, x, eps, u = R.setup(c)
    z = _ref(c)[0]["z"]
    dec = {k: v.clone().requires_grad_(True) for k, v in params.items() if k.startswith("decoder")}
    L = len(spec.hidden_sizes) + 1

    def grads(flip):
        h = z
        for i in range(L):
            h = h @ dec[f"decoder_fcnet/linear_{i}/w"] + dec[f"decoder_fcnet/linear_{i}/b"]
            if i != L - 1:
                if i == layer:
                    pre = h.detach()
                m = (h > 0).double()
                if flip is not None and i == layer:
                    m[flip] = 1.0 - m[flip]
                h = h * m
        nll = -O.bernoulli_log_prob(x.double(), h + spec.gen_bias_init).sum() / len(x)
        return pre, dict(zip(dec, torch.autograd.grad(nll, list(dec.values()))))

    pre, g0 = grads(None)
    at = divmod(int(pre.abs().argmin()), pre.shape[1])
    _, g1 = grads(at)
    return (pre.abs().min() / pre.pow(2).mean().sqrt()).item(), {n: _rel(g1[n], g0[n]) for n in g0}


def fp32_figures(c):
    """The oracle in fp32 against the fp64 oracle: true relative error of each loss term, ||g - g*|| / ||g*|| of each tensor; for
    the cases of FP32_MASK_FLIP, the decoder tensors take the larger of that and the mask-flip figure."""
    t64, g64 = _ref(c)
    t32, g32 = _ref(c, dtype=torch.float32)
    out = {k: (0.0 if t64[k].item() == 0.0 and t32[k].item() == 0.0 else abs(t32[k].item() - t64[k].item()) / abs(t64[k].item()))
           for k in TERMS}
    out.update({n: _rel(g32[n], g64[n]) for n in g64})
    if R.case_id(c) in FP32_MASK_FLIP:
        for n, v in mask_flip_figure(c, FP32_MASK_FLIP[R.case_id(c)])[1].items():
            out[n] = max(out[n], v)
    return out


def grad_bf16_figures(c):
    """The rounding-model oracle evaluated in fp32 against the same in fp64: ||g - g*|| / ||g*|| per tensor, and their rms."""
    _, g64 = _ref(c, q=Bf16Model(True))
    _, g32 = _ref(c, q=Bf16Model(True), dtype=torch.float32)
    out = {n: _rel(g32[n], g64[n]) for n in g64}
    out["rms"] = (sum(v * v for v in out.values()) / len(out)) ** 0.5
    return out


def bf16_figures(c):
    """The oracle under the bf16 rounding model against the exact one, in the units of the GPU file's term bars: loss and nll
    true relative, kl_div_z relative to max(|kl|, 1 nat), nent absolute (nats)."""
    te, _ = _ref(c)
    tm, _ = _ref(c, q=Bf16Model(True))
    d = {k: abs(tm[k].item() - te[k].item()) for k in TERMS}
    return {"loss": d["loss"] / abs(te["loss"].item()), "nll": d["nll"] / abs(te["nll"].item()),
            "kl_div_z": d["kl_div_z"] / max(abs(te["kl_div_z"].item()), KL_ABS_FLOOR), "nent": d["nent"]}


# ------------------------------------------------------------------ the builders' targets
TARGET_CASES = R.SMALL_CASES + R.BIG_CASES + R.MARGINAL_CASES + R.TEMPERATURE_CASES


def _floor(regime):
    if regime.startswith("scales:"):
        return float(regime[7:])
    return R.TRAINED_FLOOR if regime == "trained_like" else None


@pytest.mark.parametrize("c", TARGET_CASES, ids=R.case_id)
def test_regime_targets(c):
    cfg, spec, params, x, eps, u = R.setup(c)
    t, _ = _ref(c)
    reg = c["regime"]
    F = _floor(reg)
    if F is not None:
        Z = spec.latent_size
        tgt = R.scale_targets(Z, F)
        for k in ("sigma_q", "sigma_p"):
            if k not in t:
                continue
            s = t[k].reshape(-1, Z)
            med = s.median(0).values
            assert ((med / tgt).log().abs() < 0.7).all(), (k, "per-dimension median off the log-uniform target")  # factor 2
            assert F / 4 <= s.min().item() <= 2 * F, (k, s.min().item(), F)
            assert s.max().item() <= 3 * R.SCALE_HI, (k, s.max().item())
        if spec.model == "vae_gmp":
            sc = O.softplus(params["raw_scale_diag"])
            assert R.GMP_SCALE[0] * 0.99 <= sc.min().item() and sc.max().item() <= R.GMP_SCALE[1] * 1.01
            dist = torch.cdist(params["loc"], params["loc"]) + torch.eye(spec.mixture_components) * 1e9
            assert dist.min().item() >= 10 * sc.max().item(), "components are not well separated"
    if reg in ("saturated_decoder", "trained_like"):
        a = t["logits_x"].abs()
        assert a.median().item() >= 8, a.median().item()
        assert (a >= 20).double().mean().item() >= 0.05, (a >= 20).double().mean().item()
    if reg in ("peaked_y", "trained_like") and spec.model == "gmvae":
        q = torch.softmax(t["logits_y"], -1).max(-1).values
        assert (q >= 0.999).double().mean().item() >= 0.9
        assert (q >= 1 - 1e-6).double().mean().item() >= 0.5
        assert -1e-2 < t["nent"].item() < 0, t["nent"].item()


@pytest.mark.parametrize("c", TARGET_CASES, ids=R.case_id)
def test_oracle_finite(c):
    t, g = _ref(c)
    for k in TERMS:
        assert torch.isfinite(t[k]).all(), k
    for n, v in g.items():
        assert torch.isfinite(v).all(), n


# ------------------------------------------------------------------ every bound of the GPU file against the arithmetic's own figure
@pytest.mark.parametrize("c", FP32_CASES, ids=R.case_id)
def test_fp32_bounds_cover_fp32_arithmetic(c):
    fig = fp32_figures(c)
    for k, v in fig.items():
        assert fp32_bound(c, k) >= v, (R.case_id(c), k, "fp32 oracle vs fp64", v, "bound", fp32_bound(c, k))


@pytest.mark.parametrize("c", BF16_CASES, ids=R.case_id)
def test_bf16_term_bounds_cover_rounding_model(c):
    fig = bf16_figures(c)
    for k in ("loss", "nll", "kl_div_z"):
        assert terms_bf16_bound(c, k) >= fig[k], (R.case_id(c), k, "rounding model vs exact", fig[k], terms_bf16_bound(c, k))
    nent = abs(_ref(c)[0]["nent"].item())
    assert TOL["bf16"] * max(nent, NENT_ABS_FLOOR) >= fig["nent"], (R.case_id(c), "nent", fig["nent"])


@pytest.mark.parametrize("cid", sorted(FP32_MASK_FLIP))
def test_mask_flip_is_within_fp32_reach(cid):
    """The unit of each FP32_MASK_FLIP figure sits within 1e-6 of its layer's rms from zero: fp32 accumulation decides it."""
    c = {R.case_id(k): k for k in FP32_CASES}[cid]
    rel_pre, _ = mask_flip_figure(c, FP32_MASK_FLIP[cid])
    assert rel_pre < 1e-6, rel_pre


def test_listed_bounds_are_used_and_at_least_twice_their_figure():
    """Every entry of FP32_BOUND / TERMS_BF16_BOUND names a case the GPU file runs, is needed (its figure exceeds the standard
    bar) and holds 2x (at least) its figure."""
    fp32_ids = {R.case_id(c): c for c in FP32_CASES}
    bf16_ids = {R.case_id(c): c for c in BF16_CASES}
    for (cid, k), b in FP32_BOUND.items():
        assert cid in fp32_ids, cid
        fig = max(v for n, v in fp32_figures(fp32_ids[cid]).items() if n == k or n.split("/")[0] == k)
        assert b >= 2 * fig and fig > TOL["fp32"], (cid, k, b, fig)
    for (cid, k), b in TERMS_BF16_BOUND.items():
        assert cid in bf16_ids, cid
        fig = bf16_figures(bf16_ids[cid])[k]
        assert b >= 2 * fig and fig > TOL["bf16"], (cid, k, b, fig)
    for (cid, k), b in GRAD_BF16_BOUND.items():
        assert cid in bf16_ids, cid
        fig = max(v for n, v in grad_bf16_figures(bf16_ids[cid]).items() if n == k or n.split("/")[0] == k)
        assert b >= 2 * fig and fig > (1.5 if k == "rms" else 3) * TOL["bf16"], (cid, k, b, fig)
