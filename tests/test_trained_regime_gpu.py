"""The training step at the value ranges of a model that has trained for a while (tests/regimes.py): posterior and prior scales
down to 1e-8, saturated decoder logits, a nearly one-hot q(y|x), and all of them at once, against the fp64 oracle on the same
weights, inputs and noise.

Bars (those of tests/test_step_gpu.py unless a case is listed below with its figure):
  finite     wherever the fp64 oracle is finite, every loss term and every gradient tensor of the engine is finite;
  fp32 mode  every loss term (true relative) and every gradient tensor (||g - g*|| / ||g*||) within 1e-5 of the fp64 oracle;
  bf16 mode  loss and nll within 2e-3 (true relative) of the exact oracle, kl_div_z within 2e-3 * max(|kl|, 1 nat), nent within
             2e-3 * max(|nent|, NENT_ABS_FLOOR); gradients against the oracle under the bf16 rounding model: rms over tensors
             < 3e-3, every tensor < 6e-3;
  plans      the bf16 step under the launch plans 0 (heads as kernels below 4 096 rows), 8192 (heads as row jobs of one chained
             launch) and 512 (one launch per GEMM) agree with each other within the same bars, so that a failure points at one
             plan's heads.
tests/test_trained_regime_cpu.py checks every bound against the arithmetic's own figure (the oracle evaluated in fp32, and the
oracle under the bf16 rounding model) and every builder's targets."""
import pytest
import torch

from oracle import gmvae_oracle as O
from tests import regimes as R
from tests.helpers import KL_ABS_FLOOR, Bf16Model, make_engine
from tests.test_step_gpu import _record

pytestmark = pytest.mark.gpu

TOL = {"fp32": 1e-5, "bf16": 2e-3}
TERMS = ("loss", "nll", "kl_div_z", "nent")
PLANS = ("0", "8192", "512")

# Not in the fp32 mode: cfg3-peaked_y under objective M.  Its encoder_y gradient is q_k (c_k - sum_j q_j c_j) with per-component
# costs c_k ~ 500 nats that differ by less than their own fp32 rounding: the oracle evaluated in fp32 is 13 % away from the fp64
# one on those tensors, and the engine 26 % (B200), so no bar there would say anything about the kernels.  The bf16 mode runs it
# against the rounding-model bound below; tiny_gmvae-peaked_y runs objective M in both modes.
FP32_CASES = R.SMALL_CASES + [c for c in R.MARGINAL_CASES if R.case_id(c) != "cfg3-peaked_y-marginal"] + R.TEMPERATURE_CASES
BF16_CASES = R.SMALL_CASES + R.BIG_CASES + R.MARGINAL_CASES + R.TEMPERATURE_CASES   # (the deterministic case is one of BIG_CASES)

# fp32 mode, (case, loss term or network) -> bound for that term or every tensor of that network: 2x the largest figure of the
# oracle evaluated in fp32 against the fp64 oracle, where it exceeds 1e-5 (the figure beside each).  The sources of those figures:
#   scales, VAE   logq = -((z - mu) / sigma)^2 / 2 cancels in fp32 when sigma is below ulp(mu) (the kernels use eps directly);
#   peaked_y      lse = ml + log(sl) with sl = 1 + O(1e-7) loses nent's digits, and dL/dlogits_y = q (c - sum q c) cancels;
#   cfg2 saturated_decoder   the same cancellations in the mixture prior's log-sum-exp and the saturated BCE.
# Two entries have a figure of another kind, FP32_MASK_FLIP: on these weights one decoder pre-activation lies within 4e-7 of the
# layer's rms from zero, where fp32 accumulation order decides the ReLU; the figure is what flipping that one unit moves the
# decoder tensors by in the fp64 oracle (the fp32 oracle happens to decide it as fp64 does).
FP32_BOUND = {
    ("cfg3-scales:1e-05", "decoder_fcnet"): 9.0e-04,   # 4.50e-04 (mask flip, layer 0)
    ("cfg3-scales:1e-07", "decoder_fcnet"): 3.8e-03,   # 1.87e-03 (mask flip, layer 1)
    ("cfg1-scales:1e-05", "encoder_fcnet"): 4.9e-04,   # 2.43e-04
    ("cfg1-scales:1e-07", "loss"): 6.7e-05,   # 3.34e-05
    ("cfg1-scales:1e-07", "kl_div_z"): 1.4e-04,   # 6.56e-05
    ("cfg1-scales:1e-07", "encoder_fcnet"): 6.4e-02,   # 3.18e-02
    ("cfg1-scales:1e-08", "loss"): 9.3e-05,   # 4.61e-05
    ("cfg1-scales:1e-08", "kl_div_z"): 1.8e-04,   # 8.53e-05
    ("cfg1-scales:1e-08", "encoder_fcnet"): 2.3e-01,   # 1.10e-01
    ("cfg2-scales:1e-08", "encoder_fcnet"): 9.1e-05,   # 4.53e-05
    ("cfg2-saturated_decoder", "decoder_fcnet"): 1.6e-03,   # 7.84e-04
    ("cfg2-saturated_decoder", "encoder_fcnet"): 5.5e-04,   # 2.72e-04
    ("cfg3-peaked_y", "nent"): 1.4e-03,   # 6.57e-04
    ("cfg3-peaked_y", "encoder_y_fcnet"): 1.8e-03,   # 8.97e-04
    ("cfg3-trained_like", "nent"): 1.4e-03,   # 6.57e-04
    ("cfg3-trained_like", "encoder_y_fcnet"): 4.9e-03,   # 2.41e-03
    ("k20_ragged-peaked_y", "nent"): 4.0e-04,   # 1.98e-04
    ("k20_ragged-peaked_y", "encoder_y_fcnet"): 4.6e-04,   # 2.27e-04
    ("k20_ragged-trained_like", "nent"): 4.0e-04,   # 1.98e-04
    ("k20_ragged-trained_like", "encoder_y_fcnet"): 5.9e-04,   # 2.91e-04
    ("k128_gmvae-peaked_y", "nent"): 5.0e-04,   # 2.45e-04
    ("k128_gmvae-peaked_y", "encoder_y_fcnet"): 2.6e-04,   # 1.29e-04
    ("k128_gmvae-trained_like", "nent"): 5.0e-04,   # 2.45e-04
    ("k128_gmvae-trained_like", "encoder_y_fcnet"): 1.4e-03,   # 6.55e-04
    ("z65_gmp-scales:1e-08", "encoder_fcnet"): 7.9e-05,   # 3.93e-05
    ("z260_gmvae-peaked_y", "nent"): 1.8e-04,   # 8.67e-05
    ("z260_gmvae-peaked_y", "encoder_y_fcnet"): 2.6e-04,   # 1.29e-04
    ("z260_gmvae-trained_like", "nent"): 1.8e-04,   # 8.67e-05
    ("z260_gmvae-trained_like", "encoder_y_fcnet"): 2.7e-03,   # 1.33e-03
    ("tiny_gmvae-peaked_y-marginal", "nent"): 6.8e-05,   # 3.36e-05
    ("tiny_gmvae-peaked_y-marginal", "encoder_y_fcnet"): 2.7e-03,   # 1.31e-03
    ("cfg3-peaked_y-T=0.5", "nent"): 1.4e-03,   # 6.57e-04
    ("cfg3-peaked_y-T=0.5", "encoder_y_fcnet"): 3.2e-04,   # 1.56e-04
    ("k20_ragged-peaked_y-T=0.5", "nent"): 4.0e-04,   # 1.98e-04
    ("k20_ragged-peaked_y-T=0.5", "encoder_y_fcnet"): 1.4e-04,   # 6.57e-05
}
FP32_MASK_FLIP = {"cfg3-scales:1e-05": 0, "cfg3-scales:1e-07": 1}     # case -> decoder layer of the flipped unit
# bf16 loss terms, (case, term) -> bound: 2x the figure of the oracle under the bf16 rounding model against the exact oracle,
# where it exceeds 2e-3 (the figure beside each).  With prior scales down to 1e-7, kl_div_z is dominated by
# (z - mu_p)^2 / sigma_p^2 ~ 1e15, which the bf16 rounding of the encoder's and the prior's GEMM operands moves by that much.
TERMS_BF16_BOUND = {
    ("cfg3-scales:1e-07", "loss"): 4.4e-03,   # 2.20e-03
    ("cfg3-scales:1e-07", "kl_div_z"): 4.4e-03,   # 2.20e-03
    ("cfg3-scales:1e-08", "loss"): 5.2e-03,   # 2.59e-03
    ("cfg3-scales:1e-08", "kl_div_z"): 5.2e-03,   # 2.59e-03
    ("tiny_gmvae-scales:1e-05-marginal", "loss"): 4.6e-03,   # 2.25e-03
    ("tiny_gmvae-scales:1e-05-marginal", "kl_div_z"): 4.6e-03,   # 2.25e-03
    ("tiny_gmvae-scales:1e-08-marginal", "loss"): 6.2e-03,   # 3.08e-03
    ("tiny_gmvae-scales:1e-08-marginal", "kl_div_z"): 6.2e-03,   # 3.08e-03
    ("cfg3-scales:1e-08-marginal", "loss"): 4.6e-03,   # 2.27e-03
    ("cfg3-scales:1e-08-marginal", "kl_div_z"): 4.6e-03,   # 2.27e-03
}
# bf16 gradients against the rounding-model oracle, (case, network or "rms") -> bound: 2x the figure of the rounding-model oracle
# evaluated in fp32 against the same in fp64, where it exceeds 6e-3 (3e-3 for the rms).  Objective M with a peaked q(y|x):
# dL/dlogits_y = q (c - sum_k q_k c_k), and the per-component costs c_k = kl_k - rec_k (~500 nats, summed in fp32 over 784
# pixels) differ by far less than their own fp32 rounding.
GRAD_BF16_BOUND = {
    ("cfg3-peaked_y-marginal", "encoder_y_fcnet"): 2.9e-01,   # 1.41e-01
    ("cfg3-peaked_y-marginal", "rms"): 1.5e-01,               # 7.44e-02
}
# nent under a peaked q(y|x) is -1e-5 ... -1e-3 nats, and a relative bar cannot be met by bf16 storage: the bf16 logits of
# encoder_y move the entropy of the least peaked rows.  Below NENT_ABS_FLOOR nats the bar is absolute, 2e-3 * 0.025 = 5e-5 nats;
# the oracle under the rounding model moves nent by at most 2.09e-5 nats from the exact oracle on these cases
# (tiny_gmvae-peaked_y-marginal; 1.75e-6 at most under objective R).
NENT_ABS_FLOOR = 0.025


def fp32_bound(c, k):
    """Bound of loss term or gradient tensor `k` in the fp32 mode (a tensor takes its network's entry)."""
    cid = R.case_id(c)
    return FP32_BOUND.get((cid, k), FP32_BOUND.get((cid, k.split("/")[0]), TOL["fp32"]))


def grad_bf16_bound(c, k):
    """Bound of gradient tensor `k` (or of their rms, k = "rms") in the bf16 mode against the rounding-model oracle."""
    cid = R.case_id(c)
    std = 1.5 * TOL["bf16"] if k == "rms" else 3 * TOL["bf16"]
    return GRAD_BF16_BOUND.get((cid, k), GRAD_BF16_BOUND.get((cid, k.split("/")[0]), std))


def terms_bf16_bound(c, k):
    return TERMS_BF16_BOUND.get((R.case_id(c), k), TOL["bf16"])


def _oracle(c, spec, params, x, eps, u, q=O.EXACT):
    t, g = O.loss_and_grads(spec, params, x.bool(), eps, u, objective=c["objective"], q=q)
    return [t[k].item() for k in TERMS], g


def _step(c, cfg, precision, params, x, eps, u, **kw):
    """Loss terms and gradients (fp64, on the host) of one forward_backward of the engine."""
    eng = make_engine(cfg, precision, objective=c["objective"], **kw)
    eng.set_parameters(params)
    t = eng.forward_backward(x, eps=eps, gumbel_u=u)
    torch.cuda.synchronize()
    out = (t.cpu().double().tolist(), {n: v.detach().cpu().double().clone() for n, v in eng.gradients().items()})
    eng.close()
    return out


def _rel(a, b):
    b = b.double()
    return ((a.reshape(b.shape) - b).norm() / b.norm().clamp_min(1e-30)).item()


def _check_finite(cid, terms, grads, ref_t, ref_g):
    for i, k in enumerate(TERMS):
        if torch.isfinite(torch.tensor(ref_t[i])):
            assert torch.isfinite(torch.tensor(terms[i])), (cid, k, "not finite", terms[i])
    for n, r in ref_g.items():
        if torch.isfinite(r).all():
            assert torch.isfinite(grads[n]).all(), (cid, n, "not finite")


def _term_errors(terms, ref_t, ref_exact):
    """Errors of [loss, nll, kl_div_z, nent] against ref_t in the units of the bf16 bars (the floors taken on the exact oracle)."""
    d = [abs(a - b) for a, b in zip(terms, ref_t)]
    return {"loss": d[0] / abs(ref_exact[0]), "nll": d[1] / abs(ref_exact[1]),
            "kl_div_z": d[2] / max(abs(ref_exact[2]), KL_ABS_FLOOR), "nent": d[3] / max(abs(ref_exact[3]), NENT_ABS_FLOOR)}


def _check_bf16_terms(c, terms, ref_t, ref_exact, what):
    cid = R.case_id(c)
    err = _term_errors(terms, ref_t, ref_exact)
    for k, v in err.items():
        lim = TOL["bf16"] if k == "nent" else terms_bf16_bound(c, k)
        assert v < lim, (cid, what, k, v, lim)
    return err


def _check_bf16_grads(c, grads, ref_g, what):
    cid = R.case_id(c)
    err = {n: _rel(grads[n], r) for n, r in ref_g.items()}
    rms = (sum(v * v for v in err.values()) / len(err)) ** 0.5
    _record(cid, {"precision": "bf16", "what": what, "grad_max": max(err.values()), "grad_rms": rms, "grad": err})
    assert rms < grad_bf16_bound(c, "rms"), (cid, what, "rms over tensors", rms)
    for n, v in err.items():
        assert v < grad_bf16_bound(c, n), (cid, what, n, v)
    return err, rms


def _check_bf16(c, cfg, spec, params, x, eps, u, tag, **kw):
    """One bf16 step against the exact oracle (terms) and the rounding-model oracle (gradients); returns (terms, grads)."""
    cid = R.case_id(c)
    ref_t, ref_g = _oracle(c, spec, params, x, eps, u)
    _, mod_g = _oracle(c, spec, params, x, eps, u, q=Bf16Model(True))
    terms, grads = _step(c, cfg, "bf16", params, x, eps, u, **kw)
    _check_finite(cid, terms, grads, ref_t, ref_g)
    _record(cid, {"precision": "bf16", "plan": tag, "terms": terms, "terms_ref": ref_t})
    _check_bf16_terms(c, terms, ref_t, ref_t, tag + " vs exact oracle")
    _check_bf16_grads(c, grads, mod_g, tag + " vs rounding model")
    return terms, grads, ref_t


# ------------------------------------------------------------------ fp32 mode
@pytest.mark.parametrize("c", FP32_CASES, ids=R.case_id)
def test_fp32(c):
    cid = R.case_id(c)
    cfg, spec, params, x, eps, u = R.setup(c)
    ref_t, ref_g = _oracle(c, spec, params, x, eps, u)
    terms, grads = _step(c, cfg, "fp32", params, x, eps, u)
    _check_finite(cid, terms, grads, ref_t, ref_g)
    err = {k: (0.0 if ref_t[i] == 0.0 and terms[i] == 0.0 else abs(terms[i] - ref_t[i]) / abs(ref_t[i])) for i, k in enumerate(TERMS)}
    err.update({n: _rel(grads[n], r) for n, r in ref_g.items()})
    _record(cid, {"precision": "fp32", "err": err})
    for k, v in err.items():
        assert v < fp32_bound(c, k), (cid, k, v, fp32_bound(c, k))


# ------------------------------------------------------------------ bf16 mode under the three launch plans, and across them
@pytest.mark.parametrize("c", R.SMALL_CASES + R.TEMPERATURE_CASES, ids=R.case_id)
def test_bf16_launch_plans(c, monkeypatch):
    cfg, spec, params, x, eps, u = R.setup(c)
    runs = {}
    for flags in PLANS:
        monkeypatch.setenv("GMVAE_DEBUG_FLAGS", flags)
        runs[flags] = _check_bf16(c, cfg, spec, params, x, eps, u, "flags=" + flags)
    ref_t = runs[PLANS[0]][2]
    for i, a in enumerate(PLANS):
        for b in PLANS[i + 1:]:
            what = f"flags={a} vs flags={b}"
            _check_bf16_terms(c, runs[a][0], runs[b][0], ref_t, what)
            _check_bf16_grads(c, runs[a][1], runs[b][1], what)


# ------------------------------------------------------------------ the cfg4 model on the default plan (one chained launch)
@pytest.mark.parametrize("c", R.BIG_CASES, ids=R.case_id)
def test_bf16_cfg4_default_plan(c):
    cfg, spec, params, x, eps, u = R.setup(c)
    _check_bf16(c, cfg, spec, params, x, eps, u, "default")


# ------------------------------------------------------------------ objective M, deterministic mode
@pytest.mark.parametrize("c", R.MARGINAL_CASES, ids=R.case_id)
def test_bf16_marginal(c, monkeypatch):
    monkeypatch.setenv("GMVAE_M_CHUNK_ROWS", "512")          # as test_step_gpu.test_parity_marginal_bf16
    cfg, spec, params, x, eps, u = R.setup(c)
    _check_bf16(c, cfg, spec, params, x, eps, u, "marginal")


def test_bf16_deterministic():
    """Deterministic mode on the same plan: the bars, and a second engine gives the same bits."""
    c = R.DETERMINISTIC_CASE
    cfg, spec, params, x, eps, u = R.setup(c)
    terms, grads, _ = _check_bf16(c, cfg, spec, params, x, eps, u, "deterministic", deterministic=True)
    terms2, grads2 = _step(c, cfg, "bf16", params, x, eps, u, deterministic=True)
    assert terms == terms2
    for n in grads:
        assert torch.equal(grads[n], grads2[n]), n
