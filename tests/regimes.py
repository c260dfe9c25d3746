"""Weights that look like a model that has trained for a while, built from the perturbed init of tests/helpers.py: small
posterior and prior scales, saturated decoder logits, a nearly one-hot q(y|x), and all of them at once.

Every builder takes a Spec and an fp64 parameter dict, edits a copy deterministically and returns it.  The targets each one
reaches (scale range, |logit| percentiles, peakedness of q(y|x)) are asserted on the oracle's forward pass by
tests/test_trained_regime_cpu.py, on the inputs the GPU parity tests use."""
import math

import torch

from oracle import gmvae_oracle as O
from tests.helpers import CONFIGS, make_spec, perturbed_params

SCALE_HI = 0.1             # largest scale of the log-uniform spread
RAW_W_SCALE = 0.1          # the raw (scale) half of the last layer's weights is shrunk by this: the bias sets the scale
FLOORS = (1e-3, 1e-5, 1e-7, 1e-8)   # 1e-8: exp(t) < 2^-24, where 1 + exp(t) rounds to 1 in fp32
TRAINED_FLOOR = 1e-4
GMP_SCALE = (0.02, 0.1)    # VAE_GMP component scales, log-uniform
GMP_LOC_SPREAD = 2.0       # VAE_GMP component means ~ N(0, 2^2) per coordinate
LOGIT_SCALE = 12.0         # saturated_decoder: median |logit| on its probe batch
PEAK_MEDIAN = 15.5         # peaked_y: median over a probe of the margin of component 0 over the rest, less ln(K - 1) ...
PEAK_SPREAD = 3.0          # ... and its standard deviation


def _last(spec, net):
    n = 1 if net == "prior_gmm" else len(spec.hidden_sizes) + 1
    return f"{net}_fcnet/linear_{n - 1}/w", f"{net}_fcnet/linear_{n - 1}/b"


def _inv_softplus(s):
    return torch.log(torch.expm1(s))


def scale_targets(Z, floor, hi=SCALE_HI):
    """Per latent dimension: hi, ..., floor, log-uniform."""
    if Z == 1:
        return torch.tensor([floor], dtype=torch.float64)
    return hi * (floor / hi) ** torch.linspace(0.0, 1.0, Z, dtype=torch.float64)


def scales(spec, params, floor):
    """softplus(raw + raw_sigma_bias) spread log-uniformly per latent dimension from SCALE_HI down to `floor`, in q(z|.) and,
    for the GMVAE, in p(z|y).  VAE_GMP: tight components (scales in GMP_SCALE) with means spread apart."""
    p = dict(params)
    Z = spec.latent_size
    tgt = _inv_softplus(scale_targets(Z, floor)) - spec.raw_sigma_bias
    for net in (("encoder_gmm", "prior_gmm") if spec.model == "gmvae" else ("encoder",)):
        wn, bn = _last(spec, net)
        w, b = p[wn].clone(), p[bn].clone()
        w[:, Z:] *= RAW_W_SCALE
        b[Z:] = tgt
        p[wn], p[bn] = w, b
    if spec.model == "vae_gmp":
        g = torch.Generator().manual_seed(11)
        K = spec.mixture_components
        lo, hi = GMP_SCALE
        sc = lo * (hi / lo) ** torch.rand(K, Z, generator=g, dtype=torch.float64)
        p["raw_scale_diag"] = _inv_softplus(sc)
        p["loc"] = GMP_LOC_SPREAD * torch.randn(K, Z, generator=g, dtype=torch.float64)
    return p


def saturated_decoder(spec, params):
    """The decoder's last layer scaled so that the median |logit| is LOGIT_SCALE on a probe batch of synthetic rows, run through
    the model as it stands (so that, after `scales`, the codes are the near-deterministic ones of a small-scale posterior)."""
    p = dict(params)
    x, _, eps, u = O.synthetic_batch(spec, 256, seed_data=12, seed_noise=21)
    lg = O.loss_terms(spec, p, x, eps, u)["logits_x"] - spec.gen_bias_init
    f = LOGIT_SCALE / lg.abs().median().item()
    wn, bn = _last(spec, "decoder")
    p[wn], p[bn] = p[wn] * f, p[bn] * f
    return p


def peaked_y(spec, params):
    """GMVAE: q(y|x) nearly one-hot on component 0 (a collapsed mixture).  encoder_y's last layer is scaled and component 0's
    logit raised so that, on a probe of synthetic rows, the margin l_0 - max_{k>0} l_k has median PEAK_MEDIAN + ln(K - 1) and
    standard deviation PEAK_SPREAD: most rows have 1 - q(y=0|x) around 1e-7, a tail of rows around 1e-3."""
    K = spec.mixture_components
    if spec.model != "gmvae" or K == 1:
        return dict(params)
    p = dict(params)
    x = O.synthetic_batch(spec, 512, seed_data=13)[0].double()
    lg = O.mlp(p, "encoder_y", x, len(spec.hidden_sizes) + 1)
    d = lg[:, 0] - lg[:, 1:].max(-1).values
    s = PEAK_SPREAD / d.std().item()
    wn, bn = _last(spec, "encoder_y")
    b = p[bn] * s
    b[0] += PEAK_MEDIAN + math.log(K - 1) - s * d.median().item()
    p[wn], p[bn] = p[wn] * s, b
    return p


def trained_like(spec, params):
    return saturated_decoder(spec, peaked_y(spec, scales(spec, params, TRAINED_FLOOR)))


def build(regime, spec, params):
    """`regime`: "scales:<floor>", "saturated_decoder", "peaked_y" or "trained_like"."""
    if regime.startswith("scales:"):
        return scales(spec, params, float(regime[7:]))
    return {"saturated_decoder": saturated_decoder, "peaked_y": peaked_y, "trained_like": trained_like}[regime](spec, params)


SCALES = [f"scales:{f:g}" for f in FLOORS]
REGIMES = SCALES + ["saturated_decoder", "peaked_y", "trained_like"]


# --------------------------------------------------------------------------- the cases of tests/test_trained_regime_gpu.py
# Z = 64 (the chained kernel's z row job) with the fused y head (K = 10), the warp y head (K = 20), K = 128, and the generic z
# heads (Z = 65, Z = 260).  The cfg4 model (`big`) runs on B rows of tests/test_step_gpu.py's full-size inputs.
SMALL = ["cfg1", "cfg2", "cfg3", "k20_ragged", "k128_gmvae", "z65_gmp", "z260_gmvae"]
BIG_BATCHES = (4096, 16384)
BIG_REGIMES = ("scales:1e-05", "trained_like")


def regimes_of(name):
    return [r for r in REGIMES if r != "peaked_y" or CONFIGS[name]["model"] == "gmvae"]


def case(name, regime, objective="reference", T=None, B=None):
    return dict(name=name, regime=regime, objective=objective, T=T, B=B)


def case_id(c):
    s = f"{c['name']}{'_B%d' % c['B'] if c['B'] else ''}-{c['regime']}"
    if c["objective"] != "reference":
        s += "-" + c["objective"]
    if c["T"] is not None:
        s += f"-T={c['T']:g}"
    return s


SMALL_CASES = [case(n, r) for n in SMALL for r in regimes_of(n)]
BIG_CASES = [case("cfg4", r, B=B) for B in BIG_BATCHES for r in BIG_REGIMES]
MARGINAL_CASES = [case(n, r, objective="marginal") for n in ("tiny_gmvae", "cfg3") for r in ("scales:1e-05", "scales:1e-08", "peaked_y")]
TEMPERATURE_CASES = [case(n, "peaked_y", T=0.5) for n in ("cfg3", "k20_ragged")]
DETERMINISTIC_CASE = case("cfg4", "scales:1e-05", B=4096)


def setup(c):
    """(cfg, spec, params, x, eps, u) of a case: the regime's weights and the inputs the GPU test feeds the engine."""
    if c["B"]:
        from tests.test_step_gpu import FULL, _full_inputs
        cfg = dict(FULL, batch=c["B"])
        x, eps, u = _full_inputs(c["B"])
    else:
        cfg = dict(CONFIGS[c["name"]])
        x, _, eps, u = O.synthetic_batch(make_spec(cfg), cfg["batch"], objective=c["objective"])
    if c["T"] is not None:
        cfg["temperature"] = c["T"]
    spec = make_spec(cfg)
    return cfg, spec, build(c["regime"], spec, perturbed_params(spec)), x, eps, u
