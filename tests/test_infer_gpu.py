"""The inference entry points -- gmvae_encode, gmvae_decode, gmvae_condition (all four networks), gmvae_prior_table -- and the
distribution kernels (gmvae_dist_*) against fp64 references, element by element.

Inference never runs the chained kernel: its GEMMs are the stand-alone persistent tensor-core kernel with A K-major and the
weight MN-major, followed by separate head kernels, and some epilogues (the fp32 [mu|raw] store, decode's sigmoid +
gen_bias_init store) run only here.  So it is checked here on its own:

  fp32 mode  against the exact fp64 oracle.
  bf16 mode  against an INFERENCE rounding model (InferRound): every weight operand rounded to bf16 (inference uses the bf16
             shadows of all layers), hidden activations rounded after bias + ReLU, the GEMM inputs z and y rounded (x is
             exact), last-layer outputs (logits_y, [mu|raw], decoder logits) kept in fp32; in encode y is sampled from the
             logits and then rounded as encoder_gmm's operand.  A loose bound against the exact oracle is kept as well.

Every bound is element-wise and scaled by the ABSOLUTE NETWORK: the same MLP evaluated with |W|, |b| and |input|, which bounds
how far an error of relative size tol in every layer can move each output.  A wrong row, column or tile therefore cannot hide
under a large value elsewhere, as it can under max|got - ref| / max|ref|.  Per output, with S its absolute-network scale:

  logits, mu        |d| <= tol * S
  sigma             |d log sigma| <= tol * S_raw + 2^-22 (d log softplus(t) / dt <= 1; 2^-22: the fp32 result); entries the
                    clamp holds at sigma_min (off its kink by more than the tolerance) must equal sigma_min exactly
  decode            |d p| <= p (1 - p) tol S + 2^-23 p + 2^-126: a probability of 1e-13 is held to its own relative precision
  z_sample          |d z| <= tol (S_mu + sigma |eps| S_raw) + 2^-22 (|mu| + sigma |eps|)

Each figure reported (and recorded through test_step_gpu._record) is the worst of (|d| - floor) / scale over an output, i.e.
the smallest tol that passes.  tests/test_infer_cpu.py shows that every fp32 bound is at least twice the oracle's own fp32
evaluation error and that these comparisons reject planted errors that the max-normalised bar accepts."""
import math
import time

import pytest
import torch

from gmvae_b200 import _lib
from gmvae_b200.base import COND_DECODER, COND_ENCODER, COND_ENCODER_Y, COND_PRIOR_GMM
from oracle import gmvae_oracle as O
from tests import regimes
from tests.helpers import CONFIGS, make_engine, make_spec, perturbed_params
from tests.test_config_edges_gpu import _condition
from tests.test_step_gpu import FULL, _full_inputs, _record

pytestmark = pytest.mark.gpu

# Bounds in units of the absolute-network scale (see the module docstring), each at least twice the worst figure measured on one
# B200 (NVIDIA B200, power limit 1000 W) over every case of this file:
#   fp32        measured 8.9e-7 (condition(PRIOR_GMM) mu, k128_gmvae); the oracle evaluated in fp32 instead of fp64 moves the same
#               output by the same 8.9e-7 (the fp32 parameters and inputs), and no output of any case by more (test_infer_cpu.py)
#   bf16        against the rounding model: measured 1.4e-6 (decode, the cfg4-wide VAE_GMP at 16 384 rows); the rounding model
#               evaluated in fp32 instead of fp64 moves condition(ENCODER) mu of k128_gmvae by 1.4e-5 (fp32 accumulation moving an
#               activation across a bf16 rounding boundary), and the bound covers twice that
#   bf16_exact  against the exact oracle: measured 5.5e-3 (condition(PRIOR_GMM) mu, cfg4 at 16 384 rows)
TOL = {"fp32": 2e-6,
       "bf16": 3e-5,
       "bf16_exact": 1.2e-2}
OLD_BAR = 2e-2                 # max|got - ref| / max|ref|, the bar of the earlier inference tests


# --------------------------------------------------------------------------- references
class InferRound:
    """Where the bf16 inference path stores reduced precision (no rounding at all when `on` is False)."""

    def __init__(self, on):
        self.on = on

    def r(self, t):
        return t.to(torch.bfloat16).to(t.dtype) if self.on else t


EXACT = InferRound(False)


def _layer(params, name, i):
    return params[f"{name}_fcnet/linear_{i}/w"], params[f"{name}_fcnet/linear_{i}/b"]


def mlp_abs(params, name, h, s, n_layers, q):
    """(output, absolute-network scale) of an MLP on input h whose entries are known to within relative error ~ s / |h|."""
    for i in range(n_layers):
        w, b = _layer(params, name, i)
        h = h @ q.r(w) + b
        s = s @ w.abs() + b.abs()
        if i != n_layers - 1:
            h = q.r(torch.relu(h))
    return h, s


def _normal(spec, out, s, dt):
    Z = spec.latent_size
    c = spec.raw_sigma_bias
    mu, raw = out[:, :Z], out[:, Z:]
    return {"mu": ("lin", mu, s[:, :Z]), "sigma": ("sigma", O.softplus(raw + c), s[:, Z:] + abs(c))}


def reference(spec, params, x, eps, u, z, y, q=EXACT, dt=torch.float64):
    """Every output of the inference entry points on rows x (encode: with noise eps, u) and on inputs z (decode,
    condition(DECODER)) and y (condition(ENCODER), condition(PRIOR_GMM)): name -> (kind, value, scale[, ...])."""
    dev = x.device
    p = {k: v.to(dev, dt) for k, v in params.items()}
    x, eps = x.to(dt), eps.to(dt)
    L = len(spec.hidden_sizes) + 1
    T = float(torch.tensor(spec.temperature, dtype=torch.float32))
    gm = spec.model == "gmvae"
    out = {}
    xa = x.abs()
    # encode
    if gm:
        ly, sly = mlp_abs(p, "encoder_y", x, xa, L, q)
        g = -torch.log(-torch.log(u.to(dt)))
        ys = torch.softmax((ly + g) / T, -1)
        # y carries the relative error 2 max_k |d logit_k| / T of the softmax: scale its absolute-network input accordingly
        sy = ys * (1 + 2 * sly.max(1, keepdim=True).values / T)
        eo, so = mlp_abs(p, "encoder_gmm", torch.cat([x, q.r(ys)], 1), torch.cat([xa, sy], 1), L, q)
        out["encode.logits_y"] = ("lin", ly, sly)
        out["encode.y"] = ("lin", ys, sy)                                # not an engine output: the sample case_inputs reuses
    else:
        eo, so = mlp_abs(p, "encoder", x, xa, L, q)
    nrm = _normal(spec, eo, so, dt)
    out["encode.z_mean"] = nrm["mu"]
    out["encode.z_sample"] = ("z", nrm["mu"][1], nrm["mu"][2], nrm["sigma"][1], nrm["sigma"][2], eps, spec.sigma_min)
    if z is None:
        return out
    # decode / condition(DECODER)
    zq = q.r(z.to(dt))
    lx, slx = mlp_abs(p, "decoder", zq, zq.abs(), L, q)
    gb = spec.gen_bias_init
    out["decode"] = ("prob", torch.sigmoid(lx + gb), slx + abs(gb))
    out["condition.decoder"] = ("lin", lx + gb, slx + abs(gb))
    # condition(ENCODER) and the GMVAE's other two
    if gm:
        yq = q.r(y.to(dt))
        eo, so = mlp_abs(p, "encoder_gmm", torch.cat([x, yq], 1), torch.cat([xa, yq.abs()], 1), L, q)
        for k, v in _normal(spec, eo, so, dt).items():
            out["condition.encoder." + k] = v
        out["condition.encoder_y"] = out["encode.logits_y"]
        po, sp = mlp_abs(p, "prior_gmm", yq, yq.abs(), 1, q)
        for k, v in _normal(spec, po, sp, dt).items():
            out["condition.prior_gmm." + k] = v
    else:
        for k, v in _normal(spec, eo, so, dt).items():
            out["condition.encoder." + k] = v
    return out


def prior_reference(spec, params):
    """gmvae_prior_table: (mu, sigma) of the K prior components from the fp32 parameters."""
    K, Z = spec.K, spec.latent_size
    p = {k: v.double() for k, v in params.items()}
    if spec.model == "gmvae":
        w, b = _layer(p, "prior_gmm", 0)
        out = _normal(spec, w + b, w.abs() + b.abs(), torch.float64)
        return {"prior.mu": out["mu"], "prior.sigma": out["sigma"]}
    if spec.model == "vae_gmp":                 # (loc, softplus(raw_scale_diag)): neither sigma_min nor raw_sigma_bias applies
        return {"prior.mu": ("lin", p["loc"], p["loc"].abs()),
                "prior.sigma": ("sigma", O.softplus(p["raw_scale_diag"]), p["raw_scale_diag"].abs(), 0.0)}
    one = torch.ones(1, Z, dtype=torch.float64)
    return {"prior.mu": ("lin", 0 * one, one), "prior.sigma": ("sigma", one, one, 0.0)}


# --------------------------------------------------------------------------- comparisons
def _f64(t, like):
    return torch.as_tensor(t).to(like.device, torch.float64)


def figure(rec, got, tol, sigma_min=0.0):
    """Worst (|d| - floor) / scale of `got` against the reference record `rec` (<= tol passes); +inf where an entry held at
    sigma_min is not sigma_min exactly, or got is not finite."""
    kind, ref = rec[0], rec[1]
    got = _f64(got, ref)
    if not bool(torch.isfinite(got).all()):
        return math.inf
    if kind == "lin":
        return ((got - ref).abs() / rec[2].clamp_min(1e-300)).max().item()
    if kind == "prob":
        pq = (ref * (1 - ref)) * rec[2]
        return (((got - ref).abs() - (2 ** -23 * ref + 2 ** -126)).clamp_min(0) / pq.clamp_min(1e-300)).max().item()
    if kind == "sigma":
        t, s = ref, rec[2]
        smin = rec[3] if len(rec) > 3 else sigma_min
        want = t.clamp_min(smin)
        if bool((got <= 0).any()):
            return math.inf
        f = (((got.log() - want.log()).abs() - 2 ** -22).clamp_min(0) / s).max().item()
        if smin > 0:
            held = t.log() < math.log(smin) - tol * s                # clamped, and off the kink by more than the tolerance
            if bool((got[held] != float(torch.tensor(smin, dtype=torch.float32))).any()):
                return math.inf
        return f
    if kind == "z":
        _, mu, smu, t, sraw, eps, smin = rec
        sig = t.clamp_min(smin)
        se = sig * eps.abs()
        ref = mu + sig * eps
        return (((got - ref).abs() - 2 ** -22 * (mu.abs() + se)).clamp_min(0) / (smu + se * sraw)).max().item()
    raise ValueError(kind)


def old_bar(rec, got):
    ref = rec[1] if rec[0] != "z" else rec[1] + rec[3].clamp_min(rec[6]) * rec[5]
    if rec[0] == "sigma":
        ref = ref.clamp_min(rec[3] if len(rec) > 3 else 0.0)
    got = _f64(got, ref)
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def value(rec, sigma_min=0.0):
    """The reference value of a record, as the engine returns it."""
    if rec[0] == "z":
        return rec[1] + rec[3].clamp_min(rec[6]) * rec[5]
    if rec[0] == "sigma":
        return rec[1].clamp_min(rec[3] if len(rec) > 3 else sigma_min)
    return rec[1]


def sliced(rec, n):
    return tuple(t[:n] if torch.is_tensor(t) and t.dim() == 2 else t for t in rec)


# --------------------------------------------------------------------------- engine side
def infer_outputs(eng, x, eps, u, z, y):
    """The engine's outputs under the names of `reference`."""
    n, D, Z, K = x.shape[0], eng.data_size, eng.latent_size, eng.mixture_components
    gm = eng.model == "gmvae"
    ly, zm, zs = eng.encode(x, eps=eps, gumbel_u=u if gm else None)
    out = {"encode.z_mean": zm, "encode.z_sample": zs, "decode": eng.decode(z),
           "condition.decoder": _condition(eng, COND_DECODER, z, None, n, D)[0]}
    if gm:
        out["encode.logits_y"] = ly
        out["condition.encoder.mu"], out["condition.encoder.sigma"] = _condition(eng, COND_ENCODER, x.float(), y, n, Z, Z)
        out["condition.encoder_y"] = _condition(eng, COND_ENCODER_Y, x.float(), None, n, K)[0]
        out["condition.prior_gmm.mu"], out["condition.prior_gmm.sigma"] = _condition(eng, COND_PRIOR_GMM, y, None, n, Z, Z)
    else:
        out["condition.encoder.mu"], out["condition.encoder.sigma"] = _condition(eng, COND_ENCODER, x.float(), None, n, Z, Z)
    mu, sg = eng.prior_table()
    out["prior.mu"], out["prior.sigma"] = mu, sg
    torch.cuda.synchronize()
    return {k: v.clone() for k, v in out.items()}


def case_inputs(spec, params, x, eps, u, dev="cpu"):
    """z and y for decode / condition: the exact oracle's own encode samples on these rows, so that a trained-like decoder sees
    the codes it saturates on and prior_gmm the peaked y of q(y|x)."""
    ref = reference(spec, params, x.to(dev), eps.to(dev), None if u is None else u.to(dev), None, None)
    return value(ref["encode.z_sample"]).float(), (ref["encode.y"][1].float() if "encode.y" in ref else None)


def _prior_spec_fix(spec, params):
    return prior_reference(spec, {k: v.float() for k, v in params.items()})


def _tol(key, which, precision):
    if key.startswith("prior."):                 # computed from the fp32 parameters in both modes
        return TOL["fp32"]
    return TOL["bf16_exact"] if (precision == "bf16" and which == "exact") else TOL[precision]


def compare(name, precision, spec, params, x, eps, u, eng=None, rows=None, max_batch=None, tag=""):
    """Runs one case; returns the worst figures per output and asserts the bounds."""
    dev = "cuda"
    z, y = case_inputs(spec, params, x, eps, u, dev)
    bf16 = precision == "bf16"
    exact = reference(spec, params, x.to(dev), eps.to(dev), None if u is None else u.to(dev), z, y)
    model = reference(spec, params, x.to(dev), eps.to(dev), None if u is None else u.to(dev), z, y, InferRound(True)) if bf16 else exact
    prior = _prior_spec_fix(spec, params)
    own = eng is None
    if own:
        cfg = dict(model=spec.model, latent_size=spec.latent_size, hidden_sizes=spec.hidden_sizes,
                   mixture_components=spec.mixture_components, data_size=spec.data_size, batch=x.shape[0],
                   sigma_min=spec.sigma_min, raw_sigma_bias=spec.raw_sigma_bias, gen_bias_init=spec.gen_bias_init,
                   temperature=spec.temperature)
        eng = make_engine(cfg, precision, max_batch=max_batch)
        eng.set_parameters(params)
    worst = {}
    for n in rows or [x.shape[0]]:
        got = infer_outputs(eng, x[:n], eps[:n], None if u is None else u[:n], z[:n], None if y is None else y[:n])
        for k, g in got.items():
            if k.startswith("prior."):
                recs = {"model": prior[k]}
            else:
                recs = {"model": sliced(model[k], n), "exact": sliced(exact[k], n)}
            for which, rec in recs.items():
                tol = _tol(k, which, precision)
                f = figure(rec, g, tol, spec.sigma_min)
                key = f"{k}/{which}"
                if f > worst.get(key, (-1.0, 0))[0]:
                    worst[key] = (f, n)
    if own:
        eng.close()
    _record(name, {"test": "infer", "tag": tag, "precision": precision, "figures": {k: v[0] for k, v in worst.items()},
                   "at_rows": {k: v[1] for k, v in worst.items()}})
    bad = {}
    for key, (f, n) in worst.items():
        which = key.rsplit("/", 1)[1]
        tol = _tol(key, which, precision)
        if not f <= tol:
            bad[key] = (f, tol, n)
    assert not bad, (name, precision, tag, bad)
    return worst


# --------------------------------------------------------------------------- (a) the shape catalogue
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_catalogue(name, precision):
    cfg = CONFIGS[name]
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    compare(name, precision, spec, params, x, eps, u)


# --------------------------------------------------------------------------- (b) row counts of a training batch
ROWS = [1, 127, 128, 129, 4095, 4096, 4097, 16384]
BIG = {"gmvae": FULL, "vae": dict(FULL, model="vae", mixture_components=1), "vae_gmp": dict(FULL, model="vae_gmp")}


def crossing_rows(widths):
    """Row counts at which a layer's tile count reaches the SM count and passes it (128-row m-tiles, 256-wide n-tiles)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    out = []
    for w in widths:
        nt = -(-w // 256)
        m = sms // nt
        out += [128 * m, 128 * m + 1]
    return out


def _big_case(model, n, regime=None):
    cfg = BIG[model]
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    if regime:
        params = regimes.build(regime, spec, params)
    x, eps, u = _full_inputs(n)
    return cfg, spec, params, x.bool(), eps, (u if model == "gmvae" else None)


@pytest.mark.parametrize("model", list(BIG))
def test_row_counts(model):
    """bf16 at every row count (the oracle once at 16 384 rows, sliced), then fp32 at 16 384; handles of max_batch 16 384."""
    rows = sorted(set(ROWS + crossing_rows([784, 512])))
    cfg, spec, params, x, eps, u = _big_case(model, 16384)
    t0 = time.perf_counter()
    compare(f"cfg4_{model}", "bf16", spec, params, x, eps, u, rows=rows, max_batch=16384, tag="rows")
    compare(f"cfg4_{model}", "fp32", spec, params, x, eps, u, max_batch=16384, tag="rows")
    _record(f"cfg4_{model}", {"test": "infer_rows", "rows": rows, "seconds": time.perf_counter() - t0})


# --------------------------------------------------------------------------- (c) trained-model values
TRAINED = [(n, r) for n in ("cfg1", "cfg2", "cfg3", "k20_ragged")
           for r in ("scales:1e-08", "saturated_decoder", "peaked_y", "trained_like")
           if r != "peaked_y" or CONFIGS[n]["model"] == "gmvae"]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name,regime", TRAINED, ids=[f"{n}-{r}" for n, r in TRAINED])
def test_trained_regime(name, regime, precision):
    cfg = CONFIGS[name]
    spec = make_spec(cfg)
    params = regimes.build(regime, spec, perturbed_params(spec))
    x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    compare(name, precision, spec, params, x, eps, u, tag=regime)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_trained_regime_cfg4(precision):
    cfg, spec, params, x, eps, u = _big_case("gmvae", 16384, "trained_like")
    compare("cfg4", precision, spec, params, x, eps, u, max_batch=16384, tag="trained_like")


# --------------------------------------------------------------------------- (d) state left by training
STATE = ["h33_7", "z3_gmvae", "k33_gmvae", "d97", "nohidden_gmvae", "cfg4_B4097"]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", STATE)
def test_inference_after_training(name, precision):
    """3 training steps and one replay of a captured step, then every entry point equals, bit for bit, a fresh handle given the
    same parameters: the chained step writes the buffers (padding columns included) that inference then contracts over."""
    if name == "cfg4_B4097":
        cfg, spec, params, x, eps, u = _big_case("gmvae", 4097)
        cfg = dict(cfg, batch=4097)
    else:
        cfg = CONFIGS[name]
        spec = make_spec(cfg)
        params = perturbed_params(spec)
        x, _, eps, u = O.synthetic_batch(spec, cfg["batch"])
    trained = make_engine(cfg, precision)
    trained.set_parameters(params)
    xs = x.to(torch.uint8).cuda(); e_d, u_d = eps.cuda(), u.cuda()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(3):
            trained.train_step(xs, eps=e_d, gumbel_u=u_d)
        trained.capture_step(xs, eps=e_d, gumbel_u=u_d)
        trained.replay()
    side.synchronize()
    assert trained.global_step == 4
    fresh = make_engine(cfg, precision)
    fresh.set_parameters({k: v.detach().clone() for k, v in trained.parameters().items()})
    z, y = case_inputs(spec, params, x, eps, u)
    a = infer_outputs(trained, x, eps, u, z, y)
    b = infer_outputs(fresh, x, eps, u, z, y)
    for k in a:
        assert torch.isfinite(a[k]).all(), (name, k)
        assert torch.equal(a[k], b[k]), (name, precision, k, (a[k] - b[k]).abs().max().item())
    trained.close(); fresh.close()


# --------------------------------------------------------------------------- (e) distribution kernels
def _lib_stream():
    return _lib.load(), torch.cuda.current_stream().cuda_stream


def _dev(t):
    return t.to("cuda", torch.float32).contiguous()


# Bounds in units of the condition of each formula (see each test), at least twice the worst figure measured on one B200
# (power limit 1000 W): normal log_prob 3.9e-7 (d = 33, n = 100 003); Bernoulli log_prob 1.4e-7 (d = 97) and mean 2.3e-7 (d = 784); relaxed
# sample 1.4e-7 (K = 32, T = 2).
DIST_TOL = {"normal_log_prob": 1e-6, "bernoulli_log_prob": 3e-7, "bernoulli_mean": 5e-7, "relaxed_sample": 3e-7}


@pytest.mark.parametrize("n", [1, 7, 8, 9, 100003])
@pytest.mark.parametrize("d", [1, 31, 32, 33, 260, 784])
def test_dist_normal_log_prob(d, n):
    """log N(z; mu, diag sigma^2) per row; |d| <= tol * sum_j (|t_j^2 / 2| + |log sigma_j| + log(2 pi) / 2), scales from 1e-8 to
    10 and z up to 1e4 standard deviations from mu."""
    g = torch.Generator().manual_seed(d * 100 + n)
    mu = 3 * torch.randn(n, d, generator=g)
    sig = 10 ** (torch.rand(n, d, generator=g) * 9 - 8)
    far = 10 ** (torch.rand(n, d, generator=g) * 5 - 1)
    z = (mu.double() + sig.double() * torch.randn(n, d, generator=g, dtype=torch.float64) * far).float()
    lib, st = _lib_stream()
    m_d, s_d, z_d = _dev(mu), _dev(sig), _dev(z)
    out = torch.empty(n, device="cuda")
    _lib.check(lib.gmvae_dist_normal_log_prob(m_d.data_ptr(), s_d.data_ptr(), z_d.data_ptr(), n, d, out.data_ptr(), st))
    t = (z_d.double() - m_d.double()) / s_d.double()
    half_t2, log_s = 0.5 * t * t, s_d.double().log()
    ref = (-half_t2 - log_s - 0.5 * O.LOG_2PI).sum(1)
    scale = (half_t2 + log_s.abs() + 0.5 * O.LOG_2PI).sum(1)
    f = ((out.double() - ref).abs() / scale).max().item()
    _record("dist", {"test": "normal_log_prob", "d": d, "n": n, "figure": f})
    assert f <= DIST_TOL["normal_log_prob"], (d, n, f)


def _bernoulli_inputs(n, d, seed):
    """Logits up to |100|: half the rows uniform in [-100, 100] with random x, half well predicted (x = [l > 0], |l| in
    [10, 100]) where every term is a small -log1p(exp(-|l|))."""
    g = torch.Generator().manual_seed(seed)
    lg = (torch.rand(n, d, generator=g) * 2 - 1) * 100
    x = (torch.rand(n, d, generator=g) < 0.5).float()
    h = n // 2
    mag = 10 + 90 * torch.rand(h, d, generator=g) ** 3
    sign = torch.where(torch.rand(h, d, generator=g) < 0.5, -1.0, 1.0)
    lg[h:] = sign * mag
    x[h:] = (sign > 0).float()
    return lg, x


@pytest.mark.parametrize("d", [97, 784])
def test_dist_bernoulli(d):
    """Bernoulli log_prob (|d| <= tol * sum_j |x l - max(l, 0) - log1p(exp(-|l|))|: all terms are <= 0, so this is the relative
    error of the row) and mean (element-wise relative, absolute floor 2^-126)."""
    n = 1000
    lg, x = _bernoulli_inputs(n, d, d)
    lib, st = _lib_stream()
    l_d, x_d = _dev(lg), _dev(x)
    out = torch.empty(n, device="cuda")
    _lib.check(lib.gmvae_dist_bernoulli_log_prob(l_d.data_ptr(), x_d.data_ptr(), n, d, out.data_ptr(), st))
    mean = torch.empty(n, d, device="cuda")
    _lib.check(lib.gmvae_dist_bernoulli_mean(l_d.data_ptr(), n * d, mean.data_ptr(), st))
    l64 = l_d.double()
    terms = x_d.double() * l64 - l64.clamp_min(0) - torch.log1p(torch.exp(-l64.abs()))
    f_lp = ((out.double() - terms.sum(1)).abs() / terms.abs().sum(1)).max().item()
    p = torch.sigmoid(l64)
    f_mean = (((mean.double() - p).abs() - 2 ** -126).clamp_min(0) / p).max().item()
    _record("dist", {"test": "bernoulli", "d": d, "log_prob": f_lp, "mean": f_mean})
    assert f_lp <= DIST_TOL["bernoulli_log_prob"], (d, f_lp)
    assert f_mean <= DIST_TOL["bernoulli_mean"], (d, f_mean)


@pytest.mark.parametrize("T", [0.1, 0.5, 1.0, 2.0])
@pytest.mark.parametrize("K", [1, 2, 31, 32, 33, 128])
def test_dist_relaxed_sample(K, T):
    """softmax((l + g) / T), g = -log(-log u), with u at the smallest positive float and at 1 - 2^-24 and logits spread over
    +-50; element-wise |d| <= tol * y * (1 + max_k |(l_k + g_k) / T|) + 2^-126 (the softmax's own condition in fp32)."""
    n = 64
    g = torch.Generator().manual_seed(K * 10 + int(T * 10))
    lg = (torch.rand(n, K, generator=g) * 2 - 1) * 50
    u = torch.rand(n, K, generator=g).clamp_min(torch.finfo(torch.float32).tiny)
    u[0::3, 0] = 2.0 ** -149
    u[1::3, -1] = 1 - 2.0 ** -24
    u[2::5] = 2.0 ** -149
    u[3::5] = 1 - 2.0 ** -24
    lib, st = _lib_stream()
    l_d, u_d = _dev(lg), _dev(u)
    out = torch.empty(n, K, device="cuda")
    _lib.check(lib.gmvae_dist_relaxed_sample(l_d.data_ptr(), u_d.data_ptr(), n, K, float(T), out.data_ptr(), st))
    T32 = float(torch.tensor(T, dtype=torch.float32))
    arg = (l_d.double() - torch.log(-torch.log(u_d.double()))) / T32
    y = torch.softmax(arg, 1)
    cond = 1 + arg.abs().max(1, keepdim=True).values
    f = (((out.double() - y).abs() - 2 ** -126).clamp_min(0) / (y * cond).clamp_min(1e-300)).max().item()
    _record("dist", {"test": "relaxed_sample", "K": K, "T": T, "figure": f})
    assert torch.isfinite(out).all()
    assert f <= DIST_TOL["relaxed_sample"], (K, T, f)


# --------------------------------------------------------------------------- (f) prior_table
def prior_case(model, K, Z):
    """A small model with raw_sigma_bias = -0.3 and a sigma_min that holds about half of the GMVAE's component scales (the
    midpoint of the widest gap between consecutive scales around the median, so none is on the kink)."""
    cfg = dict(model=model, latent_size=Z, hidden_sizes=[16], mixture_components=K if model != "vae" else 1, batch=4,
               data_size=32, raw_sigma_bias=-0.3)
    spec = make_spec(dict(cfg, sigma_min=0.0))
    params = perturbed_params(spec, bias_scale=0.5)
    if model == "gmvae":
        s = prior_reference(spec, {k: v.float() for k, v in params.items()})["prior.sigma"][1].reshape(-1).sort().values
    else:
        s = O.softplus(params["raw_scale_diag"]).reshape(-1).sort().values if model == "vae_gmp" else torch.ones(1, dtype=torch.float64)
    if s.numel() < 4:
        thr = 2 * s.max().item()
    else:
        lo, hi = int(0.3 * s.numel()), int(0.7 * s.numel())
        i = lo + int((s[lo + 1:hi + 1] - s[lo:hi]).argmax())
        thr = 0.5 * (s[i] + s[i + 1]).item()
    cfg["sigma_min"] = float(torch.tensor(thr, dtype=torch.float32))
    return cfg, make_spec(cfg), params


PRIOR_CASES = [(m, K, Z) for m in ("vae", "vae_gmp", "gmvae") for K, Z in ((1, 1), (128, 260), (1, 260), (128, 1))
               if m != "vae" or K == 1]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("model,K,Z", PRIOR_CASES, ids=[f"{m}-K{K}-Z{Z}" for m, K, Z in PRIOR_CASES])
def test_prior_table(model, K, Z, precision):
    cfg, spec, params = prior_case(model, K, Z)
    eng = make_engine(cfg, precision)
    eng.set_parameters(params)
    mu, sg = eng.prior_table()
    torch.cuda.synchronize()
    ref = prior_reference(spec, {k: v.float() for k, v in params.items()})
    figs = {"mu": figure(ref["prior.mu"], mu, TOL["fp32"]), "sigma": figure(ref["prior.sigma"], sg, TOL["fp32"], spec.sigma_min)}
    if model == "gmvae":
        held = ref["prior.sigma"][1] < spec.sigma_min
        figs["held_share"] = held.double().mean().item()
        assert 0 < figs["held_share"] <= 1 or K * Z == 1
    _record(f"prior_{model}_K{K}_Z{Z}", {"test": "prior_table", "precision": precision, "figures": figs})
    assert figs["mu"] <= TOL["fp32"] and figs["sigma"] <= TOL["fp32"], figs
    eng.close()


# --------------------------------------------------------------------------- (g) Engine.encode past max_batch
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["cfg1", "cfg3"])
def test_encode_slices_rows(name, precision):
    """203 rows on a handle of max_batch 100: Engine.encode equals three calls on rows 0-99, 100-199 and 200-202, bit for bit."""
    cfg = CONFIGS[name]
    spec = make_spec(cfg)
    params = perturbed_params(spec)
    x, _, eps, u = O.synthetic_batch(spec, 203)
    eng = make_engine(cfg, precision, max_batch=100)
    eng.set_parameters(params)
    whole = [t.clone() if t is not None else None for t in eng.encode(x, eps=eps, gumbel_u=u)]
    parts = [eng.encode(x[a:b], eps=eps[a:b], gumbel_u=None if u is None else u[a:b]) for a, b in ((0, 100), (100, 200), (200, 203))]
    torch.cuda.synchronize()
    for i, w in enumerate(whole):
        if w is None:
            assert all(p[i] is None for p in parts)
            continue
        assert torch.equal(w, torch.cat([p[i] for p in parts])), (name, precision, i)
    eng.close()
