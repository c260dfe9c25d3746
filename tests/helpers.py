"""Shared helpers of the GPU parity tests: build an Engine and an oracle Spec from one
description, copy oracle weights into the engine, compare loss terms and gradients."""
import torch

from oracle import gmvae_oracle as O

CONFIGS = {
    # BASELINE.json configs[0..2] (cfg1-3): H=512x2, Z=64, B=100
    "cfg1": dict(model="vae", latent_size=64, hidden_sizes=[512, 512], mixture_components=1, batch=100),
    "cfg2": dict(model="vae_gmp", latent_size=64, hidden_sizes=[512, 512], mixture_components=10, batch=100),
    "cfg3": dict(model="gmvae", latent_size=64, hidden_sizes=[512, 512], mixture_components=10, batch=100),
    # small / ragged shapes: nothing is a multiple of a tile
    "tiny_gmvae": dict(model="gmvae", latent_size=24, hidden_sizes=[72, 40], mixture_components=7, batch=37, data_size=200),
    "tiny_vae": dict(model="vae", latent_size=10, hidden_sizes=[48], mixture_components=1, batch=5, data_size=120),
    "tiny_gmp": dict(model="vae_gmp", latent_size=12, hidden_sizes=[40, 56], mixture_components=5, batch=33, data_size=136),
    "nohidden_gmvae": dict(model="gmvae", latent_size=16, hidden_sizes=[], mixture_components=4, batch=19, data_size=64),
    # the run_train.sh example shape (bin/run_train.sh:5-11): z=128, h=512 x 1, batch 64
    "run_train_sh": dict(model="gmvae", latent_size=128, hidden_sizes=[512], mixture_components=10, batch=64),
    # BASELINE.json configs[4] (cfg5) at a batch the oracle finishes in seconds: K=50 > 16 leaves the fused y head
    # (engine.cu forward_encoder / head_y_*_kernel), Z=128 > 64 leaves the z row job of the chained kernel
    "cfg5_small": dict(model="gmvae", latent_size=128, hidden_sizes=[1024, 1024], mixture_components=50, batch=200),
    # 16 < K <= 32, nothing a multiple of a tile, more than one 128-row block
    "k20_ragged": dict(model="gmvae", latent_size=40, hidden_sizes=[96, 72], mixture_components=20, batch=150, data_size=200),
    "k17_gmp": dict(model="vae_gmp", latent_size=20, hidden_sizes=[64], mixture_components=17, batch=130, data_size=96),
    # the dispatch boundaries of the heads (engine.cu forward_encoder / the z head) and padded row strides
    # K = 1: a one-way softmax (y = 1, zero entropy, exactly zero encoder_y gradients)
    "k1_gmvae": dict(model="gmvae", latent_size=16, hidden_sizes=[64], mixture_components=1, batch=40, data_size=120),
    # K = 16: the largest y head fused into the GEMM epilogue (Kp = 16, the second uint4 store)
    "k16_gmvae": dict(model="gmvae", latent_size=24, hidden_sizes=[64, 48], mixture_components=16, batch=100, data_size=200),
    # K = 32 / 33: the last lane slot of the warp head that is full / the first one past it
    "k32_gmvae": dict(model="gmvae", latent_size=16, hidden_sizes=[80], mixture_components=32, batch=90, data_size=144),
    "k33_gmvae": dict(model="gmvae", latent_size=16, hidden_sizes=[80], mixture_components=33, batch=90, data_size=144),
    # K = 128 = HEAD_MAXK; VAE_GMP with a small Z: gmp_prior_kernel's shared-memory table
    "k128_gmvae": dict(model="gmvae", latent_size=32, hidden_sizes=[96], mixture_components=128, batch=150, data_size=200),
    "k128_gmp": dict(model="vae_gmp", latent_size=4, hidden_sizes=[64], mixture_components=128, batch=100, data_size=120),
    # Z = 1, 3: the _cs z head with Zp = 8
    "z1_vae": dict(model="vae", latent_size=1, hidden_sizes=[48], mixture_components=1, batch=60, data_size=112),
    "z3_gmvae": dict(model="gmvae", latent_size=3, hidden_sizes=[40], mixture_components=5, batch=70, data_size=96),
    # Z = 65: odd width past 64 (generic forward head, _cs backward with 3 rows per block)
    "z65_gmp": dict(model="vae_gmp", latent_size=65, hidden_sizes=[64], mixture_components=6, batch=80, data_size=128),
    # Z = 256: the largest v4 / _cs head; Z = 260: the generic z head with the bias gradient left unfused
    "z256_gmvae": dict(model="gmvae", latent_size=256, hidden_sizes=[128], mixture_components=4, batch=60, data_size=160),
    "z260_gmvae": dict(model="gmvae", latent_size=260, hidden_sizes=[96], mixture_components=3, batch=40, data_size=120),
    "z260_vae": dict(model="vae", latent_size=260, hidden_sizes=[128], mixture_components=1, batch=50, data_size=104),
    # hidden widths that are not multiples of 8: padded row strides that the tensor-core GEMMs contract over
    "h33_7": dict(model="gmvae", latent_size=12, hidden_sizes=[33, 7], mixture_components=6, batch=64, data_size=120),
    "h129_gmp": dict(model="vae_gmp", latent_size=20, hidden_sizes=[129], mixture_components=5, batch=50, data_size=152),
    # odd image rows: the byte path of the BCE x load
    "d97": dict(model="gmvae", latent_size=10, hidden_sizes=[40], mixture_components=5, batch=80, data_size=97),
    # objective M shapes (its layer 0 must be a multiple of 4 wide), also run under objective R
    "m_h36_20_k33": dict(model="gmvae", latent_size=12, hidden_sizes=[36, 20], mixture_components=33, batch=20, data_size=100),
    "m_k128_z8": dict(model="gmvae", latent_size=8, hidden_sizes=[32], mixture_components=128, batch=10, data_size=64),
}


# Model hyperparameters a cfg dict may set; absent ones take the defaults of runners.create_model (the oracle's Spec and Engine
# share them: sigma_min 0, raw_sigma_bias 0.5, gen_bias_init 0, temperature 1).
KNOBS = ("sigma_min", "raw_sigma_bias", "gen_bias_init", "temperature")


def make_spec(cfg):
    return O.Spec(model=cfg["model"], data_size=cfg.get("data_size", 784), latent_size=cfg["latent_size"],
                  hidden_sizes=list(cfg["hidden_sizes"]), mixture_components=cfg["mixture_components"],
                  **{k: cfg[k] for k in KNOBS if k in cfg})


def make_engine(cfg, precision, max_batch=None, objective="reference", **kw):
    import gmvae_b200
    return gmvae_b200.Engine(model=cfg["model"], data_size=cfg.get("data_size", 784), latent_size=cfg["latent_size"],
                             hidden_sizes=cfg["hidden_sizes"], mixture_components=cfg["mixture_components"],
                             precision=precision, objective=objective, max_batch=max_batch or cfg["batch"], init=False,
                             **{k: cfg[k] for k in KNOBS if k in cfg}, **kw)


def perturbed_params(spec, seed=2024, bias_scale=0.05):
    """Xavier weights plus small non-zero biases so that every bias-gradient path is exercised."""
    p = O.init_params(spec, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    for n in p:
        if n.endswith("/b"):
            p[n] = bias_scale * torch.randn(p[n].shape, generator=g, dtype=torch.float64)
    return p


def rel(a, b):
    return abs(a - b) / max(abs(b), 1e-30)


def grad_errors(engine, grads_ref):
    """||g - g*||_2 / ||g*||_2 per tensor (SURVEY.md §8(d))."""
    out = {}
    for name, g in engine.gradients().items():
        r = grads_ref[name].to(torch.float64)
        d = g.detach().cpu().to(torch.float64).reshape(r.shape)
        out[name] = ((d - r).norm() / r.norm().clamp_min(1e-30)).item()
    return out


def run_parity(cfg, precision, seed=2024, rounding_model=None, objective="reference", want_ref=False):
    """Returns (loss-term errors, per-tensor gradient errors) of the CUDA step against the oracle.
    With `rounding_model` the oracle restates the bf16 storage points of the CUDA path."""
    spec = make_spec(cfg)
    params = perturbed_params(spec, seed)
    x, labels, eps, u = O.synthetic_batch(spec, cfg["batch"], objective=objective)
    terms_ref, grads_ref = O.loss_and_grads(spec, params, x, eps, u, objective=objective, q=rounding_model or O.EXACT)
    eng = make_engine(cfg, precision, objective=objective)
    eng.set_parameters(params)
    loss = eng.forward_backward(x, eps=eps, gumbel_u=u)
    torch.cuda.synchronize()
    t = loss.detach().cpu().tolist()
    terr = term_errors(t, terms_ref, spec)
    gerr = grad_errors(eng, grads_ref)
    eng.close()
    if want_ref:
        return terr, gerr, {k: terms_ref[k].item() for k in ("loss", "nll", "kl_div_z", "nent")}
    return terr, gerr


def term_errors(t, terms_ref, spec):
    """Relative error of [loss, nll, kl_div_z, nent] against the oracle's terms.  All four are TRUE relative errors
    |t - ref| / |ref|.  (nent of the VAE models is identically 0 on both sides: error 0.)"""
    out = {}
    for i, k in enumerate(("loss", "nll", "kl_div_z", "nent")):
        ref = terms_ref[k].item() if hasattr(terms_ref[k], "item") else float(terms_ref[k])
        out[k] = 0.0 if (ref == 0.0 and t[i] == 0.0) else abs(t[i] - ref) / max(abs(ref), 1e-30)
    return out


KL_ABS_FLOOR = 1.0   # nats


def bf16_term_ok(terr, terms_ref, tol=2e-3):
    """The bf16 bar on the loss terms, stated explicitly: loss, nll and nent within TRUE relative `tol` of the exact fp64
    oracle; kl_div_z within `tol` * max(|kl_div_z|, 1 nat).  kl_div_z = mean_b[log q(z) - log p(z)] is a difference of two
    log-densities of ~Z nats each and is 0.1-0.5 nats at fresh weights, so below 1 nat the bar is ABSOLUTE (2e-3 nats,
    i.e. 4e-6 of the loss it is a summand of); the true relative error is what `terr` holds and what the tests report."""
    bad = {}
    for k, v in terr.items():
        ref = abs(float(terms_ref[k]))
        lim = tol * max(ref, KL_ABS_FLOOR) / max(ref, 1e-30) if k == "kl_div_z" else tol
        if v >= lim:
            bad[k] = (v, lim)
    return bad


# --------------------------------------------------------------------------- bf16 rounding model
class _RoundBoth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, t):
        return t.to(torch.bfloat16).to(t.dtype)

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).to(g.dtype)


class _RoundFwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, t):
        return t.to(torch.bfloat16).to(t.dtype)

    @staticmethod
    def backward(ctx, g):
        return g


class _RoundGrad(torch.autograd.Function):
    @staticmethod
    def forward(ctx, t):
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).to(g.dtype)


class Bf16Model(O.Exact):
    """Where the bf16 CUDA path stores reduced precision (DESIGN.md "Precision"): hidden
    activations and their gradients, z as the decoder's input, y as a GEMM operand, the gradients
    w.r.t. the decoder logits, the encoders' outputs and the prior's output, and -- when the
    tensor-core path is on -- the weight operand of every GEMM (engine.cu lin_fwd / lin_dgrad)."""

    def __init__(self, tensor_core_weights=True):
        self.tcw = tensor_core_weights

    def act(self, t):
        return _RoundBoth.apply(t)

    def fwd(self, t):
        return _RoundFwd.apply(t)

    def grad(self, t):
        return _RoundGrad.apply(t)

    def weight(self, name, w):
        return _RoundFwd.apply(w) if self.tcw else w

    def yin(self, t):            # y is the bf16 operand of the second K segment (tensor-core path)
        return _RoundFwd.apply(t) if self.tcw else t


# --------------------------------------------------------------------------- sigma_min cases
def active_clamp(cfg, params, x, eps, u=None, objective="reference"):
    """`cfg` with raw_sigma_bias = 0 and a sigma_min that clamps about half of the scales: the midpoint of the widest gap between
    consecutive values of softplus(raw) (q(z) and, for the GMVAE, p(z|y) pooled) between their 40th and 60th percentiles, on
    these weights and inputs, rounded to fp32 (the type of gmvae_config::sigma_min).  Taking a gap keeps every entry off the
    kink of the clamp."""
    t = O.loss_terms(make_spec(dict(cfg, sigma_min=0.0, raw_sigma_bias=0.0)), params, x, eps, u, objective)
    s = torch.cat([t[k].reshape(-1) for k in ("sigma_q", "sigma_p") if k in t]).sort().values
    lo, hi = int(0.4 * s.numel()), int(0.6 * s.numel())
    i = lo + int((s[lo + 1:hi + 1] - s[lo:hi]).argmax())
    thr = torch.tensor(0.5 * (s[i] + s[i + 1]).item(), dtype=torch.float32).item()
    return dict(cfg, sigma_min=thr, raw_sigma_bias=0.0)


def clamp_stats(cfg, params, x, eps, u=None, objective="reference"):
    """From the oracle's forward pass: the share of the scales of q(z) and p(z|y) that cfg's sigma_min clamps, and how many
    entries of softplus(raw + raw_sigma_bias) lie within 1e-5 (relative) of it."""
    t = O.loss_terms(make_spec(dict(cfg, sigma_min=0.0)), params, x, eps, u, objective)
    thr = float(cfg.get("sigma_min", 0.0))
    out = {"sigma_min": thr, "near_threshold": 0}
    for k in ("sigma_q", "sigma_p"):
        if k in t:
            out[k + "_clamped"] = (t[k] < thr).double().mean().item()
            out["near_threshold"] += int(((t[k] - thr).abs() <= 1e-5 * thr).sum())
    return out
