"""CPU oracle for the GMVAE / VAE / VAE_GMP training step.  TEST INFRASTRUCTURE ONLY.

This file is a CPU restatement (PyTorch, float64 by default) of the arithmetic that the
reference's `run_gmvae.py --mode=train` executes per step.  It is the checker the CUDA
path is compared with; nothing in the product package (`gmvae_b200/`) imports it.  Only
`tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU-baseline / `--impl reference`
legs may import it.

PARITY UNPINNED: the reference itself (TensorFlow 1.13.1 + TFP 0.6.0 + Sonnet v1) cannot
be imported in this image and ships no tests, golden vectors or fixtures (SURVEY.md §4,
§8c).  The oracle is therefore pinned only by (1) closed-form known-answer tests,
(2) an independent re-implementation through `torch.distributions`, and (3) finite
differences of its own autograd graph -- see tests/test_oracle.py.

Reference lines followed (all paths relative to /root/reference/scripts):
  base.py:46-60,114-127,177-190   MLP = chain of linear layers, ReLU between, none at the end
  base.py:63-72                   ConditionalNormal.condition: mu, sigma = max(softplus(raw+bias), min)
  base.py:130-135                 ConditionalBernoulli.condition: logits = MLP(z) + bias_init
  base.py:193-209                 ConditionalCategorical -> RelaxedOneHotCategorical(T, logits)
  base.py:12                      Xavier-uniform weights, zero biases
  gmvae.py:238-267                TrainableGMVAE.run_model (objective "reference")
  gmvae.py:170-173                prior_gmm evaluated at one-hot y (basis of objective "marginal")
  vae.py:167-185, 231-250         TrainableVAE.run_model and the two priors
  utils.py:165-170                entropy(logits, targets)
  runners.py:78-101               hyper-parameters passed by create_model
  runners.py:181-183              tf.train.AdamOptimizer(lr).compute_gradients/apply_gradients
Third-party semantics (TF / TFP / Sonnet are not vendored in the reference) are restated
from their published behaviour, see SURVEY.md Appendix B.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch

LOG_2PI = math.log(2.0 * math.pi)


@dataclass
class Spec:
    """Static description of one model (what runners.create_model passes, runners.py:65-103)."""
    model: str = "gmvae"                 # 'vae' | 'vae_gmp' | 'gmvae'   (run_gmvae.py:14-16)
    data_size: int = 784
    latent_size: int = 64
    hidden_sizes: List[int] = field(default_factory=lambda: [512, 512])
    mixture_components: int = 10
    sigma_min: float = 0.0               # runners.py:84,93,100
    raw_sigma_bias: float = 0.5          # runners.py:85,94,101
    gen_bias_init: float = 0.0           # gmvae.py:284 / vae.py:198 default
    temperature: float = 1.0             # runners.py:86

    @property
    def K(self) -> int:
        return self.mixture_components if self.model != "vae" else 1


def _mlp_shapes(name: str, in_size: int, sizes: List[int]) -> List[Tuple[str, Tuple[int, ...]]]:
    """Sonnet variable names `{name}_fcnet/linear_{i}/{w,b}` (base.py:53,60; Appendix B.1)."""
    out = []
    prev = in_size
    for i, s in enumerate(sizes):
        out.append((f"{name}_fcnet/linear_{i}/w", (prev, s)))
        out.append((f"{name}_fcnet/linear_{i}/b", (s,)))
        prev = s
    return out


def param_shapes(spec: Spec) -> List[Tuple[str, Tuple[int, ...]]]:
    """All trainable variables, in graph-construction order of the reference factories."""
    D, Z, H, K = spec.data_size, spec.latent_size, list(spec.hidden_sizes), spec.mixture_components
    if spec.model == "gmvae":                                   # gmvae.py:321-353
        t = []
        t += _mlp_shapes("prior_gmm", K, [2 * Z])               # hidden_layer_sizes=None -> one linear
        t += _mlp_shapes("decoder", Z, H + [D])
        t += _mlp_shapes("encoder_y", D, H + [K])
        t += _mlp_shapes("encoder_gmm", D + K, H + [2 * Z])
        return t
    t = []
    if spec.model == "vae_gmp":                                 # vae.py:231-238
        t += [("loc", (K, Z)), ("raw_scale_diag", (K, Z)), ("mixture_logits", (K,))]
    elif spec.model != "vae":
        raise ValueError(spec.model)
    t += _mlp_shapes("decoder", Z, H + [D])                     # vae.py:254-259
    t += _mlp_shapes("encoder", D, H + [2 * Z])                 # vae.py:262-268
    return t


def glorot_limit(shape: Tuple[int, ...]) -> float:
    """xavier_initializer / glorot_uniform limit sqrt(6/(fan_in+fan_out)); 1-D: fan_in=fan_out=n."""
    if len(shape) == 1:
        fi = fo = shape[0]
    else:
        fi, fo = shape[0], shape[1]
    return math.sqrt(6.0 / (fi + fo))


def init_params(spec: Spec, seed: int = 2024, dtype=torch.float64) -> Dict[str, torch.Tensor]:
    """Xavier-uniform weights, zero biases (base.py:12); glorot-uniform for the VAE_GMP prior
    variables created by tf.get_variable without an initializer (vae.py:233-238)."""
    g = torch.Generator().manual_seed(seed)
    params = {}
    for name, shape in param_shapes(spec):
        if name.endswith("/b"):
            params[name] = torch.zeros(shape, dtype=dtype)
        else:
            lim = glorot_limit(shape)
            u = torch.rand(shape, generator=g, dtype=torch.float64)
            params[name] = ((2.0 * u - 1.0) * lim).to(dtype)
    return params


class Exact:
    """Rounding model of the arithmetic: the default is none (exact fp64/fp32 evaluation).
    tests/helpers.py subclasses it to restate WHERE the bf16 CUDA path rounds (stored activations,
    stored activation gradients, tensor-core weight operands), so that bf16 gradients can be
    compared without the ReLU-mask flips that any reduced-precision forward pass produces."""

    def act(self, t):            # a stored hidden activation (and its stored gradient)
        return t

    def fwd(self, t):            # stored in reduced precision in the forward pass only
        return t

    def grad(self, t):           # only the gradient flowing back through t is stored reduced
        return t

    def weight(self, name, w):   # GEMM weight operand
        return w

    def yin(self, t):            # the relaxed sample y as input of encoder_gmm
        return t


EXACT = Exact()


def mlp(params: Dict[str, torch.Tensor], name: str, h: torch.Tensor, n_layers: int, q: Exact = EXACT) -> torch.Tensor:
    """snt.nets.MLP(activation=relu, activate_final=False): relu between layers only."""
    for i in range(n_layers):
        wn = f"{name}_fcnet/linear_{i}/w"
        h = h @ q.weight(wn, params[wn]) + params[f"{name}_fcnet/linear_{i}/b"]
        if i != n_layers - 1:
            h = q.act(torch.relu(h))
    return h


def softplus(t: torch.Tensor) -> torch.Tensor:
    return torch.logaddexp(t, torch.zeros_like(t))


def normal_params(spec: Spec, outs: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """base.py:69-70."""
    mu, raw = outs.chunk(2, dim=1)
    sigma = torch.clamp_min(softplus(raw + spec.raw_sigma_bias), spec.sigma_min)
    return mu, sigma


def mvn_diag_log_prob(z, mu, sigma):
    """tfd.MultivariateNormalDiag.log_prob (Appendix B.3)."""
    Zd = z.shape[-1]
    return (-0.5 * (((z - mu) / sigma) ** 2).sum(-1) - torch.log(sigma).sum(-1) - 0.5 * Zd * LOG_2PI)


def bernoulli_log_prob(x, logits):
    """tfd.Independent(tfd.Bernoulli(logits),1).log_prob = -sum sigmoid_cross_entropy (B.4)."""
    return (x * logits - torch.clamp_min(logits, 0) - torch.log1p(torch.exp(-logits.abs()))).sum(-1)


def gumbel_softmax_sample(logits, u, temperature):
    """tfd.RelaxedOneHotCategorical.sample with injected uniforms u in [tiny,1) (B.5)."""
    g = -torch.log(-torch.log(u))
    return torch.softmax((logits + g) / temperature, dim=-1)


def entropy(logits, targets):
    """utils.py:165-170."""
    return -(targets * torch.log_softmax(logits, dim=-1)).sum(dim=1)


def loss_terms(spec: Spec, params: Dict[str, torch.Tensor], x: torch.Tensor,
               eps: torch.Tensor, u: Optional[torch.Tensor] = None,
               objective: str = "reference", global_batch: Optional[int] = None, q: Exact = EXACT) -> Dict[str, torch.Tensor]:
    """Forward pass.  Returns loss, nll, kl_div_z, nent (nent == 0 for VAE models) and a few
    intermediates used by the tests (among them the clamped scales sigma_q of q(z|.) and, for the
    GMVAE, sigma_p of p(z|y)).  `global_batch` (default: len(x)) is the divisor of the
    batch means, so that shards of a data-parallel batch can be summed."""
    dt = next(iter(params.values())).dtype
    x = x.to(dt)
    B = x.shape[0]
    Bg = float(global_batch if global_batch is not None else B)
    L = len(spec.hidden_sizes) + 1
    out: Dict[str, torch.Tensor] = {}
    if spec.model in ("vae", "vae_gmp"):                                   # vae.py:167-185
        mu_q, sg_q = normal_params(spec, q.grad(mlp(params, "encoder", x, L, q)))
        z = mu_q + sg_q * eps.to(dt)
        logits = q.grad(mlp(params, "decoder", q.fwd(z), L, q)) + spec.gen_bias_init
        nll = -bernoulli_log_prob(x, logits).sum() / Bg
        logq = mvn_diag_log_prob(z, mu_q, sg_q)
        if spec.model == "vae":                                           # vae.py:247-250
            logp = -0.5 * (z ** 2).sum(-1) - 0.5 * spec.latent_size * LOG_2PI
        else:                                                             # vae.py:240-244
            comp = mvn_diag_log_prob(z[:, None, :], params["loc"][None], softplus(params["raw_scale_diag"])[None])
            logp = torch.logsumexp(comp + torch.log_softmax(params["mixture_logits"], -1)[None], dim=-1)
        kl = (logq - logp).sum() / Bg
        zero = torch.zeros((), dtype=dt)
        out.update(loss=nll + kl, nll=nll, kl_div_z=kl, nent=zero, z=z, logits_x=logits, sigma_q=sg_q)
        return out
    if spec.model != "gmvae":
        raise ValueError(spec.model)
    K, Z = spec.mixture_components, spec.latent_size
    ly = q.grad(mlp(params, "encoder_y", x, L, q))                         # gmvae.py:238
    py = torch.softmax(ly, -1)
    nent = -entropy(ly, py).sum() / Bg                                     # gmvae.py:262-263
    if objective == "reference":
        y = gumbel_softmax_sample(ly, u.to(dt), spec.temperature)          # gmvae.py:240
        mu_p, sg_p = normal_params(spec, q.grad(mlp(params, "prior_gmm", q.yin(y), 1, q)))   # gmvae.py:243
        mu_q, sg_q = normal_params(spec, q.grad(mlp(params, "encoder_gmm", torch.cat([x, q.yin(y)], 1), L, q)))  # :246
        z = mu_q + sg_q * eps.to(dt)                                       # gmvae.py:248
        logits = q.grad(mlp(params, "decoder", q.fwd(z), L, q)) + spec.gen_bias_init   # gmvae.py:251
        nll = -bernoulli_log_prob(x, logits).sum() / Bg                    # gmvae.py:254
        kl = (mvn_diag_log_prob(z, mu_q, sg_q) - mvn_diag_log_prob(z, mu_p, sg_p)).sum() / Bg  # :258
        out.update(y=y, z=z, logits_x=logits, sigma_q=sg_q, sigma_p=sg_p)
    elif objective == "marginal":
        # SURVEY.md Appendix A.3: the reference's own blocks evaluated at y = e_k for every k,
        # weighted by q(y|x), with the analytic Gaussian KL.  eps has shape [B, K, Z].
        eye = torch.eye(K, dtype=dt)
        mu_p, sg_p = normal_params(spec, mlp(params, "prior_gmm", eye, 1))            # [K,Z]  (exact: a table)
        xk = x[:, None, :].expand(B, K, x.shape[1]).reshape(B * K, -1)
        # encoder_gmm([x, e_k]): layer 0 written as x W[:D] + W[D+k] + b (identical to the concat form,
        # base.py:66) so that the rounding model can mirror the CUDA path: the x-projection uses the
        # GEMM weight operand, the one-hot row and the bias are added in full precision.
        D = x.shape[1]
        w0n = "encoder_gmm_fcnet/linear_0/w"
        w0, b0 = params[w0n], params["encoder_gmm_fcnet/linear_0/b"]
        xproj = q.grad(x @ q.weight(w0n, w0)[:D])                                   # [B, H0], once per sample
        h = q.act(torch.relu(xproj[:, None, :] + w0[D:][None, :, :] + b0)).reshape(B * K, -1)
        for i in range(1, L):
            wn = f"encoder_gmm_fcnet/linear_{i}/w"
            h = h @ q.weight(wn, params[wn]) + params[f"encoder_gmm_fcnet/linear_{i}/b"]
            if i != L - 1:
                h = q.act(torch.relu(h))
        mu_q, sg_q = normal_params(spec, q.grad(h))
        z = mu_q + sg_q * eps.to(dt).reshape(B * K, Z)
        logits = q.grad(mlp(params, "decoder", q.fwd(z), L, q)) + spec.gen_bias_init
        rec = bernoulli_log_prob(xk, logits).reshape(B, K)
        mu_q = mu_q.reshape(B, K, Z); sg_q = sg_q.reshape(B, K, Z)
        klk = (torch.log(sg_p[None] / sg_q) + (sg_q ** 2 + (mu_q - mu_p[None]) ** 2) / (2 * sg_p[None] ** 2) - 0.5).sum(-1)
        nll = -(py * rec).sum() / Bg
        kl = (py * klk).sum() / Bg
        out.update(z=z, logits_x=logits, sigma_q=sg_q, sigma_p=sg_p)
    else:
        raise ValueError(objective)
    out.update(loss=nll + kl + nent, nll=nll, kl_div_z=kl, nent=nent, logits_y=ly)
    return out


def loss_and_grads(spec, params, x, eps, u=None, objective="reference", global_batch=None, q: Exact = EXACT):
    """opt.compute_gradients(loss, tf.trainable_variables()) (runners.py:182) by autograd."""
    leaf = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    terms = loss_terms(spec, leaf, x, eps, u, objective, global_batch, q)
    names = list(leaf)
    gs = torch.autograd.grad(terms["loss"], [leaf[n] for n in names], allow_unused=True)
    grads = {n: (g if g is not None else torch.zeros_like(leaf[n])) for n, g in zip(names, gs)}
    return {k: v.detach() for k, v in terms.items()}, grads


@dataclass
class AdamState:
    m: Dict[str, torch.Tensor]
    v: Dict[str, torch.Tensor]
    t: int = 0


def adam_init(params) -> AdamState:
    return AdamState({k: torch.zeros_like(p) for k, p in params.items()},
                     {k: torch.zeros_like(p) for k, p in params.items()}, 0)


def adam_tf_step(params, grads, st: AdamState, lr=1e-3, beta1=0.9, beta2=0.999, epsilon=1e-8):
    """tf.train.AdamOptimizer ("epsilon-hat" form, Appendix B.6), in place:
       lr_t = lr*sqrt(1-b2^t)/(1-b1^t); m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
       theta -= lr_t * m / (sqrt(v) + eps)."""
    st.t += 1
    lr_t = lr * math.sqrt(1.0 - beta2 ** st.t) / (1.0 - beta1 ** st.t)
    for k, p in params.items():
        g = grads[k]
        st.m[k].mul_(beta1).add_(g, alpha=1.0 - beta1)
        st.v[k].mul_(beta2).addcmul_(g, g, value=1.0 - beta2)
        p.sub_(lr_t * st.m[k] / (st.v[k].sqrt() + epsilon))
    return params


def train_step(spec, params, st, x, eps, u=None, objective="reference", lr=1e-3):
    """One iteration of the hot loop runners.py:231-232: loss -> grads -> Adam."""
    terms, grads = loss_and_grads(spec, params, x, eps, u, objective)
    adam_tf_step(params, grads, st, lr=lr)
    return terms, grads


# ----------------------------------------------------------------------------- synthetic inputs
def synthetic_batch(spec: Spec, batch: int, seed_data=1234, seed_noise=4321, objective="reference"):
    """SURVEY.md §8(d): per-pixel rate p_d ~ U(0,1); x = U<p_d (bool); eps ~ N(0,I);
    u ~ U[tiny,1)."""
    gd = torch.Generator().manual_seed(seed_data)
    gn = torch.Generator().manual_seed(seed_noise)
    p = torch.rand(spec.data_size, generator=gd)
    x = torch.rand(batch, spec.data_size, generator=gd) < p
    labels = torch.randint(0, 10, (batch,), generator=gd)
    if spec.model == "gmvae" and objective == "marginal":
        eps = torch.randn(batch, spec.mixture_components, spec.latent_size, generator=gn)
    else:
        eps = torch.randn(batch, spec.latent_size, generator=gn)
    u = None
    if spec.model == "gmvae":
        u = torch.rand(batch, spec.mixture_components, generator=gn).clamp_min(torch.finfo(torch.float32).tiny)
    return x, labels, eps, u
