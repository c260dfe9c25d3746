"""Engine: owns the device buffers (PyTorch tensors) of one model replica and drives the native
training step through the C ABI.  Mirrors what the reference's TF graph + session own:
the trainable variables (runners.py:182), Adam slots and global_step (runners.py:181-183),
and one `sess.run([train_op, global_step])` per `train_step()` (runners.py:231-232)."""
from __future__ import annotations

import ctypes as C
import math
from collections import OrderedDict
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from . import _lib


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class Engine:
    def __init__(self, model: str = "gmvae", data_size: int = 784, latent_size: int = 64,
                 hidden_sizes: Sequence[int] = (512, 512), mixture_components: int = 10, *,
                 objective: str = "reference", precision: str = "bf16", max_batch: int = 128,
                 sigma_min: float = 0.0, raw_sigma_bias: float = 0.5, gen_bias_init: float = 0.0,
                 temperature: float = 1.0, learning_rate: float = 1e-3, beta1: float = 0.9,
                 beta2: float = 0.999, epsilon: float = 1e-8, device: Optional[int] = None,
                 seed: Optional[int] = None, init: bool = True, deterministic: bool = False):
        """deterministic=True: bitwise-reproducible training steps (gmvae_config::deterministic, DESIGN.md section 9).
        mixture_components: up to 1024 for the GMVAE under objective "reference", up to 128 for VAE_GMP and "marginal"."""
        if not torch.cuda.is_available():
            raise RuntimeError("gmvae_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self.model, self.objective, self.precision = model, objective, precision
        self.data_size, self.latent_size = int(data_size), int(latent_size)
        self.hidden_sizes = [int(h) for h in hidden_sizes]
        self.mixture_components = int(mixture_components)
        self.max_batch = int(max_batch)
        self.deterministic = bool(deterministic)
        cfg = _lib.Config()
        cfg.abi_version = _lib.ABI_VERSION
        cfg.model = _lib.MODEL_IDS[model]
        cfg.objective = _lib.OBJECTIVE_IDS[objective]
        cfg.precision = _lib.PRECISION_IDS[precision]
        cfg.data_size, cfg.latent_size = self.data_size, self.latent_size
        cfg.mixture_components = self.mixture_components
        if len(self.hidden_sizes) > _lib.MAX_HIDDEN:
            raise ValueError(f"at most {_lib.MAX_HIDDEN} hidden layers")
        cfg.num_hidden = len(self.hidden_sizes)
        for i, hs in enumerate(self.hidden_sizes):
            cfg.hidden_sizes[i] = hs
        cfg.max_batch = self.max_batch
        cfg.sigma_min, cfg.raw_sigma_bias = sigma_min, raw_sigma_bias
        cfg.gen_bias_init, cfg.temperature = gen_bias_init, temperature
        cfg.learning_rate, cfg.beta1, cfg.beta2, cfg.epsilon = learning_rate, beta1, beta2, epsilon
        cfg.device = self.device_index
        cfg.deterministic = 1 if self.deterministic else 0
        self.cfg = cfg
        self._h = C.c_void_p()
        _lib.check(self.lib.gmvae_create(C.byref(cfg), C.byref(self._h)), "gmvae_create")
        n = self.lib.gmvae_param_count(self._h)
        ng = self.lib.gmvae_grad_count(self._h)
        with torch.cuda.device(self.device):
            self.params = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.grads = torch.zeros(ng, dtype=torch.float32, device=self.device)
            self.adam_m = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.adam_v = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.workspace = torch.zeros(self.lib.gmvae_workspace_bytes(self._h) + 256, dtype=torch.uint8, device=self.device)
            self.loss_buf = torch.zeros(4, dtype=torch.float32, device=self.device)
        ws_ptr = (self.workspace.data_ptr() + 255) // 256 * 256
        _lib.check(self.lib.gmvae_bind(self._h, self.params.data_ptr(), self.grads.data_ptr(), self.adam_m.data_ptr(),
                                       self.adam_v.data_ptr(), ws_ptr, self.lib.gmvae_workspace_bytes(self._h)), "gmvae_bind")
        k = self.lib.gmvae_num_params(self._h)
        table = (_lib.ParamDesc * k)()
        self.lib.gmvae_param_table(self._h, table, k)
        self.table = [(d.name.decode(), int(d.offset), int(d.rows), int(d.cols)) for d in table]
        self._keep = []          # tensors referenced by in-flight / captured work
        self._graph_ready = False
        self.world_size, self.rank = 1, 0
        self.peer_attached = False
        if seed is not None:
            _lib.check(self.lib.gmvae_set_seed(self._h, int(seed) & (2 ** 64 - 1)))
        if init:
            self.initialize(2024 if seed is None else seed)

    # ------------------------------------------------------------------ variables
    def _views(self, flat: torch.Tensor) -> "OrderedDict[str, torch.Tensor]":
        out = OrderedDict()
        for name, off, rows, cols in self.table:
            v = flat[off:off + rows * cols]
            out[name] = v.view(cols) if (rows == 1 and (name.endswith("/b") or name == "mixture_logits")) else v.view(rows, cols)
        return out

    def parameters(self):
        """name -> view into the flat fp32 parameter buffer (the reference's TF variable names)."""
        return self._views(self.params)

    def gradients(self):
        return self._views(self.grads)

    def initialize(self, seed: int = 2024):
        """Xavier-uniform weights / zero biases (base.py:12); glorot-uniform for the VAE_GMP prior
        variables created without an initializer (vae.py:233-238)."""
        g = torch.Generator().manual_seed(int(seed))
        for name, view in self.parameters().items():
            if name.endswith("/b"):
                view.zero_()
                continue
            shape = tuple(view.shape)
            fi, fo = (shape[0], shape[0]) if len(shape) == 1 else shape
            lim = math.sqrt(6.0 / (fi + fo))
            u = torch.rand(shape, generator=g, dtype=torch.float64)
            view.copy_(((2.0 * u - 1.0) * lim).to(torch.float32))
        self.adam_m.zero_(); self.adam_v.zero_()
        self.params_updated()

    def set_parameters(self, values: Dict[str, torch.Tensor]):
        views = self.parameters()
        for name, val in values.items():
            views[name].copy_(torch.as_tensor(val).to(torch.float32).reshape(views[name].shape))
        self.params_updated()

    def params_updated(self):
        _lib.check(self.lib.gmvae_params_updated(self._h, self._stream()), "gmvae_params_updated")

    # ------------------------------------------------------------------ helpers
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _as_u8(self, x) -> torch.Tensor:
        if isinstance(x, np.ndarray):
            x = torch.from_numpy(x)
        x = x.reshape(x.shape[0], -1)
        if x.shape[1] != self.data_size:
            raise ValueError(f"expected {self.data_size} features, got {x.shape[1]}")
        if x.dtype != torch.uint8:
            x = x.to(torch.uint8) if x.dtype == torch.bool else (x != 0).to(torch.uint8)
        return x.to(self.device, non_blocking=True).contiguous()

    def _as_f32(self, t, shape) -> Optional[torch.Tensor]:
        if t is None:
            return None
        t = torch.as_tensor(t).to(self.device, torch.float32).contiguous()
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f"noise shape {tuple(t.shape)} != {tuple(shape)}")
        return t

    def _noise(self, B, eps, gumbel_u):
        Z, K = self.latent_size, self.mixture_components
        eshape = (B, K, Z) if (self.model == "gmvae" and self.objective == "marginal") else (B, Z)
        e = self._as_f32(eps, eshape)
        u = self._as_f32(gumbel_u, (B, K)) if self.model == "gmvae" else None
        return e, u

    # ------------------------------------------------------------------ the step
    def forward_backward(self, x, eps=None, gumbel_u=None, global_batch: Optional[int] = None, finalize: bool = True):
        """run_model + compute_gradients.  Loss terms land in `loss_terms()`, gradients in `gradients()`."""
        xu = self._as_u8(x)
        B = xu.shape[0]
        e, u = self._noise(B, eps, gumbel_u)
        self._keep = [xu, e, u]
        st = self._stream()
        _lib.check(self.lib.gmvae_forward_backward(self._h, xu.data_ptr(), B, int(global_batch or B), _ptr(e), _ptr(u), st),
                   "gmvae_forward_backward")
        if finalize:
            _lib.check(self.lib.gmvae_finalize_loss(self._h, self.loss_buf.data_ptr(), st), "gmvae_finalize_loss")
        return self.loss_buf

    def allreduce_grads(self):
        _lib.check(self.lib.gmvae_allreduce_grads(self._h, self._stream()), "gmvae_allreduce_grads")

    def finalize_loss(self):
        _lib.check(self.lib.gmvae_finalize_loss(self._h, self.loss_buf.data_ptr(), self._stream()), "gmvae_finalize_loss")
        return self.loss_buf

    def adam_step(self):
        _lib.check(self.lib.gmvae_adam_step(self._h, self._stream()), "gmvae_adam_step")

    def train_step(self, x, eps=None, gumbel_u=None, global_batch: Optional[int] = None) -> torch.Tensor:
        """One `sess.run([train_op, ...])`: returns the device tensor [loss, nll, kl_div_z, nent]
        (not synchronised)."""
        xu = self._as_u8(x)
        B = xu.shape[0]
        e, u = self._noise(B, eps, gumbel_u)
        self._keep = [xu, e, u]
        gb = int(global_batch or B * self.world_size)
        _lib.check(self.lib.gmvae_train_step(self._h, xu.data_ptr(), B, gb, _ptr(e), _ptr(u), self.loss_buf.data_ptr(),
                                             self._stream()), "gmvae_train_step")
        return self.loss_buf

    # ------------------------------------------------------------------ input pipeline on the device
    def binarize(self, intensities: torch.Tensor, batch: Optional[int] = None, first_row: int = 0,
                 row_index: Optional[torch.Tensor] = None, draw: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Dynamic binarisation of runners.create_dataset._preprocess (runners.py:44-47), `intensity/255 < uniform`,
        on device-resident bytes `intensities` [N, D].  Rows `first_row .. first_row+batch` (the reference's
        contiguous batches) or the rows named by `row_index` (int64 CUDA tensor).  Returns uint8 {0,1} [batch, D]."""
        if intensities.dtype != torch.uint8 or not intensities.is_cuda or not intensities.is_contiguous() or intensities.dim() != 2:
            raise ValueError("intensities must be a contiguous uint8 CUDA tensor [N, D]")
        N, D = intensities.shape
        if D != self.data_size:
            raise ValueError(f"expected {self.data_size} features, got {D}")
        if row_index is not None:
            if row_index.dtype != torch.int64 or not row_index.is_cuda or not row_index.is_contiguous():
                raise ValueError("row_index must be a contiguous int64 CUDA tensor")
            B, src, n_rows = int(row_index.numel()), intensities, N
        else:
            B = int(N - first_row if batch is None else batch)
            if first_row < 0 or B < 0 or first_row + B > N:
                raise ValueError(f"rows [{first_row}, {first_row + B}) outside the {N} intensity rows")
            src, n_rows = intensities[first_row:], N - first_row
        if out is None:
            out = torch.empty(B, D, dtype=torch.uint8, device=self.device)
        elif out.dtype != torch.uint8 or not out.is_cuda or not out.is_contiguous() or tuple(out.shape) != (B, D):
            raise ValueError("out must be a contiguous uint8 CUDA tensor [batch, D]")
        self._keep_in = [intensities, row_index, out]
        _lib.check(self.lib.gmvae_binarize(self._h, src.data_ptr(), n_rows, _ptr(row_index), B, int(draw) & (2 ** 64 - 1),
                                           out.data_ptr(), self._stream()), "gmvae_binarize")
        return out

    def unpack_bits(self, packed: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Bit-packed binary images (numpy.packbits(x, axis=1): ceil(D/8) bytes per row, most significant bit first) ->
        uint8 {0,1} [batch, D] on the device.  `packed` is a uint8 CUDA tensor [batch, ceil(D/8)]; pass the captured step's
        input as `out` to refill it in place before `replay()`."""
        rb = (self.data_size + 7) // 8
        if packed.dtype != torch.uint8 or not packed.is_cuda or not packed.is_contiguous() or packed.dim() != 2 or packed.shape[1] != rb:
            raise ValueError(f"packed must be a contiguous uint8 CUDA tensor [batch, {rb}]")
        B = packed.shape[0]
        if out is None:
            out = torch.empty(B, self.data_size, dtype=torch.uint8, device=self.device)
        elif out.dtype != torch.uint8 or not out.is_cuda or not out.is_contiguous() or tuple(out.shape) != (B, self.data_size):
            raise ValueError("out must be a contiguous uint8 CUDA tensor [batch, D]")
        self._keep_in = [packed, out]
        _lib.check(self.lib.gmvae_unpack_bits(self._h, packed.data_ptr(), B, out.data_ptr(), self._stream()), "gmvae_unpack_bits")
        return out

    # ------------------------------------------------------------------ forward-only helpers
    def encode(self, x, eps=None, gumbel_u=None):
        """(logits_y or None, z_mean, z_sample): encoder side of the forward pass (gmvae.py:140-150, vae.py:105-112)."""
        xu = self._as_u8(x)
        B = xu.shape[0]
        Z, K = self.latent_size, self.mixture_components
        e = self._as_f32(eps, (B, Z))
        u = self._as_f32(gumbel_u, (B, K)) if self.model == "gmvae" else None
        logits = torch.empty(B, K, dtype=torch.float32, device=self.device) if self.model == "gmvae" else None
        zm = torch.empty(B, Z, dtype=torch.float32, device=self.device)
        zs = torch.empty(B, Z, dtype=torch.float32, device=self.device)
        self._keep = [xu, e, u]
        # gmvae_encode takes at most max_batch rows: larger batches go in slices, as in decode (rows are independent)
        for i in range(0, B, self.max_batch):
            n = min(self.max_batch, B - i)
            ei = None if e is None else e[i:i + n]
            ui = None if u is None else u[i:i + n]
            li = None if logits is None else logits[i:i + n]
            _lib.check(self.lib.gmvae_encode(self._h, xu[i:i + n].data_ptr(), n, _ptr(ei), _ptr(ui), _ptr(li), zm[i:i + n].data_ptr(),
                                             zs[i:i + n].data_ptr(), self._stream()), "gmvae_encode")
        return logits, zm, zs

    def decode(self, z) -> torch.Tensor:
        """Bernoulli mean sigmoid(decoder(z)) [n, data_size] (base.py:138-146)."""
        z = torch.as_tensor(z).to(self.device, torch.float32).reshape(-1, self.latent_size).contiguous()
        out = torch.empty(z.shape[0], self.data_size, dtype=torch.float32, device=self.device)
        for i in range(0, z.shape[0], self.max_batch):
            zc = z[i:i + self.max_batch]
            _lib.check(self.lib.gmvae_decode(self._h, zc.data_ptr(), zc.shape[0], out[i:i + self.max_batch].data_ptr(), self._stream()),
                       "gmvae_decode")
        self._keep = [z]
        return out

    def prior_table(self):
        """(mu [K,Z], sigma [K,Z]) of the prior components: prior_gmm(one_hot(k)) for the GMVAE
        (gmvae.py:170-173), (loc, softplus(raw_scale_diag)) for VAE_GMP, N(0,I) for the VAE."""
        K = self.mixture_components if self.model != "vae" else 1
        mu = torch.empty(K, self.latent_size, dtype=torch.float32, device=self.device)
        sg = torch.empty_like(mu)
        _lib.check(self.lib.gmvae_prior_table(self._h, mu.data_ptr(), sg.data_ptr(), self._stream()), "gmvae_prior_table")
        return mu, sg

    # ------------------------------------------------------------------ CUDA graph of the whole step
    def capture_step(self, x_static: torch.Tensor, eps=None, gumbel_u=None, global_batch: Optional[int] = None):
        """Captures train_step on fixed buffers; refill `x_static` (uint8 [B, D] on this device) in
        place and call `replay()`."""
        if x_static.dtype != torch.uint8 or not x_static.is_cuda or not x_static.is_contiguous():
            raise ValueError("x_static must be a contiguous uint8 CUDA tensor")
        B = x_static.shape[0]
        e, u = self._noise(B, eps, gumbel_u)
        self._graph_keep = [x_static, e, u]
        gb = int(global_batch or B * self.world_size)
        st = torch.cuda.current_stream(self.device)
        if st.cuda_stream == 0:
            raise RuntimeError("capture_step must run inside `with torch.cuda.stream(side_stream)`")
        _lib.check(self.lib.gmvae_step_graph_capture(self._h, x_static.data_ptr(), B, gb, _ptr(e), _ptr(u),
                                                     self.loss_buf.data_ptr(), st.cuda_stream), "gmvae_step_graph_capture")
        self._graph_ready = True

    def replay(self) -> torch.Tensor:
        if not self._graph_ready:
            raise RuntimeError("capture_step() first")
        _lib.check(self.lib.gmvae_step_graph_launch(self._h, self._stream()), "gmvae_step_graph_launch")
        return self.loss_buf

    # ------------------------------------------------------------------ optimiser state / checkpoints
    @property
    def global_step(self) -> int:
        s = C.c_int64()
        _lib.check(self.lib.gmvae_get_step(self._h, C.byref(s), self._stream()))
        return int(s.value)

    def set_global_step(self, step: int):
        _lib.check(self.lib.gmvae_set_step(self._h, int(step), self._stream()))

    def launch_count(self) -> int:
        return int(self.lib.gmvae_launch_count(self._h))

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """Keys follow the TF Saver naming of the reference (var, var/Adam, var/Adam_1, global_step)."""
        out = OrderedDict()
        for name, v in self.parameters().items():
            out[name] = v.detach().cpu().clone()
        for name, v in self._views(self.adam_m).items():
            out[name + "/Adam"] = v.detach().cpu().clone()
        for name, v in self._views(self.adam_v).items():
            out[name + "/Adam_1"] = v.detach().cpu().clone()
        t = self.global_step
        out["global_step"] = torch.tensor(t, dtype=torch.int64)
        out["beta1_power"] = torch.tensor(float(self.cfg.beta1) ** (t + 1))
        out["beta2_power"] = torch.tensor(float(self.cfg.beta2) ** (t + 1))
        return out

    def load_state_dict(self, sd: Dict[str, torch.Tensor]):
        pv, mv, vv = self.parameters(), self._views(self.adam_m), self._views(self.adam_v)
        for name in pv:
            pv[name].copy_(sd[name].reshape(pv[name].shape))
            if name + "/Adam" in sd:
                mv[name].copy_(sd[name + "/Adam"].reshape(mv[name].shape))
                vv[name].copy_(sd[name + "/Adam_1"].reshape(vv[name].shape))
        if "global_step" in sd:
            self.set_global_step(int(sd["global_step"]))
        self.params_updated()

    # ------------------------------------------------------------------ data parallel (NCCL over NVLink)
    def init_data_parallel(self):
        """One process per GPU; the NCCL unique id travels through torch.distributed (any backend)."""
        import torch.distributed as dist
        if not dist.is_initialized() or dist.get_world_size() == 1:
            return
        self.world_size, self.rank = dist.get_world_size(), dist.get_rank()
        buf = C.create_string_buffer(128)
        if self.rank == 0:
            _lib.check(self.lib.gmvae_nccl_unique_id(buf), "gmvae_nccl_unique_id")
        obj = [bytes(buf.raw)]
        dist.broadcast_object_list(obj, src=0)
        _lib.check(self.lib.gmvae_nccl_init(self._h, obj[0], self.world_size, self.rank), "gmvae_nccl_init")
        import os
        if os.environ.get("GMVAE_DP_PEER", "1") != "0":
            self.attach_peers()
        if self.deterministic and not self.peer_attached:
            import warnings
            warnings.warn("deterministic=True: the NCCL all-reduce adds the ranks' gradients in an order of its own; "
                          "steps are bitwise reproducible only with the peer-memory exchange")

    def attach_peers(self) -> bool:
        """The exchange step over NVLink peer memory, fused with Adam (csrc/peer.cuh), in place of the NCCL all-reduce (default
        under data parallelism; GMVAE_DP_PEER=0 keeps NCCL).  Every rank exports its symmetric region, the cudaIpc handles travel
        through torch.distributed, and a barrier separates attaching from the first step.  The gradient buffer moves into the
        region: `self.grads` is re-pointed at it (zero-copy view of library-owned memory).  The ranks agree after each phase on
        whether it worked everywhere; if the regions cannot be exported (no P2P / IPC) every rank stays with NCCL and this returns
        False."""
        import warnings
        import torch.distributed as dist

        def everywhere(ok: bool) -> bool:
            oks = [None] * self.world_size
            dist.all_gather_object(oks, bool(ok))
            return all(oks)

        buf = C.create_string_buffer(64)
        err = None
        try:
            _lib.check(self.lib.gmvae_peer_export(self._h, self.world_size, self.rank, buf), "gmvae_peer_export")
        except RuntimeError as e:
            err = e
        if not everywhere(err is None):
            warnings.warn(f"peer-memory gradient exchange unavailable ({err or 'another rank could not export its region'}); using the NCCL all-reduce")
            return False
        handles = [None] * self.world_size
        dist.all_gather_object(handles, bytes(buf.raw))
        try:
            _lib.check(self.lib.gmvae_peer_attach(self._h, b"".join(handles)), "gmvae_peer_attach")
        except RuntimeError as e:
            err = e
        if not everywhere(err is None):
            # a rank that did attach has already moved its gradient buffer: there is no common fallback left
            raise RuntimeError(f"the peer-memory exchange could be attached on some ranks only ({err}); run with GMVAE_DP_PEER=0")
        ptr = self.lib.gmvae_peer_grads(self._h)

        class _Raw:                                              # torch.as_tensor understands the CUDA array interface: no copy
            __cuda_array_interface__ = {"shape": (int(self.grads.numel()),), "typestr": "<f4", "data": (int(ptr), False), "version": 2}
        with torch.cuda.device(self.device):
            self._grads_bound = self.grads
            self.grads = torch.as_tensor(_Raw(), device=self.device)
        self._graph_ready = False
        self.peer_attached = True
        dist.barrier()
        return True

    PROFILE_CLASSES = ["tc_gemm_fwd_dgrad", "tc_gemm_wgrad", "simt_gemm", "heads", "bias_grad", "adam_refresh", "misc", "comm"]

    def profile(self, on: bool):
        _lib.check(self.lib.gmvae_profile_enable(self._h, int(on)))

    def profile_read(self) -> Dict[str, dict]:
        ms = (C.c_double * 8)(); n = (C.c_int64 * 8)()
        self.lib.gmvae_profile_read(self._h, ms, n, 8)
        return {name: {"ms": ms[i], "launches": int(n[i])} for i, name in enumerate(self.PROFILE_CLASSES)}

    def debug_noise(self, n_eps: int, n_u: int):
        """Draws from the step's device noise generator (test hook)."""
        e = torch.empty(n_eps, dtype=torch.float32, device=self.device)
        u = torch.empty(n_u, dtype=torch.float32, device=self.device)
        _lib.check(self.lib.gmvae_debug_noise(self._h, e.data_ptr() if n_eps else None, n_eps, u.data_ptr() if n_u else None,
                                              n_u, self._stream()), "gmvae_debug_noise")
        return e, u

    def debug_gemm(self, impl: int, A: torch.Tensor, B: torch.Tensor, transA=False, transB=False, split_k=1) -> torch.Tensor:
        """C = op(A) op(B) through the step's own GEMM kernels (impl 0 SIMT fp32, 1 tcgen05 bf16).  impl 1 takes
        (transA, transB) = (False, True): both operands K-major, the data-gradient GEMMs; (False, False): A K-major and B
        MN-major, the forward GEMM of a layer outside the chained kernel (what encode / decode / condition run); and
        (True, False): both MN-major, the weight-gradient GEMMs."""
        A = A.to(self.device, torch.float32).contiguous(); B = B.to(self.device, torch.float32).contiguous()
        M, K = (A.shape[1], A.shape[0]) if transA else A.shape
        N = B.shape[0] if transB else B.shape[1]
        out = torch.empty(M, N, dtype=torch.float32, device=self.device)
        _lib.check(self.lib.gmvae_debug_gemm(self._h, impl, int(transA), int(transB), M, N, K, A.data_ptr(), B.data_ptr(),
                                             out.data_ptr(), split_k, self._stream()), "gmvae_debug_gemm")
        return out

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            torch.cuda.synchronize(self.device)
            self.lib.gmvae_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
