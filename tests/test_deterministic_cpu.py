"""Deterministic mode without a GPU: the ABI field, the create-time checks (made before the device probe), the Python and
CLI switches, and the weight-gradient slice arithmetic compiled for the host (tests/native/host_det_slices.cu)."""
import ctypes as C
import os
import shutil
import subprocess
import types

import pytest

from gmvae_b200 import _lib, run_gmvae, runners

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_config_field_and_offset():
    # the field takes the place of reserved[0]: the struct keeps its size
    assert _lib.Config.deterministic.offset == 4 * (4 + 3 + 1 + 8 + 1 + 8 + 1)
    assert _lib.Config.reserved.offset == _lib.Config.deterministic.offset + 4
    assert C.sizeof(_lib.Config) == 4 * (4 + 3 + 1 + 8 + 1 + 8 + 1 + 7)
    src = open(os.path.join(ROOT, "include", "gmvae_abi.h")).read()
    assert "int32_t deterministic;" in src and "int32_t reserved[6];" in src


def _cfg(**kw):
    cfg = _lib.Config()
    cfg.abi_version = _lib.ABI_VERSION; cfg.model = 2; cfg.precision = 1; cfg.data_size = 784; cfg.latent_size = 8
    cfg.mixture_components = 10; cfg.num_hidden = 1; cfg.hidden_sizes[0] = 64; cfg.max_batch = 16
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


def _create_error(cfg):
    lib = _lib.load()
    h = C.c_void_p()
    rc = lib.gmvae_create(C.byref(cfg), C.byref(h))
    if rc == 0:
        lib.gmvae_destroy(h)
        return None
    return lib.gmvae_last_error().decode()


def test_create_rejects_flag_value():
    assert _create_error(_cfg(deterministic=2)) == "deterministic must be 0 or 1"
    assert _create_error(_cfg(deterministic=-1)) == "deterministic must be 0 or 1"


def test_create_rejects_marginal_objective():
    assert _create_error(_cfg(deterministic=1, objective=1)) == "deterministic mode supports objective=reference only"


@pytest.mark.parametrize("var", ["GMVAE_DEBUG_FLAGS", "GMVAE_CHAIN_SPLIT", "GMVAE_CHAIN_QUAD"])
def test_create_rejects_opt_in_plans(var, monkeypatch):
    monkeypatch.setenv(var, "8")
    assert _create_error(_cfg(deterministic=1)) == f"deterministic mode cannot be combined with {var}"
    monkeypatch.setenv(var, "0")
    assert _create_error(_cfg(deterministic=1)) != f"deterministic mode cannot be combined with {var}"


def test_cli_flag_parses():
    p = run_gmvae.build_parser()
    assert p.parse_args([]).deterministic is False
    assert p.parse_args(["--deterministic"]).deterministic is True


def test_configure_passes_the_switch():
    cfg = types.SimpleNamespace(model="gmvae", latent_size=8, hidden_size=64, num_layers=1, mixture_components=10,
                                logdir="/tmp/l")
    m = runners.create_model(cfg, 784)
    assert m._deterministic is False
    m.configure(deterministic=True)
    assert m._deterministic is True
    m.configure(precision="fp32")
    assert m._deterministic is True          # untouched by a call that does not name it


NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.fixture(scope="module")
def slices(tmp_path_factory):
    if not (os.path.exists(NVCC) or shutil.which("nvcc")):
        pytest.skip("nvcc not available")
    out = str(tmp_path_factory.mktemp("host_det") / "libhost_det.so")
    cmd = [NVCC if os.path.exists(NVCC) else "nvcc", "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC",
           os.path.join(ROOT, "tests", "native", "host_det_slices.cu"), "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    L = C.CDLL(out)
    L.host_det_check.argtypes = [C.c_int] * 7
    return L


# (rows = in, cols = out, tile width, requested k-splits, k-blocks over the batch): weight gradients of cfg4 / cfg5 / ragged shapes,
# the 784, 794, 10 and 50-row jobs among them (ragged row blocks that must not spill into the next slice)
WG_JOBS = [(784, 512, 256, 9, 256), (512, 784, 256, 9, 256), (512, 512, 256, 9, 256), (10, 512, 256, 37, 256), (512, 10, 64, 37, 256),
           (794, 512, 256, 9, 256), (50, 256, 256, 18, 128), (1024, 1024, 256, 4, 1024), (784, 1024, 256, 4, 1024),
           (64, 512, 256, 37, 256), (200, 72, 128, 3, 3), (37, 72, 128, 1, 1), (5, 13, 64, 2, 2), (130, 640, 256, 5, 79)]


@pytest.mark.parametrize("job", WG_JOBS)
@pytest.mark.parametrize("cl,grid", [(1, 148), (1, 37), (2, 148), (2, 74), (2, 10)])
def test_weight_gradient_slices(slices, job, cl, grid):
    assert slices.host_det_check(*job, cl, grid) == 0
