"""Matern 1/2, 3/2, 5/2 factors (SVGP_K_MATERN12 / 32 / 52) on the CPU: the oracle classes against scikit-learn and
against their closed-form adjoints (including r = 0), and productSVGP with Matern kinds through elbo_step on the float64
oracle backend against the streamlined float64 oracle on the same kernel matrices."""
import math
import os
import re

import numpy as np
import pytest
import torch

import refs
from conftest import ROOT, rel_err
import matern_oracle as mo
import svgp_vae_b200 as pkg
from svgp_vae_b200 import _lib, backend, configs

F64 = torch.float64
TOL = 2e-5          # as test_host_logic: the stand-in backend rounds K_nm, p, ... to fp32 like the CUDA path
CLASSES = {0.5: mo.MaternOneHalf, 1.5: mo.MaternThreeHalves, 2.5: mo.MaternFiveHalves}
CODES = {"matern12": 5, "matern32": 6, "matern52": 7}


def _closed_form(nu, r, a, l):
    """(k, C, dk/dl) of the issue table: dk/dz_f = C (x_f - z_f), dk/dx_f = -C (x_f - z_f); C = 0 at r = 0 for nu = 1/2."""
    c = {0.5: 1.0, 1.5: math.sqrt(3.0), 2.5: math.sqrt(5.0)}[nu]
    u = c * r / l
    e = a * a * torch.exp(-u)
    if nu == 0.5:
        k = e
        C = torch.where(r > 0, k / (l * torch.where(r > 0, r, torch.ones_like(r))), torch.zeros_like(r))
        dl = k * u / l
    elif nu == 1.5:
        k = (1 + u) * e
        C = 3 * e / l ** 2
        dl = e * u * u / l
    else:
        k = (1 + u + u * u / 3) * e
        C = 5 * (1 + u) * e / (3 * l ** 2)
        dl = e * (u * u / 3) * (1 + u) / l
    return k, C, dl


@pytest.mark.parametrize("nu", [0.5, 1.5, 2.5])
def test_oracle_matern_against_sklearn(nu):
    from sklearn.gaussian_process.kernels import ConstantKernel, Matern
    g = torch.Generator().manual_seed(0)
    x, z = torch.randn(17, 5, generator=g, dtype=F64), torch.randn(9, 5, generator=g, dtype=F64)
    z[3] = x[4]                                                      # one pair at distance zero
    amp, ls = 0.7, 1.9
    k = CLASSES[nu](torch.tensor(amp, dtype=F64), torch.tensor(ls, dtype=F64))
    ref = (ConstantKernel(amp ** 2) * Matern(length_scale=ls, nu=nu))(x.numpy(), z.numpy())
    assert np.abs(k.matrix(x, z).numpy() - ref).max() < 1e-12
    assert torch.allclose(k.apply(x[:9], z), torch.diagonal(k.matrix(x[:9], z)), rtol=1e-15, atol=0)
    assert float(k.apply(x[4:5], z[3:4])) == pytest.approx(amp ** 2, rel=1e-15)


@pytest.mark.parametrize("nu", [0.5, 1.5, 2.5])
def test_oracle_matern_gradients_against_closed_form(nu):
    g = torch.Generator().manual_seed(1)
    n = 64
    x = torch.randn(n, 3, generator=g, dtype=F64)
    z = torch.randn(n, 3, generator=g, dtype=F64)
    z[::8] = x[::8]                                                  # r = 0 on every 8th pair
    w = torch.randn(n, generator=g, dtype=F64)
    a = torch.tensor(0.8, dtype=F64, requires_grad=True)
    l = torch.tensor(1.3, dtype=F64, requires_grad=True)
    xr, zr = x.clone().requires_grad_(True), z.clone().requires_grad_(True)
    k = CLASSES[nu](a, l).apply(xr, zr)
    gx, gz, ga, gl = torch.autograd.grad((w * k).sum(), [xr, zr, a, l])
    for t in (gx, gz, ga, gl):
        assert torch.isfinite(t).all()
    r = (x - z).norm(dim=1)
    kc, C, dl = _closed_form(nu, r, a.detach(), l.detach())
    assert rel_err(k, kc) < 1e-14
    dz = (w * C)[:, None] * (x - z)
    assert rel_err(gz, dz) < 1e-13 and rel_err(gx, -dz) < 1e-13
    assert (gz[::8] == 0).all() and (gx[::8] == 0).all()             # finite, zero at r = 0
    assert float(ga) == pytest.approx(float((w * 2 * kc / a.detach()).sum()), rel=1e-13)
    assert float(gl) == pytest.approx(float((w * dl).sum()), rel=1e-13)
    # the total derivative of k(z, z) = a^2 in z, both arguments moving together, is zero
    zz = z.clone().requires_grad_(True)
    (gzz,) = torch.autograd.grad((w * CLASSES[nu](a, l).apply(zz, zz)).sum(), [zz])
    assert (gzz == 0).all()


def test_matern_constants_match_the_header():
    hdr = open(os.path.join(ROOT, "include", "svgp_b200.h")).read()
    defs = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (SVGP_K_MATERN\d\d) (\d+)", hdr)}
    assert defs == {"SVGP_K_MATERN12": _lib.SVGP_K_MATERN12, "SVGP_K_MATERN32": _lib.SVGP_K_MATERN32,
                    "SVGP_K_MATERN52": _lib.SVGP_K_MATERN52} == {"SVGP_K_MATERN%s" % k[-2:]: v for k, v in CODES.items()}
    for name, code in CODES.items():
        assert pkg.productSVGP._TYPES[name] == code


@pytest.fixture
def matern_oracle_backend():
    """The float64 CPU stand-in backend with the Matern factors (tests/matern_oracle.py)."""
    old = backend.set_backend_for_tests(mo.MaternOracleBackend())
    yield
    backend.set_backend_for_tests(old)


def _check_step(kinds, N=500, M=48, L=3, Z_on_data=False, hyp=(0.9, 1.3, 1.1, 0.8)):
    cfg = configs.sweep_inputs(N, M, L)
    if Z_on_data:
        cfg["ctor"]["initial_inducing_points"] = cfg["aux"][::N // M][:M].numpy().copy()
    da, db = (8, 0) if kinds[1] == "none" else (4, 4)
    s = pkg.productSVGP(**dict(cfg["ctor"], dim_a=da, dim_b=db), kind_a=kinds[0], kind_b=kinds[1], amplitude=hyp[0::2],
                        length_scale=hyp[1::2])
    spec = s._spec()
    assert spec == (s._TYPES[kinds[0]], da, s._TYPES[kinds[1]], db)
    o = mo.ContinuousProduct(cfg["ctor"]["initial_inducing_points"], hyp, spec, cfg["ctor"]["jitter"], cfg["ctor"]["N_train"])
    op, sp = [o.inducing_index_points, o.hyp], [s.inducing_index_points, s._hyp()]
    r0, J0, g0 = refs.streamlined_objective(o, op, cfg["aux"], cfg["y"], cfg["noise"])
    r1, J1, g1 = refs.product_objective(s, sp, cfg["aux"], cfg["y"], cfg["noise"])
    assert rel_err(r1["p_m"], r0["p_m"]) < TOL and rel_err(r1["p_v"], r0["p_v"]) < TOL
    for k in ("inside_elbo_recon", "inside_elbo_kl", "ce_term", "KL_term"):
        assert abs(float(r1[k]) - float(r0[k])) < TOL * abs(float(r0[k])), k
    for name, a, b in zip(["dy", "dnoise", "dZ", "dhyp"], g0, g1):
        assert torch.isfinite(b).all(), name
        if a.abs().max() > 0:
            assert rel_err(b, a) < TOL, (name, rel_err(b, a))
    return g1


@pytest.mark.parametrize("kinds", [("matern52", "matern52"), ("matern32", "matern12"), ("matern12", "se"),
                                   ("matern52", "linear"), ("matern32", "none")])
def test_step_matern_against_streamlined_oracle(matern_oracle_backend, kinds):
    _check_step(kinds)


@pytest.mark.parametrize("kinds", [("matern12", "matern12"), ("matern52", "matern32")])
def test_step_matern_inducing_points_on_data_points(matern_oracle_backend, kinds):
    """Z initialised as a subset of the data rows: K_nm has entries at r = 0 besides the diagonal of K_mm."""
    g1 = _check_step(kinds, Z_on_data=True)
    assert torch.isfinite(g1[2]).all() and g1[2].abs().max() > 0


def test_unknown_kind_raises():
    cfg = configs.sweep_inputs(10, 4, 1)
    with pytest.raises(KeyError):
        pkg.productSVGP(**cfg["ctor"], kind_a="matern72")
    with pytest.raises(KeyError):
        pkg.productSVGP(**cfg["ctor"], kind_b="Matern52")
