"""ARD length scales (SVGP_K_ARD) on the CPU: the float64 oracle against scikit-learn's anisotropic RBF / Matern and
against the closed-form adjoints, productSVGP with per-feature length scales through elbo_step on the float64 stand-in
backend against the streamlined float64 oracle, and the constructor's layout and validation."""
import math
import os
import re

import numpy as np
import pytest
import torch

import ard_oracle as ao
import refs
from conftest import ROOT, rel_err
import svgp_vae_b200 as pkg
from svgp_vae_b200 import _lib, backend, configs

F64 = torch.float64
TOL = 2e-5          # as test_matern: the stand-in backend rounds K_nm, p, ... to fp32 like the CUDA path
SE, M12, M32, M52, LINEAR, NONE, ARD = 1, 5, 6, 7, 3, 0, 16
NU = {M12: 0.5, M32: 1.5, M52: 2.5}
LS5 = [0.4, 1.1, 3.9, 0.7, 2.3]                                     # distinct, spanning ~10x


def test_ard_constant_matches_the_header():
    hdr = open(os.path.join(ROOT, "include", "svgp_b200.h")).read()
    assert int(re.search(r"#define SVGP_K_ARD (\d+)", hdr).group(1)) == _lib.SVGP_K_ARD == ARD


@pytest.mark.parametrize("base", [SE, M12, M32, M52])
def test_oracle_ard_against_sklearn(base):
    from sklearn.gaussian_process.kernels import RBF, ConstantKernel, Matern
    g = torch.Generator().manual_seed(0)
    x, z = torch.randn(17, 5, generator=g, dtype=F64), torch.randn(9, 5, generator=g, dtype=F64)
    z[3] = x[4]                                                      # one pair at distance zero
    amp, ls = 0.7, torch.tensor(LS5, dtype=F64)
    k = ao.ARDKernel(base, torch.tensor(amp, dtype=F64), ls)
    skl = RBF(length_scale=LS5) if base == SE else Matern(length_scale=LS5, nu=NU[base])
    ref = (ConstantKernel(amp ** 2) * skl)(x.numpy(), z.numpy())
    assert np.abs(k.matrix(x, z).numpy() - ref).max() < 1e-12
    assert torch.allclose(k.apply(x[:9], z), torch.diagonal(k.matrix(x[:9], z)), rtol=1e-15, atol=0)
    assert float(k.apply(x[4:5], z[3:4])) == pytest.approx(amp ** 2, rel=1e-15)


def _coefficient(base, r, a):
    """(k, C) of the scaled distance r (length scale 1): dk/dz'_f = C (x'_f - z'_f); C = 0 at r = 0 for Matern 1/2."""
    if base == SE:
        k = a * a * torch.exp(-0.5 * r * r)
        return k, k
    c = {M12: 1.0, M32: math.sqrt(3.0), M52: math.sqrt(5.0)}[base]
    u = c * r
    e = a * a * torch.exp(-u)
    if base == M12:
        return e, torch.where(r > 0, e / torch.where(r > 0, r, torch.ones_like(r)), torch.zeros_like(r))
    if base == M32:
        return (1 + u) * e, 3 * e
    return (1 + u + u * u / 3) * e, 5 * (1 + u) * e / 3


@pytest.mark.parametrize("base", [SE, M12, M32, M52])
def test_oracle_ard_gradients_against_closed_form(base):
    """dk/dz_f = C (x_f - z_f) / l_f^2 and dk/dl_f = C (x_f - z_f)^2 / l_f^3, also for offset features (time stamps in
    the thousands) and at r = 0."""
    g = torch.Generator().manual_seed(1)
    n = 64
    x = torch.randn(n, 5, generator=g, dtype=F64) * torch.tensor(LS5, dtype=F64)
    x[:, 2] += 3000.0
    z = x + 0.7 * torch.randn(n, 5, generator=g, dtype=F64)
    z[::8] = x[::8]                                                  # r = 0 on every 8th pair
    w = torch.randn(n, generator=g, dtype=F64)
    a = torch.tensor(0.8, dtype=F64, requires_grad=True)
    ls = torch.tensor(LS5, dtype=F64, requires_grad=True)
    xr, zr = x.clone().requires_grad_(True), z.clone().requires_grad_(True)
    k = ao.ARDKernel(base, a, ls).apply(xr, zr)
    gx, gz, ga, gl = torch.autograd.grad((w * k).sum(), [xr, zr, a, ls])
    for t in (gx, gz, ga, gl):
        assert torch.isfinite(t).all()
    L = ls.detach()
    diff = x - z
    r = (diff / L).norm(dim=1)
    kc, C = _coefficient(base, r, a.detach())
    assert rel_err(k, kc) < 1e-14
    dz = (w * C)[:, None] * diff / L ** 2
    assert rel_err(gz, dz) < 1e-13 and rel_err(gx, -dz) < 1e-13
    assert (gz[::8] == 0).all() and (gx[::8] == 0).all()
    assert float(ga) == pytest.approx(float((w * 2 * kc / a.detach()).sum()), rel=1e-13)
    dl = ((w * C)[:, None] * diff ** 2 / L ** 3).sum(0)
    assert rel_err(gl, dl) < 1e-13


@pytest.mark.parametrize("base", [SE, M52])
def test_oracle_ard_reduces_to_isotropic(base):
    """Equal length scales: the isotropic kernel, and sum_f dk/dl_f = dk/dl."""
    g = torch.Generator().manual_seed(2)
    spec_i, spec_a = (base, 3, M32, 2), (base | ARD, 3, M32, 2)
    Fx, Fz = torch.randn(20, 5, generator=g, dtype=F64), torch.randn(11, 5, generator=g, dtype=F64)
    hyp_i = torch.tensor([0.9, 1.7, 1.1, 0.8], dtype=F64)
    hyp_a = torch.tensor([0.9, 1.0, 1.1, 0.8, 1.7, 1.7, 1.7, 1.0, 1.0], dtype=F64)
    assert rel_err(ao.kernel_value(spec_a, Fx, Fz, hyp_a), ao.kernel_value(spec_i, Fx, Fz, hyp_i)) < 1e-15
    G = torch.randn(20, 11, generator=g, dtype=F64)
    ora = ao.ARDOracleBackend()
    _, _, hi = ora.kernel_bwd(spec_i, Fx, Fz, hyp_i, G)
    _, _, ha = ora.kernel_bwd(spec_a, Fx, Fz, hyp_a, G)
    assert float(ha[1]) == 0.0 and (ha[7:] == 0).all()              # the slots an ARD spec does not read
    assert float(ha[4:7].sum()) == pytest.approx(float(hi[1]), rel=1e-12)
    assert rel_err(ha[[0, 2, 3]], hi[[0, 2, 3]]) < 1e-12


@pytest.fixture
def ard_oracle_backend():
    """The float64 CPU stand-in backend with the ARD flag (tests/ard_oracle.py)."""
    old = backend.set_backend_for_tests(ao.ARDOracleBackend())
    yield
    backend.set_backend_for_tests(old)


def _check_step(kinds, length_scale, dims=(4, 4), N=500, M=48, L=3, Z_on_data=False, amplitude=(0.9, 1.1)):
    cfg = configs.sweep_inputs(N, M, L)
    if Z_on_data:
        cfg["ctor"]["initial_inducing_points"] = cfg["aux"][::N // M][:M].numpy().copy()
    da, db = dims
    s = pkg.productSVGP(**dict(cfg["ctor"], dim_a=da, dim_b=db), kind_a=kinds[0], kind_b=kinds[1], amplitude=amplitude,
                        length_scale=length_scale)
    spec, hyp = s._spec(), s._hyp().detach()
    assert hyp.numel() == 4 + da + db
    o = ao.ContinuousProduct(cfg["ctor"]["initial_inducing_points"], hyp, spec, cfg["ctor"]["jitter"], cfg["ctor"]["N_train"])
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
    return spec, g1


LS4A, LS4B = [0.5, 1.3, 4.2, 0.9], [2.0, 0.6, 1.1, 5.0]


@pytest.mark.parametrize("kinds,length_scale", [(("se", "se"), (LS4A, LS4B)), (("matern52", "se"), (LS4A, 1.2)),
                                                (("matern32", "matern12"), (0.9, LS4B)), (("se", "linear"), (LS4A, 1.0))])
def test_step_ard_against_streamlined_oracle(ard_oracle_backend, kinds, length_scale):
    spec, g1 = _check_step(kinds, length_scale)
    dh = g1[3]
    for i in range(2):                                    # an ARD block's isotropic slot and an isotropic block's l_f
        if np.ndim(length_scale[i]):
            assert float(dh[2 * i + 1]) == 0.0
        else:
            assert (dh[4 + 4 * i:8 + 4 * i] == 0).all()


def test_step_ard_inducing_points_on_data_points(ard_oracle_backend):
    _, g1 = _check_step(("matern12", "matern52"), (LS4A, LS4B), Z_on_data=True)
    assert torch.isfinite(g1[2]).all() and g1[2].abs().max() > 0


def test_productsvgp_ard_layout():
    cfg = configs.sweep_inputs(10, 4, 1)
    c = dict(cfg["ctor"], dim_a=1, dim_b=3)
    s = pkg.productSVGP(**c, kind_a="matern32", kind_b="matern52", amplitude=(0.9, 1.1), length_scale=(10.0, [0.5, 0.5, 2.0]))
    assert s._spec() == (M32, 1, M52 | ARD, 3)
    assert s._hyp().detach().tolist() == pytest.approx([0.9, 10.0, 1.1, 1.0, 1.0, 0.5, 0.5, 2.0])
    assert s._hyp().requires_grad
    s = pkg.productSVGP(**dict(cfg["ctor"]), kind_a="se", kind_b="se", length_scale=(np.array([1, 2, 3, 4.0]), 0.5))
    assert s._spec() == (SE | ARD, 4, SE, 4)
    assert s._hyp().numel() == 12


def test_productsvgp_isotropic_unchanged():
    cfg = configs.sweep_inputs(10, 4, 1)
    s = pkg.productSVGP(**cfg["ctor"], kind_a="matern52", kind_b="se", amplitude=(0.9, 1.1), length_scale=(1.3, 0.8))
    assert s._spec() == (M52, 4, SE, 4)
    assert s._hyp().detach().tolist() == pytest.approx([0.9, 1.3, 1.1, 0.8])
    assert pkg.productSVGP(**cfg["ctor"])._hyp().numel() == 4


def test_productsvgp_ard_validation():
    cfg = configs.sweep_inputs(10, 4, 1)
    c = cfg["ctor"]
    with pytest.raises(ValueError):
        pkg.productSVGP(**c, kind_a="se", length_scale=([1.0, 2.0, 3.0], 1.0))            # dim_a = 4
    with pytest.raises(ValueError):
        pkg.productSVGP(**c, kind_b="matern32", length_scale=(1.0, [1.0] * 5))
    for kind in ("linear", "cosine", "expsin"):
        with pytest.raises(ValueError):
            pkg.productSVGP(**c, kind_b=kind, length_scale=(1.0, [1.0] * 4))
    with pytest.raises(ValueError):
        pkg.productSVGP(**dict(c, dim_a=8, dim_b=0), kind_b="none", length_scale=(1.0, []))
    with pytest.raises(KeyError):
        pkg.productSVGP(**c, kind_b="expsin")                                           # no such kind, as before
