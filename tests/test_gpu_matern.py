"""Matern factors (SVGP_K_MATERN12 / 32 / 52) on the B200: every K1 variant against the float64 oracle backend, the
integer digit-plane builder, the r = 0 adjoints, and the whole step against the float64 oracle.

Tolerances are those of the SE-family tests they mirror: test_gpu_primitives.py::test_kernel_fwd_bwd,
test_gpu_i8_engine.py::test_kplanes_reassemble and test_gpu_fullsize.py (1e-4, north_star, for all ten quantities).
"""
import os
import sys

import pytest
import torch

import refs
from conftest import rel_err
from matern_oracle import ContinuousProduct, MaternOracleBackend, kernel_value
import svgp_vae_b200 as pkg
from svgp_vae_b200 import configs

pytestmark = pytest.mark.gpu
ORA = MaternOracleBackend()
M12, M32, M52, NONE, EXPSIN, LINEAR = 5, 6, 7, 0, 2, 3
SPECS = {
    "m12_m12": (M12, 4, M12, 4),
    "m32_none": (M32, 3, NONE, 0),
    "m52_m52": (M52, 4, M52, 4),
    "m52_linear": (M52, 4, LINEAR, 8),
    "m32_expsin": (M32, 4, EXPSIN, 1),
}


def _feat(spec, N, M, seed=0):
    g = torch.Generator().manual_seed(seed)
    d = spec[1] + spec[3]
    Fx, Fz = torch.randn(N, d, generator=g), torch.randn(M, d, generator=g)
    hyp = torch.tensor([0.9, 1.3, 1.1, 0.8])
    return Fx, Fz, hyp


@pytest.mark.parametrize("name", list(SPECS))
@pytest.mark.parametrize("shape", [(1, 1), (37, 15), (300, 72), (1000, 130)])
def test_matern_kernel_fwd_bwd(cuda_backend, name, shape):
    """fp32 K, the fp16 planes and their transpose, kernel_bwd, and the diagonal forward and adjoint."""
    be, spec = cuda_backend, SPECS[name]
    N, M = shape
    Fx, Fz, hyp = _feat(spec, N, M)
    ref = kernel_value(spec, Fx, Fz, hyp)
    kop = be.kernel_fwd(spec, Fx.cuda(), Fz.cuda(), hyp.cuda())
    assert rel_err(kop.K, ref) < 5e-6
    kopt = be.kernel_fwd(spec, Fx.cuda(), Fz.cuda(), hyp.cuda(), tc=True, i8=False)
    floor = 2.0 ** -24 * float(kopt.kscale[1])
    refc = ref.cuda()
    assert float((kopt.value().double() - refc).abs().max()) < 5e-6 * float(refc.abs().max()) + floor
    Kt = kopt.value_t()
    assert float((Kt.double() - refc.t()).abs().max()) < 5e-6 * float(refc.abs().max()) + floor
    assert float(kopt.value().abs().max() * kopt.kscale[0]) < 2 ** 14 + 1
    G = torch.randn(N, M, generator=torch.Generator().manual_seed(1))
    rx, rz, rh = ORA.kernel_bwd(spec, Fx, Fz, hyp, G)
    dx, dz, dh = be.kernel_bwd(spec, Fx.cuda(), Fz.cuda(), hyp.cuda(), G.cuda())
    assert rel_err(dx, rx) < 2e-5 and rel_err(dz, rz) < 2e-5
    if rh.abs().max() > 0:
        assert rel_err(dh, rh) < 2e-5
    Fy = torch.randn(N, spec[1] + spec[3], generator=torch.Generator().manual_seed(2))
    kd = be.kernel_diag_fwd(spec, Fx.cuda(), Fy.cuda(), hyp.cuda())
    assert rel_err(kd, kernel_value(spec, Fx, Fy, hyp, pairwise=False)) < 5e-6
    g = torch.randn(N, generator=torch.Generator().manual_seed(3))
    ex, ey, eh = ORA.kernel_diag_bwd(spec, Fx, Fy, hyp, g)
    fx, fy, fh = be.kernel_diag_bwd(spec, Fx.cuda(), Fy.cuda(), hyp.cuda(), g.cuda())
    assert rel_err(fx, ex) < 2e-5 and rel_err(fy, ey) < 2e-5
    if eh.abs().max() > 0:
        assert rel_err(fh, eh) < 2e-5


@pytest.mark.parametrize("spec", [(M12, 4, M12, 4), (M52, 4, M52, 4)])
@pytest.mark.parametrize("N,M", [(4096, 256), (5000, 320)])
def test_matern_kplanes_reassemble(cuda_backend, spec, N, M):
    """The integer tensor-core operand format (svgp_kernel_fwd_i8) of a Matern product: row- and column-scaled digit
    planes within 0.51 unit of their grids, identical wherever both grids hold the entry, fp16 row planes, zero pads."""
    be = cuda_backend
    cfg = configs.sweep_inputs(N, M, 2, device="cuda")
    Z = torch.from_numpy(cfg["ctor"]["initial_inducing_points"]).float().cuda()
    hyp = torch.ones(4, device="cuda")
    kop = be.kernel_fwd(spec, cfg["aux"].float().contiguous(), Z.contiguous(), hyp, tc=True, i8=True)
    K = kernel_value(spec, cfg["aux"], Z, hyp)
    Kr, Kc = kop.value_i8("r"), kop.value_i8("c")
    unit_r, unit_c = K.abs().amax(1, keepdim=True) / 2.0 ** 29, K.abs().amax(0, keepdim=True) / 2.0 ** 29
    assert ((Kr - K).abs() <= 1e-7 * K.abs() + 0.51 * unit_r).all()
    assert ((Kc - K).abs() <= 1e-7 * K.abs() + 0.51 * unit_c).all()
    assert kop.Kr[0].int().abs().max() <= 127 and kop.Kc[0].int().abs().max() <= 127
    big = (K.abs() * 64 >= K.abs().amax(1, keepdim=True)) & (K.abs() * 64 >= K.abs().amax(0, keepdim=True))
    assert big.any() and (Kr[big] == Kc[big]).all()
    assert rel_err(kop.value(), K) < 2e-6
    assert (kop.Kr[:, :, M:] == 0).all() and (kop.Kc.permute(0, 1, 3, 2).reshape(4, -1, M)[:, N:] == 0).all()


@pytest.mark.parametrize("t", [M12, M32, M52])
def test_matern_adjoints_at_distance_zero(cuda_backend, t):
    """kernel_bwd(Fz, Fz) (the K_mm adjoint: r = 0 on the diagonal) and kernel_diag_bwd(Fx, Fx) (the kappa adjoint: r = 0
    everywhere) are finite and match the oracle, whose zero gradient at r = 0 is the convention of the header."""
    be, spec = cuda_backend, (t, 4, t, 4)
    Fx, Fz, hyp = _feat(spec, 300, 130)
    G = torch.randn(130, 130, generator=torch.Generator().manual_seed(1))
    rx, rz, rh = ORA.kernel_bwd(spec, Fz, Fz, hyp, G)
    dx, dz, dh = be.kernel_bwd(spec, Fz.cuda(), Fz.cuda(), hyp.cuda(), G.cuda())
    for a in (dx, dz, dh):
        assert torch.isfinite(a).all()
    assert rel_err(dx, rx) < 2e-5 and rel_err(dz, rz) < 2e-5 and rel_err(dh, rh) < 2e-5
    # a cotangent on the diagonal alone (r = 0 only): the feature gradients are zero on each side, up to the rounding of
    # C x_f - C z_f for nu = 3/2, 5/2 (exactly zero for 1/2, where C = 0)
    D = torch.diag(torch.randn(130, generator=torch.Generator().manual_seed(4)))
    dx0, dz0, _ = be.kernel_bwd(spec, Fz.cuda(), Fz.cuda(), hyp.cuda(), D.cuda())
    bound = 1e-5 * float(D.abs().max())
    assert float(dx0.abs().max()) < bound and float(dz0.abs().max()) < bound
    if t == M12:
        assert (dx0 == 0).all() and (dz0 == 0).all()
    g = torch.randn(300, generator=torch.Generator().manual_seed(3))
    kd = be.kernel_diag_fwd(spec, Fx.cuda(), Fx.cuda(), hyp.cuda())
    assert rel_err(kd, torch.full((300,), float((hyp[0] * hyp[2]) ** 2))) < 1e-6
    ex, ey, eh = ORA.kernel_diag_bwd(spec, Fx, Fx, hyp, g)
    fx, fy, fh = be.kernel_diag_bwd(spec, Fx.cuda(), Fx.cuda(), hyp.cuda(), g.cuda())
    for a in (fx, fy, fh):
        assert torch.isfinite(a).all()
    assert (ex == 0).all() and (ey == 0).all()
    bound = 1e-5 * float(g.abs().max())
    assert float(fx.abs().max()) < bound and float(fy.abs().max()) < bound
    assert rel_err(fh, eh) < 2e-5


@pytest.mark.parametrize("n,m,l,kinds", [(262144, 1024, 8, ("matern52", "matern52")),
                                         (32768, 2048, 2, ("matern32", "matern12"))])
def test_matern_step_against_float64_oracle_on_the_gpu(cuda_backend, n, m, l, kinds):
    """The whole step on the tensor-core path against the streamlined float64 oracle evaluated on the GPU
    (tests/probes/parity_fullsize_matern.py): all ten quantities within 1e-4."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "probes"))
    import parity_fullsize_matern
    o = parity_fullsize_matern.run(n, m, l, kinds)
    print(o)
    for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l", "KL_term", "dy", "dnoise", "dhyp", "dZ"):
        assert o[k] < 1e-4, (k, o)


@pytest.mark.parametrize("kinds", [("matern12", "matern12"), ("matern52", "matern32")])
def test_matern_step_with_inducing_points_on_data_points(cuda_backend, kinds):
    """One small SIMT-path step with Z initialised as data rows (r = 0 in K_nm and on the diagonal of K_mm): finite, and
    every value and gradient within 1e-4 of the streamlined float64 oracle."""
    N, M, L = 2048, 128, 3
    cfg = configs.sweep_inputs(N, M, L)
    Z = cfg["aux"][::N // M][:M].numpy().copy()
    hyp = (0.9, 1.3, 1.1, 0.8)
    s = pkg.productSVGP(**dict(cfg["ctor"], initial_inducing_points=Z), kind_a=kinds[0], kind_b=kinds[1],
                        amplitude=hyp[0::2], length_scale=hyp[1::2]).cuda()
    o = ContinuousProduct(Z, hyp, s._spec(), cfg["ctor"]["jitter"], cfg["ctor"]["N_train"])
    r0, J0, g0 = refs.streamlined_objective(o, [o.inducing_index_points, o.hyp], cfg["aux"], cfg["y"], cfg["noise"])
    r1, J1, g1 = refs.product_objective(s, [s.inducing_index_points, s._hyp()], cfg["aux"].cuda(), cfg["y"].cuda(),
                                        cfg["noise"].cuda(), tc=False)
    assert rel_err(r1["p_m"], r0["p_m"]) < 1e-4 and rel_err(r1["p_v"], r0["p_v"]) < 1e-4
    for k in ("inside_elbo_recon", "inside_elbo_kl", "ce_term", "KL_term"):
        assert abs(float(r1[k]) - float(r0[k])) <= 1e-4 * abs(float(r0[k])), k
    for name, a, b in zip(["dy", "dnoise", "dZ", "dhyp"], g0, g1):
        assert torch.isfinite(b).all(), name
        assert rel_err(b, a) < 1e-4, (name, rel_err(b, a))
