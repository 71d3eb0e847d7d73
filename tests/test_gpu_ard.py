"""ARD length scales (SVGP_K_ARD) on the B200: every K1 variant against the float64 oracle backend, the integer
digit-plane builder, the SE44 fast path against the generic adjoint, the reduction to the isotropic kernel, the r = 0
adjoints, the whole step against the float64 oracle, and posterior_predict.

Tolerances are those of the tests they mirror: test_gpu_matern.py::test_matern_kernel_fwd_bwd,
test_gpu_matern.py::test_matern_kplanes_reassemble and test_gpu_matern.py (1e-4 for all ten quantities of the step).
"""
import os
import sys

import pytest
import torch

import refs
from ard_oracle import ARDOracleBackend, ContinuousProduct, kernel_value
from conftest import rel_err
import svgp_vae_b200 as pkg
from svgp_vae_b200 import configs

pytestmark = pytest.mark.gpu
ORA = ARDOracleBackend()
SE, M12, M32, M52, NONE, LINEAR, ARD = 1, 5, 6, 7, 0, 3, 16
SPECS = {
    "se_se44": (SE | ARD, 4, SE | ARD, 4),          # the SE44 fast path
    "m52_se": (M52 | ARD, 3, SE, 2),
    "m12_none": (M12 | ARD, 3, NONE, 0),
    "se_linear": (SE | ARD, 4, LINEAR, 8),
}
# distinct per-feature length scales spanning ~10x (an isotropic block's entries are 1, as productSVGP writes them)
LS = [0.35, 2.9, 1.3, 0.6, 3.5, 0.8, 0.45, 1.7]


def _hyp(spec):
    ta, da, tb, db = spec
    ls = [LS[f] if (ta if f < da else tb) & ARD else 1.0 for f in range(da + db)]
    return torch.tensor([0.9, 1.3, 1.1, 0.8] + ls)


def _feat(spec, N, M, seed=0):
    g = torch.Generator().manual_seed(seed)
    d = spec[1] + spec[3]
    return torch.randn(N, d, generator=g), torch.randn(M, d, generator=g), _hyp(spec)


def _unread(spec):
    """dhyp slots the spec does not read: exactly 0."""
    ta, da, tb, db = spec
    out = [2 * i + 1 for i, t in enumerate((ta, tb)) if t & ARD]
    return out + [4 + f for f in range(da + db) if not ((ta if f < da else tb) & ARD)]


@pytest.mark.parametrize("name", list(SPECS))
@pytest.mark.parametrize("shape", [(1, 1), (37, 15), (300, 72), (1000, 130)])
def test_ard_kernel_fwd_bwd(cuda_backend, name, shape):
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
    assert dh.shape == hyp.shape
    assert rel_err(dx, rx) < 2e-5 and rel_err(dz, rz) < 2e-5
    assert rel_err(dh, rh) < 2e-5
    assert (dh[_unread(spec)] == 0).all()
    Fy = torch.randn(N, spec[1] + spec[3], generator=torch.Generator().manual_seed(2))
    kd = be.kernel_diag_fwd(spec, Fx.cuda(), Fy.cuda(), hyp.cuda())
    assert rel_err(kd, kernel_value(spec, Fx, Fy, hyp, pairwise=False)) < 5e-6
    g = torch.randn(N, generator=torch.Generator().manual_seed(3))
    ex, ey, eh = ORA.kernel_diag_bwd(spec, Fx, Fy, hyp, g)
    fx, fy, fh = be.kernel_diag_bwd(spec, Fx.cuda(), Fy.cuda(), hyp.cuda(), g.cuda())
    assert rel_err(fx, ex) < 2e-5 and rel_err(fy, ey) < 2e-5
    assert rel_err(fh, eh) < 2e-5
    assert (fh[_unread(spec)] == 0).all()


@pytest.mark.parametrize("spec", [SPECS["se_se44"], (M52 | ARD, 4, M32, 4)])
@pytest.mark.parametrize("N,M", [(4096, 256), (5000, 320)])
def test_ard_kplanes_reassemble(cuda_backend, spec, N, M):
    """The integer tensor-core operand format (svgp_kernel_fwd_i8) of an ARD product -- the SE44 builder and the generic
    one: row- and column-scaled digit planes within 0.51 unit of their grids, identical wherever both grids hold the
    entry, fp16 row planes, zero pads."""
    be = cuda_backend
    cfg = configs.sweep_inputs(N, M, 2, device="cuda")
    Z = torch.from_numpy(cfg["ctor"]["initial_inducing_points"]).float().cuda()
    hyp = _hyp(spec)
    hyp[:4] = 1.0
    hyp = hyp.cuda()
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


def _bwd_both_paths(be, spec, Fx, Fz, hyp, G, monkeypatch):
    fast = be.kernel_bwd(spec, Fx, Fz, hyp, G, need_x=False)
    with monkeypatch.context() as m:
        m.setenv("SVGP_K1_BWD_GENERIC", "1")
        generic = be.kernel_bwd(spec, Fx, Fz, hyp, G, need_x=False)
    return fast, generic


def test_ard_se44_fast_and_generic_paths_agree(cuda_backend, monkeypatch):
    """SE|ARD x SE|ARD on [4 | 4]: kernel_bwd_z_se44_kernel<true> and the generic Z pass give the same dFz and dhyp,
    and both match the oracle."""
    be, spec = cuda_backend, SPECS["se_se44"]
    Fx, Fz, hyp = _feat(spec, 3000, 200, seed=5)
    G = torch.randn(3000, 200, generator=torch.Generator().manual_seed(6))
    _, rz, rh = ORA.kernel_bwd(spec, Fx, Fz, hyp, G)
    (_, zf, hf), (_, zg, hg) = _bwd_both_paths(be, spec, Fx.cuda(), Fz.cuda(), hyp.cuda(), G.cuda(), monkeypatch)
    assert rel_err(zf, zg) < 2e-5 and rel_err(hf, hg) < 2e-5
    for z, h in ((zf, hf), (zg, hg)):
        assert rel_err(z, rz) < 2e-5 and rel_err(h, rh) < 2e-5
        assert (h[_unread(spec)] == 0).all()


@pytest.mark.parametrize("base,dims", [(SE, (4, 4)), (M52, (4, 4)), (SE, (3, 2))])
def test_ard_reduces_to_isotropic(cuda_backend, monkeypatch, base, dims):
    """Every l_f = l: K (fp32, fp16 planes, integer planes) matches the isotropic spec and sum_f dl_f the isotropic dl,
    on the SE44 path and on the generic one."""
    be = cuda_backend
    spec_i, spec_a = (base, dims[0], base, dims[1]), (base | ARD, dims[0], base | ARD, dims[1])
    d = sum(dims)
    g = torch.Generator().manual_seed(7)
    Fx, Fz = torch.randn(2500, d, generator=g).cuda(), torch.randn(190, d, generator=g).cuda()
    hyp_i = torch.tensor([0.9, 1.4, 1.1, 0.7]).cuda()
    hyp_a = torch.tensor([0.9, 1.0, 1.1, 1.0] + [1.4] * dims[0] + [0.7] * dims[1]).cuda()
    assert rel_err(be.kernel_fwd(spec_a, Fx, Fz, hyp_a).K, be.kernel_fwd(spec_i, Fx, Fz, hyp_i).K) < 2e-6
    for i8 in (False, True):
        ka = be.kernel_fwd(spec_a, Fx, Fz, hyp_a, tc=True, i8=i8)
        ki = be.kernel_fwd(spec_i, Fx, Fz, hyp_i, tc=True, i8=i8)
        assert rel_err(ka.value(), ki.value()) < 2e-6
    G = torch.randn(2500, 190, generator=g).cuda()
    (_, zaf, haf), (_, zag, hag) = _bwd_both_paths(be, spec_a, Fx, Fz, hyp_a, G, monkeypatch)
    (_, zif, hif), (_, zig, hig) = _bwd_both_paths(be, spec_i, Fx, Fz, hyp_i, G, monkeypatch)
    for za, ha, zi, hi in ((zaf, haf, zif, hif), (zag, hag, zig, hig)):
        assert rel_err(za, zi) < 2e-5
        assert float(ha[1]) == 0.0 and float(ha[3]) == 0.0
        iso = torch.stack([ha[0], ha[4:4 + dims[0]].sum(), ha[2], ha[4 + dims[0]:].sum()])
        assert rel_err(iso, hi) < 2e-5


@pytest.mark.parametrize("t", [M12, M32, M52])
def test_ard_matern_adjoints_at_distance_zero(cuda_backend, t):
    """kernel_bwd(Fz, Fz) (the K_mm adjoint: r = 0 on the diagonal) and kernel_diag_bwd(Fx, Fx) (the kappa adjoint: r = 0
    everywhere) of an ARD Matern product are finite and match the oracle."""
    be, spec = cuda_backend, (t | ARD, 4, t | ARD, 4)
    Fx, Fz, hyp = _feat(spec, 300, 130)
    G = torch.randn(130, 130, generator=torch.Generator().manual_seed(1))
    rx, rz, rh = ORA.kernel_bwd(spec, Fz, Fz, hyp, G)
    dx, dz, dh = be.kernel_bwd(spec, Fz.cuda(), Fz.cuda(), hyp.cuda(), G.cuda())
    for a in (dx, dz, dh):
        assert torch.isfinite(a).all()
    assert rel_err(dx, rx) < 2e-5 and rel_err(dz, rz) < 2e-5 and rel_err(dh, rh) < 2e-5
    D = torch.diag(torch.randn(130, generator=torch.Generator().manual_seed(4)))
    dx0, dz0, dh0 = be.kernel_bwd(spec, Fz.cuda(), Fz.cuda(), hyp.cuda(), D.cuda())
    bound = 1e-5 * float(D.abs().max())
    assert float(dx0.abs().max()) < bound and float(dz0.abs().max()) < bound
    assert (dh0[4:] == 0).all()                                    # (x_f - z_f)^2 = 0 on every entry
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
    assert rel_err(fh, eh) < 2e-5 and (fh[4:] == 0).all()


@pytest.mark.parametrize("n,m,l,kinds", [(262144, 1024, 8, ("se", "se")), (32768, 2048, 2, ("matern52", "matern32"))])
def test_ard_step_against_float64_oracle_on_the_gpu(cuda_backend, n, m, l, kinds):
    """The whole step on the tensor-core path, both blocks ARD, against the streamlined float64 oracle evaluated on the
    GPU (tests/probes/parity_fullsize_ard.py): all ten quantities within 1e-4 (dhyp over the whole 4 + d vector), and
    the slots the spec does not read exactly 0."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "probes"))
    import parity_fullsize_ard
    o = parity_fullsize_ard.run(n, m, l, kinds)
    print(o)
    for k in ("p_m", "p_v", "recon_l", "kl_l", "ce_l", "KL_term", "dy", "dnoise", "dhyp", "dZ"):
        assert o[k] < 1e-4, (k, o)
    assert o["dhyp_unread"] == [1, 3] and all(o["dhyp_slots"][j] == 0.0 for j in o["dhyp_unread"])


def test_ard_step_with_inducing_points_on_data_points(cuda_backend):
    """One small SIMT-path step with Z initialised as data rows (r = 0 in K_nm and on the diagonal of K_mm), ARD Matern
    1/2 x ARD SE: finite, and every value and gradient within 1e-4 of the streamlined float64 oracle."""
    N, M, L = 2048, 128, 3
    cfg = configs.sweep_inputs(N, M, L)
    Z = cfg["aux"][::N // M][:M].numpy().copy()
    s = pkg.productSVGP(**dict(cfg["ctor"], initial_inducing_points=Z), kind_a="matern12", kind_b="se",
                        amplitude=(0.9, 1.1), length_scale=(LS[:4], LS[4:])).cuda()
    hyp = s._hyp().detach().cpu()
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
    assert float(g1[3][1]) == 0.0 and float(g1[3][3]) == 0.0


@pytest.mark.parametrize("n", [2048, 20000])
def test_ard_posterior_predict(cuda_backend, n):
    """predict.posterior_predict of an ARD model (SIMT and tensor-core sizes) against its float64 restatement on the
    oracle's kernel matrices."""
    M, L, T = 192, 3, 300
    cfg = configs.sweep_inputs(n, M, L)
    s = pkg.productSVGP(**cfg["ctor"], kind_a="matern52", kind_b="se", length_scale=(LS[:4], LS[4:])).cuda()
    spec, hyp = s._spec(), s._hyp().detach().cpu().double()
    X = cfg["aux"].double()
    Xt = X[:T] + 0.1 * torch.randn(T, 8, generator=torch.Generator().manual_seed(8), dtype=torch.float64)
    means, vars_ = cfg["y"].double(), cfg["noise"].double()
    Z = torch.from_numpy(cfg["ctor"]["initial_inducing_points"]).double()
    K_nm, K_mm, K_xm = kernel_value(spec, X, Z, hyp), kernel_value(spec, Z, Z, hyp), kernel_value(spec, Xt, Z, hyp)
    K_xx = kernel_value(spec, Xt, Xt, hyp, pairwise=False)
    eye = torch.eye(M, dtype=torch.float64)
    c, jit = s.N_train / float(n), s.jitter
    p = 1.0 / vars_
    K_inv = torch.linalg.inv(K_mm + jit * eye)
    pm0, pv0 = [], []
    for l in range(L):
        S = torch.linalg.inv(K_mm + c * K_nm.T @ (p[:, l:l + 1] * K_nm) + jit * eye)
        w = c * S @ (K_nm.T @ (p[:, l] * means[:, l]))
        pm0.append(K_xm @ w)
        pv0.append(K_xx - ((K_xm @ K_inv) * K_xm).sum(1) + ((K_xm @ S) * K_xm).sum(1))
    pm0, pv0 = torch.stack(pm0, 1), torch.stack(pv0, 1)
    pm, pv = pkg.posterior_predict(s, Xt.float().cuda(), cfg["aux"].cuda(), cfg["y"].cuda(), cfg["noise"].cuda())
    assert rel_err(pm, pm0) < 1e-4 and rel_err(pv, pv0) < 1e-4
