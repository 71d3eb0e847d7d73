"""Pin the oracle (CPU).  The reference has no tests or golden vectors for this path (SURVEY section 4), so the
oracle is anchored by: an independent kernel implementation (scikit-learn), literal == streamlined, the
exact-GP limit against the independent formulation of GPVAE_Pearce_model.py:49-84, the survey-session
numbers of SURVEY App. B (a separately written restatement), and committed golden vectors."""
import math
import os

import numpy as np
import pytest
import torch

import refs
from conftest import GOLDEN, MNIST_FIXTURE
from oracle import svgp_literal as lit
from oracle import svgp_streamlined as st
from oracle import tfp_kernels as tfk
from svgp_vae_b200 import configs

F64 = torch.float64


def test_kernels_against_sklearn():
    from sklearn.gaussian_process.kernels import RBF, ConstantKernel, DotProduct, ExpSineSquared
    g = torch.Generator().manual_seed(0)
    x, z = torch.randn(17, 5, generator=g, dtype=F64), torch.randn(9, 5, generator=g, dtype=F64)
    amp, ls = 0.7, 1.9
    t_amp, t_ls = torch.tensor(amp, dtype=F64), torch.tensor(ls, dtype=F64)
    ref = (ConstantKernel(amp ** 2) * RBF(ls))(x.numpy(), z.numpy())
    assert np.allclose(tfk.ExponentiatedQuadratic(t_amp, t_ls).matrix(x, z).numpy(), ref, rtol=1e-12)
    ref = (ConstantKernel(amp ** 2) * ExpSineSquared(length_scale=ls, periodicity=2 * math.pi))(x[:, :1].numpy(), z[:, :1].numpy())
    mine = tfk.ExpSinSquared(t_amp, t_ls, 2 * math.pi).matrix(x[:, :1], z[:, :1]).numpy()
    assert np.allclose(mine, ref, rtol=1e-12)
    assert np.allclose(tfk.Linear().matrix(x, z).numpy(), DotProduct(sigma_0=0.0)(x.numpy(), z.numpy()), rtol=1e-12)
    # .apply is the diagonal of .matrix
    k = tfk.ExpSinSquared(t_amp, t_ls, 2 * math.pi)
    assert torch.allclose(k.apply(x[:9, :1], z[:, :1]), torch.diagonal(k.matrix(x[:9, :1], z[:, :1])))


def test_survey_appendix_B1_B3_numbers():
    """SURVEY App. B1 / B3 (recipe R): values written down by the survey's own, independent restatement."""
    expect = {False: (-9619.35036449, 496.25435500, -9619.35036741, -48.1282521670,
                      (14.5026795, 53.1452734, 203.118041, 80.8026728, 44.3894938, 42.3267932)),
              True: (-1320.46166054, 352.14193847, -1320.46164688, -22.1619697264,
                     (14.4125131, 52.1874378, 23.7834950, 16.9112534, 1.22838319, 4.94716140))}
    for norm, (rec, kl, ce, J, gnorms) in expect.items():
        cfg = configs.mnist_inputs(MNIST_FIXTURE, L=4, normalize=norm)
        o, _, op, _ = refs.make_pair("mnist", cfg, "cpu")
        r, Jo, g = refs.oracle_objective(o, op, cfg["aux"], cfg["y"], cfg["noise"])
        assert abs(float(r["inside_elbo_recon"]) - rec) < 1e-7 * abs(rec)
        assert abs(float(r["inside_elbo_kl"]) - kl) < 1e-7 * abs(kl)
        assert abs(float(r["ce_term"]) - ce) < 1e-7 * abs(ce)
        assert abs(float(Jo) - J) < 1e-8 * abs(J)
        for t, n in zip(g, gnorms):
            assert abs(float(t.norm()) - n) < 1e-6 * n
        assert float(g[2][:, 0].abs().max()) == 0.0                # unused id column of the inducing points
        assert int((g[3].abs().sum(1) > 0).sum()) == 16            # exactly 16 table rows touched (ids 360..375)
    # B1 per-channel values, L = 2
    cfg = configs.mnist_inputs(MNIST_FIXTURE, L=2)
    o, _, op, _ = refs.make_pair("mnist", cfg, "cpu")
    r = lit.minibatch_glue(o, cfg["aux"], cfg["y"], cfg["noise"])
    assert np.allclose(r["recon_l"].numpy(), [-2337.5041005553, -2513.6756105578], rtol=1e-11)
    assert np.allclose(r["kl_l"].numpy(), [122.5932406250, 125.8693471589], rtol=1e-10)
    assert abs(float(r["inside_elbo"]) + 4866.8850006125) < 1e-7
    assert np.allclose(r["p_m"][:2, 0].numpy(), [0.3355118621, 0.5579539230], rtol=1e-9)


def test_survey_appendix_B2_ball():
    T, Bn = 30, 35
    t = torch.arange(T, dtype=F64)[None, :]
    b = torch.arange(Bn, dtype=F64)[:, None]
    y = torch.sin(0.3 * t + 0.7 * b)
    noise = 0.02 + 0.1 * (1 + torch.cos(0.5 * t + b))
    x = (t + 1.0).repeat(Bn, 1)
    s = lit.BallSVGP(False, 15, True, 1, 30, 2.0, True, "x", 1e-9, 1, 30, 2.0)
    mean, B, mu_hat, A_hat = s.approximate_posterior_params(x, y, noise)
    assert mean.shape == (35, 30) and B.shape == (35, 30, 30) and mu_hat.shape == (35, 15) and A_hat.shape == (35, 15, 15)
    # The survey's probe used a float64 inducing grid; the reference builds it with np.linspace(dtype=float32)
    # (SVGPVAE_model.py:46), which the oracle now follows (pinned by reference_golden.npz): agreement is ~1e-7.
    assert np.allclose(mean[0, :3].numpy(), [0.0575036480, 0.2709499525, 0.5303067273], rtol=2e-6)
    assert np.allclose(torch.diagonal(B[0])[:3].numpy(), [0.1291471822, 0.0866073092, 0.0658024436], rtol=2e-6)
    L3, KL = s.variational_loss(x, y, noise, mu_hat, A_hat)
    assert np.allclose(L3[:3].numpy(), [-0.4421172586, 1.1807586738, 2.2101319702], rtol=2e-6)
    assert np.allclose(KL[:3].numpy(), [836.2227133929, 836.1091974550, 836.0499025487], rtol=1e-7)   # the quirky KL
    assert abs(float((L3 - KL).sum()) + 29244.9691106253) < 1e-2


def test_exact_gp_limit():
    """m = T, Z = x, small jitter: the SVGP posterior equals exact GP regression (GPVAE_Pearce_model.py:49-84:
    p_m = K (K + diag s2)^-1 y, p_v = diag(K - K (K + diag s2)^-1 K))."""
    T = 12
    x = (torch.arange(T, dtype=F64) + 1.0)[None, :]
    g = torch.Generator().manual_seed(1)
    y = torch.randn(1, T, generator=g, dtype=F64)
    noise = 0.05 + torch.rand(1, T, generator=g, dtype=F64)
    s = lit.BallSVGP(False, T, True, 1, T, 1.0, True, "x", 1e-10, 1, T, 1.0)
    mean, B, _, _ = s.approximate_posterior_params(x, y, noise)
    K = tfk.ExponentiatedQuadratic(None, torch.tensor(1.0, dtype=F64)).matrix(x[0][:, None], x[0][:, None])
    G = torch.linalg.inv(K + torch.diag(noise[0]))
    assert torch.allclose(mean[0], K @ G @ y[0], atol=1e-6)
    assert torch.allclose(torch.diagonal(B[0]), torch.diagonal(K - K @ G @ K), atol=1e-6)


@pytest.mark.parametrize("kind,maker,clip", [
    ("mnist", lambda: configs.mnist_inputs(MNIST_FIXTURE, L=3), False),
    ("mnist", lambda: configs.mnist_inputs(MNIST_FIXTURE, L=3, normalize=True, rows="train", b=210, batch_index=15), False),
    ("sprites", lambda: configs.sprites_inputs(M=72, L=3), True),
    ("sprites", lambda: configs.sprites_inputs(M=72, L=3, normalize=False), True),
    ("sweep", lambda: configs.sweep_inputs(300, 40, 2), False),
])
def test_literal_equals_streamlined(kind, maker, clip):
    cfg = maker()
    o, _, op, _ = refs.make_pair(kind, cfg, "cpu")
    aux, y, nz = cfg["aux"].double(), cfg["y"].double(), cfg["noise"].double()
    r = lit.minibatch_glue(o, aux, y, nz, clip_pv=clip)
    Z = o.inducing_index_points
    t = st.streamlined_terms(o.kernel_matrix(aux, Z, x_inducing=False), o.kernel_matrix(Z, Z),
                             o.kernel_matrix(aux, aux, False, False, True), y, nz, o.N_train, o.jitter, clip_pv=clip)
    g = st.glue_from_terms(t, float(aux.shape[0]), o.N_train)
    assert torch.allclose(t["p_m"], r["p_m"], rtol=1e-9, atol=1e-11) and torch.allclose(t["p_v"], r["p_v"], rtol=1e-9, atol=1e-11)
    for k in ("inside_elbo_recon", "inside_elbo_kl", "ce_term"):
        assert abs(float(g[k]) - float(r[k])) < 1e-10 * abs(float(r[k]))
    assert abs(float(g["KL_term"]) - float(r["KL_term"])) < 1e-8 * abs(float(r["KL_term"]))
    assert torch.allclose(t["mu_hat"], r["mu_hat"], rtol=1e-9, atol=1e-12) and torch.allclose(t["A_hat"], r["A_hat"], rtol=1e-9, atol=1e-12)


def test_oracle_reproduces_committed_golden_vectors():
    gold = np.load(os.path.join(GOLDEN, "golden_outputs.npz"))
    cfg = configs.mnist_inputs(MNIST_FIXTURE, L=4)
    o, _, op, _ = refs.make_pair("mnist", cfg, "cpu")
    r, J, g = refs.oracle_objective(o, op, cfg["aux"], cfg["y"], cfg["noise"])
    assert np.allclose(r["p_m"].detach().numpy(), gold["mnist/p_m"], rtol=1e-10, atol=1e-13)
    assert np.allclose(r["p_v"].detach().numpy(), gold["mnist/p_v"], rtol=1e-10, atol=1e-13)
    assert np.allclose(g[0].numpy(), gold["mnist/grad_y"], rtol=1e-8, atol=1e-12)
    cfgb = configs.ball_inputs()
    ox, oy = lit.BallSVGP(name="x", **cfgb["ctor"]), lit.BallSVGP(name="y", **cfgb["ctor"])
    rb = lit.ball_glue(ox, oy, cfgb["y"].double(), cfgb["noise"].double())
    assert np.allclose(rb["KL_term"].numpy(), gold["ball/KL_term"], rtol=1e-10)
    # edge cases of the restatement itself
    assert float(lit.recip_no_nan(torch.tensor([0.0, 2.0], dtype=F64))[0]) == 0.0
    assert torch.equal(lit.add_jitter(torch.zeros(2, 3, 3, dtype=F64), 0.5)[1], 0.5 * torch.eye(3, dtype=F64))


# ----------------------------------------------------------------------------------------------------------
# The oracle against the REFERENCE SOURCE: tests/golden/reference_golden.npz holds the outputs of the unmodified
# /root/reference/SVGPVAE_model.py (forward_pass_SVGPVAE, mnistSVGP, spritesSVGP, SVGP) executed under the
# TensorFlow-API shim of tests/golden/tf_shim.py on the same seeded inputs (tests/golden/make_reference_golden.py).
# ----------------------------------------------------------------------------------------------------------
REF_CASES = [
    ("mnist", "mnist", lambda: configs.mnist_inputs(MNIST_FIXTURE, L=4), False, ["Z", "table", "amplitude", "length"]),
    ("mnist_norm", "mnist", lambda: configs.mnist_inputs(MNIST_FIXTURE, L=4, normalize=True), False, ["Z", "table", "amplitude", "length"]),
    ("mnist_train_last", "mnist", lambda: configs.mnist_inputs(MNIST_FIXTURE, L=2, b=210, rows="train", batch_index=15), False,
     ["Z", "table", "amplitude", "length"]),
    ("sprites72", "sprites", lambda: configs.sprites_inputs(M=72, L=4), True, ["Z", "table"]),
    ("sprites72_raw", "sprites", lambda: configs.sprites_inputs(M=72, L=4, normalize=False), True, ["Z", "table"]),
    ("sprites72_se", "sprites", lambda: configs.sprites_inputs(M=72, L=3, K_SE=True), True,
     ["Z", "table", "sigma_action", "l_action", "sigma_character", "l_character"]),
]


def _close(a, b, rtol):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() <= rtol * max(np.abs(b).max(), 1e-300)


@pytest.mark.parametrize("name,kind,maker,clip,pnames", REF_CASES, ids=[c[0] for c in REF_CASES])
def test_oracle_matches_reference_source(name, kind, maker, clip, pnames):
    gold = np.load(os.path.join(GOLDEN, "reference_golden.npz"))
    cfg = maker()
    o, _, op, _ = refs.make_pair(kind, cfg, "cpu")
    r, J, g = refs.oracle_objective(o, op, cfg["aux"], cfg["y"], cfg["noise"], clip_pv=clip)
    assert _close(r["p_m"].detach(), gold[name + "/p_m"], 1e-10)
    assert _close(r["p_v"].detach(), gold[name + "/p_v"], 1e-10)
    sc = gold[name + "/scalars"]
    for k, ref_v in zip(("inside_elbo_recon", "inside_elbo_kl", "ce_term"), sc[:3]):
        assert abs(float(r[k]) - ref_v) <= 1e-11 * abs(ref_v), k
    # KL_term and J are cancelling combinations of the above (SURVEY F11): compare at the scale of their summands
    assert abs(float(r["KL_term"]) - sc[3]) <= 1e-11 * abs(sc[2])
    assert abs(float(J) - sc[4]) <= 1e-11 * abs(sc[2])
    for t, n in zip(g, ["y", "noise"] + pnames):
        ref_g = gold[name + "/grad_" + n]
        assert _close(torch.zeros(1) if t is None else t, ref_g, 1e-8), n
    aux, Z = cfg["aux"].double(), o.inducing_index_points
    assert _close(o.kernel_matrix(aux, Z, x_inducing=False).detach(), gold[name + "/K_nm"], 1e-12)
    assert _close(o.kernel_matrix(aux, aux, False, False, True).detach(), gold[name + "/K_nn_diag"], 1e-12)
    if kind == "mnist":
        y0, n0 = cfg["y"].double()[:, 0], cfg["noise"].double()[:, 0]
        m, B, mu_hat, A_hat = o.approximate_posterior_params(aux, aux, y0, n0)
        L3, KL = o.variational_loss(aux, y0, mu_hat, A_hat, n0)
        assert _close(mu_hat.detach(), gold[name + "/ch0_mu_hat"], 1e-10) and _close(A_hat.detach(), gold[name + "/ch0_A_hat"], 1e-10)
        assert _close(torch.stack([L3, KL]).detach(), gold[name + "/ch0_L3_KL"], 1e-11)


def test_oracle_ball_matches_reference_source():
    gold = np.load(os.path.join(GOLDEN, "reference_golden.npz"))
    cfg = configs.ball_inputs()
    ox, oy = lit.BallSVGP(name="x", **cfg["ctor"]), lit.BallSVGP(name="y", **cfg["ctor"])
    y = cfg["y"].double().requires_grad_(True)
    nz = cfg["noise"].double().requires_grad_(True)
    r = lit.ball_glue(ox, oy, y, nz)
    gm, gv = refs.upstream(tuple(y.shape))
    J = r["KL_term"].sum() + (gm * r["p_m"]).sum() + (gv * r["p_v"]).sum()
    gy, gn = torch.autograd.grad(J, [y, nz])
    for k, gk in (("p_m", "ball/p_m"), ("p_v", "ball/p_v"), ("inside_elbo_recon", "ball/recon"), ("inside_elbo_kl", "ball/kl"),
                  ("B_0", "ball/B_x"), ("mu_hat_0", "ball/mu_hat_x"), ("A_hat_0", "ball/A_hat_x")):
        assert _close(r[k].detach(), gold[gk], 1e-9), k
    assert np.abs(r["KL_term"].detach().numpy() - gold["ball/KL_term"]).max() <= 1e-10 * np.abs(gold["ball/kl"]).max()
    assert abs(float(J) - float(gold["ball/J"][0])) <= 1e-10 * abs(float(gold["ball/J"][0]))
    assert _close(gy, gold["ball/grad_y"], 1e-7) and _close(gn, gold["ball/grad_noise"], 1e-7)


def test_oracle_titsias_matches_reference_source():
    """L_2 (Titsias) branch: SVGPVAE_model.py:246-259 (mini-batched, through forward_pass_SVGPVAE) and :89-101 (ball)."""
    gold = np.load(os.path.join(GOLDEN, "reference_golden.npz"))
    cfg = configs.mnist_inputs(MNIST_FIXTURE, L=2, b=64)
    cfg["ctor"]["titsias"] = True
    o, _, op, _ = refs.make_pair("mnist", cfg, "cpu")
    r, J, g = refs.oracle_objective(o, op, cfg["aux"], cfg["y"], cfg["noise"])
    sc = gold["mnist_titsias/scalars"]
    assert float(r["inside_elbo_kl"]) == 0.0 and sc[1] == 0.0
    assert abs(float(r["inside_elbo_recon"]) - sc[0]) <= 1e-10 * abs(sc[0]) and abs(float(r["KL_term"]) - sc[3]) <= 1e-10 * abs(sc[2])
    for t, n in zip(g, ["y", "noise", "Z", "table", "amplitude", "length"]):
        assert _close(t, gold["mnist_titsias/grad_" + n], 1e-7), n
    cfgb = configs.ball_inputs()
    sb = lit.BallSVGP(name="x", **dict(cfgb["ctor"], titsias=True))
    y, nz = cfgb["y"][:, :, 0].double(), cfgb["noise"][:, :, 0].double()
    x = cfgb["x"].double()
    _, _, mu_hat, A_hat = sb.approximate_posterior_params(x, y, nz)
    L2, _ = sb.variational_loss(x, y, nz, mu_hat, A_hat)
    assert _close(L2, gold["ball_titsias/L2"], 1e-10)


def test_parity_fullsize_kinds_factor_formulas():
    """tests/probes/parity_fullsize_kinds.py builds K_nm, K_mm and kappa from per-block formulas of its own (no (N, M, d)
    tensor, differences rather than the |x|^2 + |z|^2 - 2 x.z expansion): they must equal the oracle formulas
    (oracle_backend / matern_oracle.kernel_value, oracle/tfp_kernels) on every case's features, the time column offset
    by 1e4 included."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "probes"))
    import matern_oracle as mo
    import oracle_backend as ob
    import parity_fullsize_kinds as pk
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
    for case, c in pk.CASES.items():
        X, Z = pk.features(case, 300, 70, "cpu", 5)
        hyp = torch.tensor([0.9, c["ls"][0], 1.1, c["ls"][1]], dtype=torch.float64)
        spec = pk.spec_of(c["kinds"], c["dims"])
        X64, Z64 = X.double(), Z.double()
        assert rel(pk.kern64(X64, Z64, hyp, c["kinds"], c["dims"]), mo.kernel_value(spec, X, Z, hyp)) < 1e-12, case
        assert rel(pk.kern64(Z64, Z64, hyp, c["kinds"], c["dims"]), mo.kernel_value(spec, Z, Z, hyp)) < 1e-12, case
        assert rel(pk.kdiag64(X64, hyp, c["kinds"], c["dims"]), mo.kernel_value(spec, X, X, hyp, pairwise=False)) < 1e-12, case
        if "matern32" not in c["kinds"]:
            assert rel(pk.kern64(X64, Z64, hyp, c["kinds"], c["dims"]), ob.kernel_value(spec, X, Z, hyp)) < 1e-12, case
    # each factor against tfp_kernels directly, the offset time column included
    X, Z = pk.features("time_m32_se", 200, 50, "cpu", 3)
    X64, Z64 = X.double(), Z.double()
    ten = torch.tensor(10.0, dtype=torch.float64)
    assert rel(pk.factor64("se", X64[:, :1], Z64[:, :1], 1.0, ten), tfk.ExponentiatedQuadratic(1.0, ten).matrix(X64[:, :1], Z64[:, :1])) < 1e-12
    assert rel(pk.factor64("se", X64, Z64, 1.3, ten), tfk.ExponentiatedQuadratic(1.3, ten).matrix(X64, Z64)) < 1e-12
    assert rel(pk.factor64("matern32", X64[:, :1], Z64[:, :1], 1.0, ten), mo.MaternThreeHalves(1.0, ten).matrix(X64[:, :1], Z64[:, :1])) < 1e-12
    assert rel(pk.factor64("linear", X64, Z64, 1.0, 1.0), tfk.Linear().matrix(X64, Z64)) < 1e-12
