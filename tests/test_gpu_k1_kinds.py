"""K1 for every factor type at tensor-core sizes against float64 on the device.

Three parts of K1 that the sweep kernel (SE x SE on [4 | 4], centred features) never reaches:

* the adjoint (svgp_kernel_bwd) of every launcher branch -- the SE44 Z pass, the generic pass for SE off [4 | 4], EXPSIN,
  LINEAR, COSINE and the products, the ARD forms and the Matern factors -- at (65536, 1000) (ragged tiles) and
  (262144, 1024), against float64 autograd of the oracle formulas;
* offset features: a time column shifted by 1e3 and 1e4 with l = 10 on its factor.  A Z pass that forms
  dz_f = sum c x_f - z_f sum c from fp32 moments loses 1e-4 there; the per-entry differences do not;
* the integer operand builder (svgp_kernel_fwd_i8) for the kinds whose K has negative entries (LINEAR, COSINE): signed
  leading digits, kscale[6] = 0, and rows / columns of K that are exactly zero (a linear block of zeros).

Bars are those of test_gpu_primitives.py::test_kernel_fwd_bwd (2e-5 per adjoint output, 5e-6 for the fp16 planes) and
test_gpu_i8_engine.py::test_kplanes_reassemble.
"""
import pytest
import torch

from ard_oracle import kernel_value
from conftest import rel_err

pytestmark = pytest.mark.gpu
F64 = torch.float64
NONE, SE, EXPSIN, LINEAR, COSINE, M32, M52, ARD = 0, 1, 2, 3, 4, 6, 7, 16
HYP = [0.9, 1.3, 1.1, 0.8]

# one spec per branch of the svgp_kernel_bwd launcher
BWD_SPECS = {
    "se44": (SE, 4, SE, 4),
    "se44_ard": (SE | ARD, 4, SE | ARD, 4),
    "sprites_se": (SE, 8, SE, 16),
    "se_ard_3_2": (SE | ARD, 3, SE, 2),
    "m52_m52": (M52, 4, M52, 4),
    "expsin_linear": (EXPSIN, 1, LINEAR, 8),
    "expsin_cosine": (EXPSIN, 1, COSINE, 8),
    "linear_linear": (LINEAR, 8, LINEAR, 16),
    "cosine_cosine": (COSINE, 8, COSINE, 16),
    "se_linear": (SE, 4, LINEAR, 4),
    "linear_cosine_16_16": (LINEAR, 16, COSINE, 16),     # 32 features: 52 KB of shared memory in the generic passes
}


def _hyp(spec, len_a=None, ard_ls=None):
    h = list(HYP)
    if len_a is not None:
        h[1] = len_a
    if spec[0] & ARD or spec[2] & ARD:
        d = spec[1] + spec[3]
        h += ard_ls if ard_ls is not None else [0.7 + 0.15 * f for f in range(d)]
    return torch.tensor(h, device="cuda")


def _feat(spec, N, M, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    d = spec[1] + spec[3]
    return torch.randn(N, d, generator=g, device="cuda"), torch.randn(M, d, generator=g, device="cuda")


def oracle_bwd(spec, Fx, Fz, hyp, G):
    """float64 autograd of the oracle kernel on the device, chunked over rows: (dx, dz, dhyp)."""
    N, M, d = Fx.shape[0], Fz.shape[0], Fx.shape[1]
    rows = max(256, (1 << 27) // (M * d))                    # (rows, M, d) float64 intermediates of ~1 GB
    Fz_ = Fz.double().requires_grad_(True)
    h_ = hyp.double().requires_grad_(True)
    dx = torch.empty(N, d, dtype=F64, device=Fx.device)
    dz = torch.zeros(M, d, dtype=F64, device=Fx.device)
    dh = torch.zeros_like(h_)
    for i in range(0, N, rows):
        x_ = Fx[i:i + rows].double().requires_grad_(True)
        K = kernel_value(spec, x_, Fz_, h_)
        gx, gz, gh = torch.autograd.grad(K, [x_, Fz_, h_], G[i:i + rows].double(), allow_unused=True)
        dx[i:i + rows] = 0.0 if gx is None else gx
        dz += 0.0 if gz is None else gz
        dh += 0.0 if gh is None else gh
        del K, gx, gz, gh
    return dx, dz, dh


def _check_bwd(be, spec, Fx, Fz, hyp, G, bar=2e-5):
    dx, dz, dh = be.kernel_bwd(spec, Fx, Fz, hyp, G)
    rx, rz, rh = oracle_bwd(spec, Fx, Fz, hyp, G)
    errs = dict(dx=rel_err(dx, rx), dz=rel_err(dz, rz), dhyp=rel_err(dh, rh) if rh.abs().max() > 0 else 0.0)
    print(spec, errs)
    for a in (dx, dz, dh):
        assert torch.isfinite(a).all()
    assert max(errs.values()) < bar, errs
    return errs


# every spec at (65536, 1000) (ragged tiles), and one SE44, one generic SE and one non-stationary spec at (262144, 1024)
BWD_SHAPES = [(65536, 1000, n) for n in BWD_SPECS] + [(262144, 1024, n) for n in ("se44", "sprites_se", "expsin_linear")]


@pytest.mark.parametrize("N,M,name", BWD_SHAPES)
def test_kernel_bwd_at_size(cuda_backend, N, M, name, monkeypatch):
    """kernel_bwd (dx, dz, dhyp) of every launcher branch against float64 autograd.  The SE44 specs also run through the
    generic pass (SVGP_K1_BWD_GENERIC=1)."""
    spec = BWD_SPECS[name]
    Fx, Fz = _feat(spec, N, M)
    hyp = _hyp(spec)
    G = torch.randn(N, M, generator=torch.Generator(device="cuda").manual_seed(1), device="cuda")
    _check_bwd(cuda_backend, spec, Fx, Fz, hyp, G)
    if spec[1] == 4 and spec[3] == 4 and spec[0] & ~ARD == SE and spec[2] & ~ARD == SE:
        monkeypatch.setenv("SVGP_K1_BWD_GENERIC", "1")
        _check_bwd(cuda_backend, spec, Fx, Fz, hyp, G)


# (spec, time column): the shifted feature is the first of block A, whose length scale is 10
OFFSET_SPECS = {
    "se44": (SE, 4, SE, 4),
    "se44_ard": (SE | ARD, 4, SE | ARD, 4),
    "se_1_3": (SE, 1, SE, 3),
    "m32_1_se_3": (M32, 1, SE, 3),
    "se_ard_3_2": (SE | ARD, 3, SE, 2),
}


def _offset_problem(spec, N, M, offset, seed=0):
    """Features with column 0 a time stamp: offset + 10 randn, at length scale 10 (ARD: l_0 = 10)."""
    Fx, Fz = _feat(spec, N, M, seed)
    Fx[:, 0] = offset + 10.0 * Fx[:, 0]
    Fz[:, 0] = offset + 10.0 * Fz[:, 0]
    d = spec[1] + spec[3]
    hyp = _hyp(spec, len_a=None if spec[0] & ARD else 10.0, ard_ls=[10.0] + [0.7 + 0.15 * f for f in range(1, d)])
    return Fx, Fz, hyp


@pytest.mark.parametrize("name", list(OFFSET_SPECS))
@pytest.mark.parametrize("offset", [1e3, 1e4])
def test_kernel_bwd_offset_features(cuda_backend, name, offset):
    """dz, dx and dhyp at a time column offset by 1e3 / 1e4 (l = 10): the Z pass sums c (x_f - z_f) per entry."""
    spec = OFFSET_SPECS[name]
    N, M = 65536, 1000
    Fx, Fz, hyp = _offset_problem(spec, N, M, offset)
    G = torch.randn(N, M, generator=torch.Generator(device="cuda").manual_seed(1), device="cuda")
    _check_bwd(cuda_backend, spec, Fx, Fz, hyp, G)


@pytest.mark.parametrize("name", ["se44", "se_1_3", "m32_1_se_3", "se_ard_3_2"])
def test_kernel_fwd_offset_features(cuda_backend, name):
    """The fp16 planes and the integer planes keep their accuracy at a time column offset by 1e4 (the distances are
    per-entry differences of the fp32 features)."""
    be, spec = cuda_backend, OFFSET_SPECS[name]
    N, M = 8192, 1000
    Fx, Fz, hyp = _offset_problem(spec, N, M, 1e4)
    K = kernel_value(spec, Fx, Fz, hyp)
    kopt = be.kernel_fwd(spec, Fx, Fz, hyp, tc=True, i8=False)
    floor = 2.0 ** -24 * float(kopt.kscale[1])
    assert float((kopt.value().double() - K).abs().max()) < 5e-6 * float(K.abs().max()) + floor
    assert float((kopt.value_t().double() - K.t()).abs().max()) < 5e-6 * float(K.abs().max()) + floor
    _check_i8_planes(be.kernel_fwd(spec, Fx, Fz, hyp, tc=True, i8=True), K, N, M)


def _check_i8_planes(kop, K, N, M):
    """test_gpu_i8_engine.py::test_kplanes_reassemble: half a grid unit, one number on both grids, fp16 row planes, zero pads."""
    Kr, Kc = kop.value_i8("r"), kop.value_i8("c")
    unit_r, unit_c = K.abs().amax(1, keepdim=True) / 2.0 ** 29, K.abs().amax(0, keepdim=True) / 2.0 ** 29
    assert ((Kr - K).abs() <= 1e-7 * K.abs() + 0.51 * unit_r).all()
    assert ((Kc - K).abs() <= 1e-7 * K.abs() + 0.51 * unit_c).all()
    assert kop.Kr[0].int().abs().max() <= 127 and kop.Kc[0].int().abs().max() <= 127
    big = (K.abs() * 64 >= K.abs().amax(1, keepdim=True)) & (K.abs() * 64 >= K.abs().amax(0, keepdim=True))
    assert big.any() and (Kr[big] == Kc[big]).all()
    assert rel_err(kop.value(), K) < 2e-6
    assert (kop.Kr[:, :, M:] == 0).all() and (kop.Kc.permute(0, 1, 3, 2).reshape(4, -1, M)[:, N:] == 0).all()


# signed kinds (LINEAR, COSINE factors) and one non-negative EXPSIN product; lin = the LINEAR block (offset, width) or None
I8_SPECS = {
    "expsin_linear": ((EXPSIN, 1, LINEAR, 8), (1, 8)),
    "linear_cosine": ((LINEAR, 16, COSINE, 16), (0, 16)),
    "cosine_cosine": ((COSINE, 8, COSINE, 16), None),
    "se_linear": ((SE, 4, LINEAR, 4), (4, 4)),
    "expsin_se": ((EXPSIN, 1, SE, 4), None),
}


@pytest.mark.parametrize("name", list(I8_SPECS))
@pytest.mark.parametrize("N,M", [(4096, 256), (5000, 320)])
def test_kplanes_reassemble_kinds(cuda_backend, name, N, M):
    """svgp_kernel_fwd_i8 for the kinds the sweep kernel does not reach: the checks of test_kplanes_reassemble, negative
    leading digits for the signed kinds and kscale[6] (1 only when every entry of K is >= 0).  With a LINEAR block, rows
    7, 100, N - 1 and inducing point 5 have that block exactly zero: their row / column of K is exactly 0, and so are
    their digits and scales."""
    be = cuda_backend
    spec, lin = I8_SPECS[name]
    Fx, Fz = _feat(spec, N, M)
    zr, zc = [7, 100, N - 1], [5]
    if lin is not None:
        Fx[zr, lin[0]:lin[0] + lin[1]] = 0.0
        Fz[zc, lin[0]:lin[0] + lin[1]] = 0.0
    hyp = _hyp(spec)
    kop = be.kernel_fwd(spec, Fx, Fz, hyp, tc=True, i8=True)
    K = kernel_value(spec, Fx, Fz, hyp)
    _check_i8_planes(kop, K, N, M)
    signed = LINEAR in (spec[0], spec[2]) or COSINE in (spec[0], spec[2])
    assert float(kop.kscale[6]) == (0.0 if signed else 1.0)
    assert bool((K < 0).any()) == signed
    assert bool((kop.Kr[0] < 0).any()) == signed and bool((kop.Kc[0] < 0).any()) == signed
    if lin is not None:
        assert (K[zr] == 0).all() and (K[:, zc] == 0).all()
        assert (kop.Kr[:, zr] == 0).all() and (kop.value_i8("c")[zr] == 0).all() and (kop.rscale[zr] == 0).all()
        assert (kop.Kc[:, :, zc] == 0).all() and (kop.value_i8("r")[:, zc] == 0).all() and (kop.cscale[zc] == 0).all()
        assert (kop.value()[zr] == 0).all() and (kop.value()[:, zc] == 0).all()


@pytest.mark.parametrize("case", ["lin_cos", "se_lin", "cos_se", "time_m32_se"])
def test_step_kinds_against_float64_oracle_on_the_gpu(cuda_backend, case):
    """The whole tensor-core step for linear, cosine and an offset time column against the streamlined float64 oracle on
    the GPU (tests/probes/parity_fullsize_kinds.py): the case is well posed (rounding K_nm, K_mm to fp32 inside the oracle
    moves every quantity by less than 1e-5) and all ten quantities are within 1e-4."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "probes"))
    import parity_fullsize_kinds
    o = parity_fullsize_kinds.run(case)
    print(o)
    assert o["gate_max"] < 1e-5, o["gate"]
    for k in parity_fullsize_kinds.QUANTITIES:
        assert o[k] < 1e-4, (k, o)
