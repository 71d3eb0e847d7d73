"""Matern 1/2, 3/2, 5/2 kernels in float64 -- TEST INFRASTRUCTURE ONLY.

tfp.math.psd_kernels MaternOneHalf / MaternThreeHalves / MaternFiveHalves(amplitude s, length_scale l), r = ||x - y||:

    k(x, y) = s^2 exp(-u),                   u = r / l
    k(x, y) = s^2 (1 + u) exp(-u),           u = sqrt(3) r / l
    k(x, y) = s^2 (1 + u + u^2 / 3) exp(-u), u = sqrt(5) r / l

with the ``matrix`` / ``apply`` interface of oracle/tfp_kernels.py, cross-checked against scikit-learn's
Matern(nu = 0.5, 1.5, 2.5) in tests/test_matern.py.  The distance goes through a square root with a zero gradient at
r = 0: there the 1/2 kernel has no derivative and zero is its symmetric subgradient (the exact total derivative of
k(z, z) = s^2 when both arguments are the same point, SVGP_K_MATERN12 in include/svgp_b200.h); for 3/2 and 5/2 zero is
the true derivative.

``kernel_value`` extends tests/oracle_backend.kernel_value by the type codes SVGP_K_MATERN12 / 32 / 52 (5, 6, 7), and
``MaternOracleBackend`` is the float64 CPU stand-in backend with it.
"""
import math

import torch

import oracle_backend
from oracle_backend import OracleBackend
from svgp_vae_b200.backend import Kop

K_MATERN12, K_MATERN32, K_MATERN52 = 5, 6, 7
F64 = torch.float64


def safe_norm(d):
    """||d|| over the last axis, zero gradient where d = 0."""
    r2 = (d * d).sum(-1)
    pos = r2 > 0
    return torch.where(pos, torch.sqrt(torch.where(pos, r2, torch.ones_like(r2))), torch.zeros_like(r2))


class _Matern:
    c = 1.0

    def __init__(self, amplitude=None, length_scale=None):
        self.amplitude = amplitude
        self.length_scale = length_scale

    def _poly(self, u):
        raise NotImplementedError

    def finish(self, r):
        """The kernel as a function of the distance r."""
        u = self.c * r
        if self.length_scale is not None:
            u = u / self.length_scale
        k = self._poly(u) * torch.exp(-u)
        if self.amplitude is not None:
            k = k * self.amplitude ** 2
        return k

    def apply(self, x1, x2):
        return self.finish(safe_norm(x1 - x2))

    def matrix(self, x1, x2):
        return self.finish(safe_norm(x1.unsqueeze(-2) - x2.unsqueeze(-3)))


class MaternOneHalf(_Matern):
    c = 1.0

    def _poly(self, u):
        return torch.ones_like(u)


class MaternThreeHalves(_Matern):
    c = math.sqrt(3.0)

    def _poly(self, u):
        return 1.0 + u


class MaternFiveHalves(_Matern):
    c = math.sqrt(5.0)

    def _poly(self, u):
        return 1.0 + u + u * u / 3.0


CLASSES = {K_MATERN12: MaternOneHalf, K_MATERN32: MaternThreeHalves, K_MATERN52: MaternFiveHalves}
BY_KIND = {"matern12": MaternOneHalf, "matern32": MaternThreeHalves, "matern52": MaternFiveHalves}


def _factor(t, x, z, amp, length, pairwise):
    if t in CLASSES:
        k = CLASSES[t](amp, length)
        return k.matrix(x, z) if pairwise else k.apply(x, z)
    return oracle_backend._factor(t, x, z, amp, length, pairwise)


def kernel_value(spec, Fx, Fz, hyp, pairwise=True):
    """oracle_backend.kernel_value with the Matern factors."""
    ta, da, tb, db = spec
    Fx, Fz, hyp = Fx.to(F64), Fz.to(F64), hyp.to(F64)
    ka = _factor(ta, Fx[:, :da], Fz[:, :da], hyp[0], hyp[1], pairwise)
    kb = _factor(tb, Fx[:, da:da + db], Fz[:, da:da + db], hyp[2], hyp[3], pairwise)
    if ka is None:
        return kb
    return ka if kb is None else ka * kb


class MaternOracleBackend(OracleBackend):
    """OracleBackend whose K1 primitives also know the Matern type codes (float64 autograd for the adjoints)."""

    name = "oracle-cpu-f64-matern"

    def kernel_fwd(self, spec, Fx, Fz, hyp, tc=False):
        return Kop(kernel_value(spec, Fx, Fz, hyp).float())

    def kernel_fwd_f64(self, spec, Fx, Fz, hyp):
        return kernel_value(spec, Fx, Fz, hyp)

    def kernel_bwd(self, spec, Fx, Fz, hyp, G, need_x=True, need_z=True):
        with torch.enable_grad():
            Fx_, Fz_, h_ = (t.detach().to(F64).requires_grad_(True) for t in (Fx, Fz, hyp))
            K = kernel_value(spec, Fx_, Fz_, h_)
            gx, gz, gh = torch.autograd.grad(K, [Fx_, Fz_, h_], G.to(F64), allow_unused=True)
        z = lambda g, ref: torch.zeros_like(ref) if g is None else g
        return (z(gx, Fx_).float() if need_x else None, z(gz, Fz_) if need_z else None, z(gh, h_))

    def kernel_diag_fwd(self, spec, Fx, Fy, hyp):
        return kernel_value(spec, Fx, Fy, hyp, pairwise=False).float()

    def kernel_diag_bwd(self, spec, Fx, Fy, hyp, g):
        with torch.enable_grad():
            Fx_, Fy_, h_ = (t.detach().to(F64).requires_grad_(True) for t in (Fx, Fy, hyp))
            k = kernel_value(spec, Fx_, Fy_, h_, pairwise=False)
            gx, gy, gh = torch.autograd.grad(k, [Fx_, Fy_, h_], g.to(F64), allow_unused=True)
        z = lambda gg, ref: torch.zeros_like(ref) if gg is None else gg
        return z(gx, Fx_).float(), z(gy, Fy_).float(), z(gh, h_)


class ContinuousProduct:
    """productSVGP as the streamlined oracle (refs.streamlined_objective) sees it: float64 kernel matrices of the oracle
    formulas on differentiable float64 copies of the inducing points and hyper-parameters."""

    def __init__(self, Z, hyp, spec, jitter, N_train):
        self.inducing_index_points = torch.as_tensor(Z, dtype=F64).clone()
        self.hyp = torch.as_tensor(hyp, dtype=F64).clone()
        self.spec, self.jitter, self.N_train = spec, jitter, N_train

    def kernel_matrix(self, x, y, x_inducing=True, y_inducing=True, diag_only=False):
        return kernel_value(self.spec, x, y, self.hyp, pairwise=not diag_only)
