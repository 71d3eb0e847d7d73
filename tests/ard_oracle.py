"""ARD (one length scale per feature) SE and Matern factors in float64 -- TEST INFRASTRUCTURE ONLY.

With SVGP_K_ARD (16) OR'ed into SVGP_K_SE or a Matern code, a factor's distance is

    r^2 = sum_f ((x_f - z_f) / l_f)^2,        l_f = hyp[4 + f], f counted over the [A | B] feature row,

and hyp is float[4 + dim_a + dim_b]: an ARD block does not read its isotropic slot (hyp[1] / hyp[3]), an isotropic
block does not read its hyp[4 + f] (include/svgp_b200.h).  ``ARDKernel`` is the ``matrix`` / ``apply`` interface of
oracle/tfp_kernels.py and tests/matern_oracle.py on the scaled differences (x_f - z_f) / l_f, cross-checked against
scikit-learn's anisotropic RBF / Matern in tests/test_ard.py.  Its distance goes through matern_oracle.safe_norm, whose
gradient is zero at r = 0.

``kernel_value`` extends matern_oracle.kernel_value by the flag, and ``ARDOracleBackend`` is the float64 CPU stand-in
backend with it (float64 autograd for the adjoints).
"""
import torch

import matern_oracle as mo
from svgp_vae_b200.backend import Kop

K_SE, K_ARD = 1, 16
F64 = torch.float64


class ARDKernel:
    """Stationary kernel ``base`` ("se" or a Matern code of matern_oracle.CLASSES) with one length scale per feature."""

    def __init__(self, base, amplitude, length_scales):
        self.base, self.amplitude, self.length_scales = base, amplitude, length_scales

    def finish(self, d):
        """The kernel of the scaled differences d = (x - z) / l (last axis: features)."""
        if self.base == K_SE:
            k = torch.exp(-0.5 * (d * d).sum(-1))
            return k * self.amplitude ** 2
        return mo.CLASSES[self.base](self.amplitude, None).finish(mo.safe_norm(d))

    def apply(self, x1, x2):
        return self.finish((x1 - x2) / self.length_scales)

    def matrix(self, x1, x2):
        return self.finish((x1.unsqueeze(-2) - x2.unsqueeze(-3)) / self.length_scales)


def _factor(t, x, z, amp, length, ard_ls, pairwise):
    if t & K_ARD:
        k = ARDKernel(t & ~K_ARD, amp, ard_ls)
        return k.matrix(x, z) if pairwise else k.apply(x, z)
    return mo._factor(t, x, z, amp, length, pairwise)


def kernel_value(spec, Fx, Fz, hyp, pairwise=True):
    """matern_oracle.kernel_value with the ARD flag."""
    ta, da, tb, db = spec
    Fx, Fz, hyp = Fx.to(F64), Fz.to(F64), hyp.to(F64)
    ka = _factor(ta, Fx[:, :da], Fz[:, :da], hyp[0], hyp[1], hyp[4:4 + da], pairwise)
    kb = _factor(tb, Fx[:, da:da + db], Fz[:, da:da + db], hyp[2], hyp[3], hyp[4 + da:4 + da + db], pairwise)
    if ka is None:
        return kb
    return ka if kb is None else ka * kb


class ARDOracleBackend(mo.MaternOracleBackend):
    """The float64 stand-in backend whose K1 primitives also know SVGP_K_ARD."""

    name = "oracle-cpu-f64-ard"

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


class ContinuousProduct(mo.ContinuousProduct):
    """matern_oracle.ContinuousProduct with the ARD flag (hyp of 4 + d entries for ARD specs)."""

    def kernel_matrix(self, x, y, x_inducing=True, y_inducing=True, diag_only=False):
        return kernel_value(self.spec, x, y, self.hyp, pairwise=not diag_only)
