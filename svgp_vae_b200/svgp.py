"""Drop-in SVGP objects: same constructors, methods, argument order and return tuples as the
reference classes in SVGPVAE_model.py, with torch.Tensor (CUDA) in place of tf.Tensor.

  SVGP          moving-ball SVGP, one GP per video          SVGPVAE_model.py:17-171
  mainSVGP      mini-batched SVGP base                      :174-378
  mnistSVGP     ExpSinSquared(view) x Linear(object)        :381-484
  spritesSVGP   action x character, linear or SE            :487-635
  productSVGP   (new) continuous two-block product kernel used by the synthetic sweeps

Per-channel calls (the reference's calling pattern, :868-873) run on the differentiable
primitives of ops.py; ``elbo_step`` is the batched entry the PyTorch glue should use instead of
the Python loop over latent channels -- it is the L-channel fused path of step.py.
Trainable state keeps the reference's variable names (they contain 'GP', which is how the
reference's drivers split optimiser groups, MNIST_experiment.py:897,903).
"""
import math

import numpy as np
import torch

from . import ops
from ._lib import (SVGP_K_COSINE, SVGP_K_EXPSIN, SVGP_K_LINEAR, SVGP_K_MATERN12, SVGP_K_MATERN32, SVGP_K_MATERN52,
                   SVGP_K_NONE, SVGP_K_SE)
from .step import LOG_2PI, elbo_terms, svgp_step


def _torch_dtype(dt):
    if isinstance(dt, torch.dtype):
        return dt
    return {np.dtype("float32"): torch.float32, np.dtype("float64"): torch.float64}[np.dtype(dt)]


def _add_diagonal_jitter(matrix, jitter=1e-8):
    """SVGPVAE_model.py:13-14."""
    m = matrix.shape[-1]
    return matrix + jitter * torch.eye(m, dtype=matrix.dtype, device=matrix.device)


def reciprocal_no_nan(x):
    """tf.math.reciprocal_no_nan (SVGPVAE_model.py:78,282,330): 1/x, 0 where x == 0."""
    safe = torch.where(x == 0, torch.ones_like(x), x)
    return torch.where(x == 0, torch.zeros_like(x), 1.0 / safe)


def gauss_cross_entropy(mu1, var1, mu2, var2):
    """utils.py:483-504, element-wise E_{N(mu1,var1)}[log N(z | mu2, var2)]."""
    return -0.5 * (LOG_2PI + torch.log(var2) + (var1 + mu1 ** 2 - 2 * mu1 * mu2 + mu2 ** 2) / var2)


def _as_param_or_buffer(module, name, value, dtype, trainable):
    t = torch.as_tensor(np.asarray(value) if not isinstance(value, torch.Tensor) else value).to(dtype).clone()
    if trainable:
        module.register_parameter(name, torch.nn.Parameter(t))
    else:
        module.register_buffer(name, t)
    return name


class _KernelBase(torch.nn.Module):
    """Feature assembly + hyper-parameter vector for the two-block product kernel of K1."""

    def _spec(self):
        raise NotImplementedError

    def _hyp(self):
        raise NotImplementedError

    def _features(self, x, inducing):
        raise NotImplementedError

    def kernel_matrix(self, x, y, x_inducing=True, y_inducing=True, diag_only=False):
        """K(x, y) -- SVGPVAE_model.py:206 / :427 / :550.  diag_only -> element-wise k(x_i, y_i)."""
        Fx, Fy = self._features(x, x_inducing), self._features(y, y_inducing)
        if diag_only:
            return ops.kernel_diag(Fx, Fy, self._hyp(), self._spec()).to(self.dtype)
        return ops.kernel_matrix(Fx, Fy, self._hyp(), self._spec()).to(self.dtype)


# --------------------------------------------------------------------------------------
class mainSVGP(_KernelBase):
    def __init__(self, titsias, fixed_inducing_points, initial_inducing_points, name, jitter, N_train, dtype, L,
                 K_obj_normalize=False):
        super().__init__()
        self.dtype = _torch_dtype(dtype)
        self.jitter = jitter
        self.titsias = titsias
        self.nr_inducing = len(initial_inducing_points)
        self.N_train = N_train
        self.L = L
        self.K_obj_normalize = K_obj_normalize
        self._ip_name = _as_param_or_buffer(self, "Sparse_GP_inducing_points_{}".format(name), initial_inducing_points,
                                            self.dtype, not fixed_inducing_points)

    @property
    def inducing_index_points(self):
        return getattr(self, self._ip_name)

    # ---- shared pieces ---------------------------------------------------------------------
    def _inducing_factors(self):
        Fz = self._features(self.inducing_index_points, True)
        K_mm = ops.kernel_matrix(Fz, Fz, self._hyp(), self._spec()).double()
        K_mm_inv, ldK, _ = ops.spd_inverse_logdet(_add_diagonal_jitter(K_mm, self.jitter).unsqueeze(0))
        return Fz, K_mm, K_mm_inv, ldK[0]

    def approximate_posterior_params(self, index_points_test, index_points_train=None, y=None, noise=None):
        """:303-343 -> (mean_vector (x,), B (x,), mu_hat (m,), A_hat (m, m))."""
        hyp, spec = self._hyp(), self._spec()
        b = float(index_points_train.shape[0])
        c = self.N_train / b
        Fz, K_mm, K_mm_inv, _ = self._inducing_factors()
        Fx_t = self._features(index_points_test, False)
        same = index_points_train is index_points_test
        Fx_n = Fx_t if same else self._features(index_points_train, False)
        K_xx = ops.kernel_diag(Fx_t, Fx_t, hyp, spec)
        K_xm = ops.kernel_matrix(Fx_t, Fz, hyp, spec)
        K_nm = K_xm if same else ops.kernel_matrix(Fx_n, Fz, hyp, spec)
        prec = reciprocal_no_nan(noise)
        A = ops.syrk(K_nm, prec[:, None])                                          # (1,m,m)  :328-330
        sigma_l = K_mm.unsqueeze(0) + c * A
        sigma_l_inv, _, _ = ops.spd_inverse_logdet(_add_diagonal_jitter(sigma_l, self.jitter))   # :331
        v = ops.kt_matmul(K_nm, (prec * y)[:, None])                               # (1,m)
        Sv = ops.bmv64(sigma_l_inv, v)
        mean_vector = c * ops.k_matmul(K_xm, Sv)[:, 0].double()                    # :332-334
        B = K_xx.double() - ops.rowquad(K_xm, K_mm_inv)[:, 0].double() + ops.rowquad(K_xm, sigma_l_inv)[:, 0].double()
        mu_hat = c * ops.bmv64(K_mm.unsqueeze(0), Sv)[0]                           # :339-340
        A_hat = ops.bmm64(ops.bmm64(K_mm.unsqueeze(0), sigma_l_inv), K_mm.unsqueeze(0))[0]   # :341
        dt = self.dtype
        return mean_vector.to(dt), B.to(dt), mu_hat.to(dt), A_hat.to(dt)

    def variational_loss(self, x, y, mu_hat, A_hat, noise=None):
        """:220-301, Hensman branch -> (L_3 sum term, KL term)."""
        hyp, spec = self._hyp(), self._spec()
        b, m = float(x.shape[0]), float(self.nr_inducing)
        Fz, K_mm, K_mm_inv, ldK = self._inducing_factors()
        Fx = self._features(x, False)
        K_nn = ops.kernel_diag(Fx, Fx, hyp, spec).double()
        K_nm = ops.kernel_matrix(Fx, Fz, hyp, spec)
        if self.titsias:
            # :246-259 -- L_2 of Titsias: a (b x b) Gaussian log-density, small batches only (as in the reference)
            Kd = K_nm.double().unsqueeze(0)
            Q = ops.bmm64(ops.bmm64(Kd, K_mm_inv), Kd, False, True)[0]                       # K_nm Kinv K_mn   (b, b)
            yd, nd = y.double(), noise.double()
            cov_j = _add_diagonal_jitter(torch.diag(nd) + Q, self.jitter)                    # :248, :251-252
            cov_inv, cov_logdet, _ = ops.spd_inverse_logdet(cov_j.unsqueeze(0))
            trace_term = reciprocal_no_nan(nd) * (K_nn - torch.diagonal(Q))                  # :249-250
            L2 = -0.5 * (b * math.log(2 * math.pi) + cov_logdet[0] + (yd * (cov_inv[0] @ yd)).sum() + trace_term.sum())
            return L2.to(self.dtype), torch.zeros((), dtype=self.dtype, device=L2.device)    # :255-259
        mu64, A64 = mu_hat.double(), A_hat.double()
        a = ops.bmv64(K_mm_inv, mu64.unsqueeze(0))                                 # Kinv mu_hat
        mean_vector = ops.k_matmul(K_nm, a)[:, 0].double()                         # :264-265
        ld_S = ops.spd_logdet(_add_diagonal_jitter(A64, self.jitter).unsqueeze(0))[0]   # :271-274
        KL = 0.5 * (ldK - ld_S - m + (K_mm_inv[0] * A64.t()).sum() + (mu64 * a[0]).sum())   # :276-279
        prec = reciprocal_no_nan(noise).double()
        K_tilde = prec * (K_nn - ops.rowquad(K_nm, K_mm_inv)[:, 0].double())       # :284
        Wm = ops.bmm64(ops.bmm64(K_mm_inv, A64.unsqueeze(0)), K_mm_inv)            # Kinv A_hat Kinv
        trace_terms = prec * ops.rowquad(K_nm, Wm)[:, 0].double()                  # :286-294 without the (b,m,m) tensor
        yd, nd = y.double(), noise.double()
        L3 = -0.5 * (K_tilde.sum() + trace_terms.sum() + torch.log(nd).sum() + b * math.log(2 * math.pi)
                     + (prec * (yd - mean_vector) ** 2).sum())                     # :297-299
        return L3.to(self.dtype), KL.to(self.dtype)

    def mean_vector_bias_analysis(self, index_points, y=None, noise=None):
        """:345-370."""
        hyp, spec = self._hyp(), self._spec()
        c = self.N_train / float(index_points.shape[0])
        Fz = self._features(self.inducing_index_points, True)
        K_mm = ops.kernel_matrix(Fz, Fz, hyp, spec).double()
        K_bm = ops.kernel_matrix(self._features(index_points, False), Fz, hyp, spec)
        prec = reciprocal_no_nan(noise)
        sigma_l = K_mm.unsqueeze(0) + c * ops.syrk(K_bm, prec[:, None])
        sigma_l_inv, _, _ = ops.spd_inverse_logdet(_add_diagonal_jitter(sigma_l, self.jitter))
        v = ops.kt_matmul(K_bm, (prec * y)[:, None])
        return (c * ops.bmv64(K_mm.unsqueeze(0), ops.bmv64(sigma_l_inv, v))[0]).to(self.dtype)

    def variable_summary(self):
        raise NotImplementedError()

    # ---- batched entry (replaces the L-loop of forward_pass_SVGPVAE :865-898) -----------------
    def elbo_step(self, aux_data, qnet_mu, qnet_var, clip_pv=False, group=None, **kw):
        """All latent channels at once.  aux_data (b, d_aux), qnet_mu / qnet_var (b, L).

        Returns the dict of step.svgp_step plus the scalars of :880-898 (inside_elbo_recon,
        inside_elbo_kl, inside_elbo, ce_term, KL_term).  ``clip_pv`` mirrors :891-892.
        """
        if self.titsias:
            return self._elbo_step_per_channel(aux_data, qnet_mu, qnet_var, clip_pv)
        Fx = self._features(aux_data, False)
        Fz = self._features(self.inducing_index_points, True)
        res = svgp_step(self._spec(), Fx, Fz, self._hyp(), qnet_mu, qnet_var, N_train=self.N_train,
                        jitter=self.jitter, clip_pv=(1e-4, 100.0) if clip_pv else None, group=group, **kw)
        res.update(elbo_terms(res, res["b_total"], self.N_train))      # the all-reduced batch size (shards may be unequal)
        return res


    def _elbo_step_per_channel(self, aux_data, qnet_mu, qnet_var, clip_pv=False):
        """The reference's own loop (:868-898) over the per-channel methods.  Used for the Titsias bound, whose
        (b x b) Gaussian term has no channel-batched kernel here (it is a small-batch formulation by construction)."""
        recon, kl, pms, pvs, mus, Ahs = [], [], [], [], [], []
        for l in range(qnet_mu.shape[1]):
            pm, pv, mu_hat, A_hat = self.approximate_posterior_params(aux_data, aux_data, qnet_mu[:, l], qnet_var[:, l])
            r_l, k_l = self.variational_loss(x=aux_data, y=qnet_mu[:, l], noise=qnet_var[:, l], mu_hat=mu_hat, A_hat=A_hat)
            recon.append(r_l.double()); kl.append(k_l.double()); pms.append(pm); pvs.append(pv)
            mus.append(mu_hat); Ahs.append(A_hat)
        p_m, p_v = torch.stack(pms, 1), torch.stack(pvs, 1)
        if clip_pv:
            p_v = torch.clamp(p_v, 1e-4, 100.0)                                            # :891-892
        recon_l, kl_l = torch.stack(recon), torch.stack(kl)
        ce_l = gauss_cross_entropy(p_m.double(), p_v.double(), qnet_mu.double(), qnet_var.double()).sum(0)
        rec, k, ce = recon_l.sum(), kl_l.sum(), ce_l.sum()
        b = float(aux_data.shape[0])
        inside = rec - k if self.titsias else rec - (b / self.N_train) * k                 # :883-886
        return dict(p_m=p_m, p_v=p_v, recon_l=recon_l, kl_l=kl_l, ce_l=ce_l, mu_hat=torch.stack(mus).detach(),
                    A_hat=torch.stack(Ahs).detach(), inside_elbo_recon=rec, inside_elbo_kl=k, inside_elbo=inside,
                    ce_term=ce, KL_term=-ce + inside)


# --------------------------------------------------------------------------------------
class mnistSVGP(mainSVGP):
    def __init__(self, titsias, fixed_inducing_points, initial_inducing_points, fixed_gp_params, object_vectors_init,
                 name, jitter, N_train, L, K_obj_normalize):
        super().__init__(titsias=titsias, fixed_inducing_points=fixed_inducing_points,
                         initial_inducing_points=initial_inducing_points, name=name, jitter=jitter, N_train=N_train,
                         dtype=torch.float64, L=L, K_obj_normalize=K_obj_normalize)       # :404 float64 always
        self._l_name = _as_param_or_buffer(self, "GP_length_scale_{}".format(name), 1.0, self.dtype, not fixed_gp_params)
        self._amp_name = _as_param_or_buffer(self, "GP_amplitude_{}".format(name), 1.0, self.dtype, not fixed_gp_params)
        if object_vectors_init is not None:
            self._ov_name = _as_param_or_buffer(self, "GP_object_vectors_{}".format(name), object_vectors_init,
                                                self.dtype, True)
        else:
            self._ov_name = None

    l_GP = property(lambda self: getattr(self, self._l_name))
    amplitude = property(lambda self: getattr(self, self._amp_name))
    object_vectors = property(lambda self: None if self._ov_name is None else getattr(self, self._ov_name))

    def _spec(self):
        d_obj = self.inducing_index_points.shape[1] - 2
        return (SVGP_K_EXPSIN, 1, SVGP_K_COSINE if self.K_obj_normalize else SVGP_K_LINEAR, d_obj)

    def _hyp(self):
        one = torch.ones((), dtype=self.dtype, device=self.l_GP.device)
        return torch.stack([self.amplitude, self.l_GP, one, one])

    def _features(self, x, inducing):
        """:443-455 -- [angle | object vector]; data rows gather their object vector by id when the table exists."""
        if inducing or self.object_vectors is None:
            return x[:, 1:]
        obj = ops.gather_rows(self.object_vectors, x[:, 0].long())
        return torch.cat([x[:, 1:2].to(obj.dtype), obj], dim=1)

    def variable_summary(self):
        return self.l_GP, self.amplitude, self.object_vectors, self.inducing_index_points


class spritesSVGP(mainSVGP):
    def __init__(self, titsias, fixed_inducing_points, initial_inducing_points, name, jitter, N_train, L_action,
                 initial_GPLVM_action, L_character, L, fixed_GP_params=False, fixed_GPLVM=False, K_obj_normalize=False,
                 K_SE=False):
        super().__init__(titsias=titsias, fixed_inducing_points=fixed_inducing_points,
                         initial_inducing_points=initial_inducing_points, name=name, jitter=jitter, N_train=N_train,
                         dtype=torch.float32, K_obj_normalize=K_obj_normalize, L=L)        # :516 float32
        self.L_action, self.L_character, self.K_SE = L_action, L_character, K_SE
        self._act_name = _as_param_or_buffer(self, "GP_GPLVM_action_vectors_", initial_GPLVM_action, self.dtype,
                                             not fixed_GPLVM)
        if K_SE:                                                                           # :530-544
            tr = not fixed_GP_params
            _as_param_or_buffer(self, "GP_length_scale_action", 1.0, self.dtype, tr)
            _as_param_or_buffer(self, "GP_amplitude_action", 0.1, self.dtype, tr)
            _as_param_or_buffer(self, "GP_length_scale_character", 1.0, self.dtype, tr)
            _as_param_or_buffer(self, "GP_amplitude_character", 0.1, self.dtype, tr)

    GPLVM_action = property(lambda self: getattr(self, self._act_name))
    l_action = property(lambda self: self.GP_length_scale_action)
    sigma_action = property(lambda self: self.GP_amplitude_action)
    l_character = property(lambda self: self.GP_length_scale_character)
    sigma_character = property(lambda self: self.GP_amplitude_character)

    def _spec(self):
        if self.K_SE:
            t = SVGP_K_SE
        else:
            t = SVGP_K_COSINE if self.K_obj_normalize else SVGP_K_LINEAR
        return (t, self.L_action, t, self.L_character)

    def _hyp(self):
        if self.K_SE:
            return torch.stack([self.sigma_action, self.l_action, self.sigma_character, self.l_character])
        return torch.ones(4, dtype=self.dtype, device=self.GPLVM_action.device)

    def _features(self, x, inducing):
        """:562-570 -- inducing rows are [action | character]; data rows are [action id | character]."""
        if inducing:
            return x
        act = ops.gather_rows(self.GPLVM_action, x[:, 0].long())
        return torch.cat([act, x[:, 1:].to(act.dtype)], dim=1)

    def variable_summary(self):
        return self.GPLVM_action, self.inducing_index_points

    def approximate_posterior_params_precomputed_GP_posterior_params(self, index_points, mean_term, sigma_term,
                                                                     K_mm_inv=None):
        """:610-635 -> (mean_vector (b,), B (b,))."""
        hyp, spec = self._hyp(), self._spec()
        Fz = self._features(self.inducing_index_points, True)
        if K_mm_inv is None:
            K_mm = ops.kernel_matrix(Fz, Fz, hyp, spec).double()
            K_mm_inv = ops.spd_inverse_logdet(_add_diagonal_jitter(K_mm, self.jitter).unsqueeze(0))[0][0]
        Fx = self._features(index_points, False)
        K_bb = ops.kernel_diag(Fx, Fx, hyp, spec)
        K_bm = ops.kernel_matrix(Fx, Fz, hyp, spec)
        mean_vector = ops.k_matmul(K_bm, mean_term.reshape(1, -1))[:, 0]
        B = K_bb.double() - ops.rowquad(K_bm, K_mm_inv.double().unsqueeze(0))[:, 0].double() \
            + ops.rowquad(K_bm, sigma_term.double().unsqueeze(0))[:, 0].double()
        return mean_vector.to(self.dtype), B.to(self.dtype)


class productSVGP(mainSVGP):
    """Continuous two-block product kernel kA(x[:, :dA], z[:, :dA]) * kB(x[:, dA:], z[:, dA:]) with data rows laid
    out like inducing rows (no id column).  Not in the reference: it is the full-rank stand-in the synthetic sweeps
    need (SURVEY H3: the MNIST kernel is rank-deficient beyond M ~ 64); with SE x SE it is spritesSVGP's K_SE form
    (:542-544) without the action-id gather.

    ``kind_a`` / ``kind_b`` name each factor: "se" (tfk.ExponentiatedQuadratic), "matern12", "matern32", "matern52"
    (tfk.MaternOneHalf / MaternThreeHalves / MaternFiveHalves: a^2 p(u) exp(-u), u = c |x - z| / l with c = 1, sqrt 3,
    sqrt 5), "linear", "cosine" or "none" (a factor of 1; its block must be empty).  Every stationary factor takes its
    own amplitude a and length scale l from ``amplitude`` / ``length_scale``.  The Matern kinds suit rough continuous
    auxiliary data (time, position, pose), where SE's infinitely smooth prior is too strong; e.g. a Matern 3/2 kernel
    over time times a Matern 5/2 kernel over a 3-D position:

        productSVGP(Z, dim_a=1, dim_b=3, kind_a="matern32", kind_b="matern52", N_train=N, L=L)
    """

    _TYPES = {"se": SVGP_K_SE, "linear": SVGP_K_LINEAR, "cosine": SVGP_K_COSINE, "none": SVGP_K_NONE,
              "matern12": SVGP_K_MATERN12, "matern32": SVGP_K_MATERN32, "matern52": SVGP_K_MATERN52}

    def __init__(self, initial_inducing_points, dim_a, dim_b, name="prod", jitter=1e-2, N_train=1, L=1, kind_a="se",
                 kind_b="se", amplitude=(1.0, 1.0), length_scale=(1.0, 1.0), fixed_inducing_points=False,
                 fixed_gp_params=False, titsias=False, dtype=torch.float32):
        super().__init__(titsias, fixed_inducing_points, initial_inducing_points, name, jitter, N_train, dtype, L)
        self.dim_a, self.dim_b = dim_a, dim_b
        self.kinds = (self._TYPES[kind_a], self._TYPES[kind_b])
        hyp = [amplitude[0], length_scale[0], amplitude[1], length_scale[1]]
        _as_param_or_buffer(self, "GP_hypers_{}".format(name), hyp, self.dtype, not fixed_gp_params)
        self._hyp_name = "GP_hypers_{}".format(name)

    def _spec(self):
        return (self.kinds[0], self.dim_a, self.kinds[1], self.dim_b)

    def _hyp(self):
        return getattr(self, self._hyp_name)

    def _features(self, x, inducing):
        return x

    def variable_summary(self):
        return self._hyp(), self.inducing_index_points


# --------------------------------------------------------------------------------------
class SVGP(_KernelBase):
    """Moving-ball SVGP (SVGPVAE_model.py:17-171): one GP per video over a 1-D time index, RBF kernel with
    amplitude None, no N/b factor, full (tmax x tmax) posterior covariance returned, and the reference's KL quirks
    (A_hat in the quadratic term, batch-summed log-det; :132-137) reproduced literally."""

    dtype = torch.float32

    def __init__(self, titsias, num_inducing_points, fixed_inducing_points, tmin, tmax, vidlt, fixed_gp_params, name,
                 jitter, ip_min, ip_max, GP_init):
        super().__init__()
        self.titsias = titsias
        self.num_inducing_points = num_inducing_points
        self.tmin, self.tmax, self.ip_min, self.ip_max = tmin, tmax, ip_min, ip_max
        self.jitter = jitter
        lo, hi = (tmin, tmax) if fixed_inducing_points else (ip_min, ip_max)
        self._ip_name = _as_param_or_buffer(self, "inducing_index_points_{}".format(name),
                                            np.linspace(lo, hi, num_inducing_points, dtype=np.float32), self.dtype,
                                            not fixed_inducing_points)
        self._l_name = _as_param_or_buffer(self, "GP_length_scale_{}".format(name),
                                           vidlt if fixed_gp_params else GP_init, self.dtype, not fixed_gp_params)

    inducing_index_points = property(lambda self: getattr(self, self._ip_name))
    l_GP = property(lambda self: getattr(self, self._l_name))

    def _spec(self):
        return (SVGP_K_SE, 1, SVGP_K_NONE, 0)

    def _hyp(self):
        one = torch.ones((), dtype=self.dtype, device=self.l_GP.device)
        return torch.stack([one, self.l_GP, one, one])

    def _features(self, x, inducing):
        return x.reshape(-1, 1)

    def _mats(self, x):
        """Flattened (batch*tmax) rows: K_nm (BT, m) fp32, K_mm, Kinv (1,m,m), logdet, diag blocks of K_nn."""
        hyp, spec = self._hyp(), self._spec()
        Bn, T = x.shape
        Fz = self._features(self.inducing_index_points, True)
        Fx = self._features(x, False)
        K_mm = ops.kernel_matrix(Fz, Fz, hyp, spec).double()
        K_mm_inv, ldK, _ = ops.spd_inverse_logdet(_add_diagonal_jitter(K_mm, self.jitter).unsqueeze(0))
        K_nm = ops.kernel_matrix(Fx, Fz, hyp, spec)
        return Bn, T, Fx, K_mm, K_mm_inv, ldK[0], K_nm

    @staticmethod
    def _own(full, Bn, T):
        """(B*T, B) -> (B, T): entry [b, t] of column b (each video against its own channel)."""
        idx = torch.arange(Bn, device=full.device)
        return full.reshape(Bn, T, Bn)[idx, :, idx]

    @staticmethod
    def _blockdiag(vals):
        """(B, T) -> (B*T, B) with video b's values in column b, zeros elsewhere."""
        Bn, T = vals.shape
        out = vals.new_zeros(Bn, T, Bn)
        idx = torch.arange(Bn, device=vals.device)
        out[idx, :, idx] = vals
        return out.reshape(Bn * T, Bn)

    def approximate_posterior_params(self, index_points, y=None, noise=None):
        """:141-171 -> mean (B,T), cov (B,T,T), mu_hat (B,m), A_hat (B,m,m)."""
        Bn, T, Fx, K_mm, K_mm_inv, _, K_nm = self._mats(index_points)
        prec = reciprocal_no_nan(noise)
        A = ops.syrk(K_nm, self._blockdiag(prec))                                        # (B,m,m)   :160
        sigma_l_inv, _, _ = ops.spd_inverse_logdet(_add_diagonal_jitter(K_mm.unsqueeze(0) + A, self.jitter))   # :161
        v = ops.kt_matmul(K_nm, self._blockdiag(prec * y))                               # (B,m)
        Sv = ops.bmv64(sigma_l_inv, v)
        mean_vector = self._own(ops.k_matmul(K_nm, Sv), Bn, T)                           # :164
        Kb = K_nm.double().reshape(Bn, T, -1)
        K_nn = ops.kernel_matrix(Fx, Fx, self._hyp(), self._spec()).double()
        idx = torch.arange(Bn, device=K_nn.device)
        K_nn = K_nn.reshape(Bn, T, Bn, T)[idx, :, idx, :]                                # per-video (T,T) blocks
        Bcov = K_nn + ops.bmm64(ops.bmm64(Kb, sigma_l_inv - K_mm_inv), Kb, False, True)  # :165
        mu_hat = ops.bmv64(K_mm.unsqueeze(0), Sv)                                        # :167
        A_hat = ops.bmm64(ops.bmm64(K_mm.unsqueeze(0), sigma_l_inv), K_mm.unsqueeze(0))  # :169
        dt = self.dtype
        return mean_vector.to(dt), Bcov.to(dt), mu_hat.to(dt), A_hat.to(dt)

    def variational_loss(self, x, y, noise, mu_hat, A_hat):
        """:62-139, Hensman branch -> ((B,), (B,))."""
        Bn, T, Fx, K_mm, K_mm_inv, ldK, K_nm = self._mats(x)
        m = float(self.inducing_index_points.shape[0])
        prec = reciprocal_no_nan(noise).double()
        if self.titsias:
            # :89-101 -- per-video (T x T) Gaussian log-density
            Kb = K_nm.double().reshape(Bn, T, -1)
            Q = ops.bmm64(ops.bmm64(Kb, K_mm_inv), Kb, False, True)                          # (B, T, T)
            cov_j = _add_diagonal_jitter(torch.diag_embed(noise.double()) + Q, self.jitter)
            cov_inv, cov_logdet, _ = ops.spd_inverse_logdet(cov_j)
            K_nn_diag = ops.kernel_diag(Fx, Fx, self._hyp(), self._spec()).double().reshape(Bn, T)
            trace_term = prec * (K_nn_diag - torch.diagonal(Q, dim1=-2, dim2=-1))
            yd = y.double()
            L2 = -0.5 * (T * math.log(2 * math.pi) + cov_logdet + (yd * ops.bmv64(cov_inv, yd)).sum(1) + trace_term.sum(1))
            return L2.to(self.dtype), torch.zeros((), dtype=self.dtype, device=L2.device)
        mu64, A64 = mu_hat.double(), A_hat.double()
        a = ops.bmm64(mu64.unsqueeze(0), K_mm_inv)[0]                                    # (B,m) = Kinv mu_hat (Kinv symmetric)
        mean_vector = self._own(ops.k_matmul(K_nm, a), Bn, T).double()                   # :106
        K_nn_diag = ops.kernel_diag(Fx, Fx, self._hyp(), self._spec()).double().reshape(Bn, T)
        h = ops.rowquad(K_nm, K_mm_inv)[:, 0].double().reshape(Bn, T)
        K_tilde = prec * (K_nn_diag - h)                                                 # :109
        Wm = ops.bmm64(ops.bmm64(K_mm_inv, A64), K_mm_inv)                               # Kinv A_hat_b Kinv
        trace_terms = prec * self._own(ops.rowquad(K_nm, Wm), Bn, T).double()            # :112-121
        yd, nd = y.double(), noise.double()
        L3 = -0.5 * (K_tilde.sum(1) + trace_terms.sum(1) + torch.log(nd).sum(1) + T * math.log(2 * math.pi)
                     + (prec * (yd - mean_vector) ** 2).sum(1))                          # :124-126
        S_log_det = ops.spd_logdet(_add_diagonal_jitter(A64, self.jitter)).sum()          # :130,132 (whole batch)
        quirk = (A64 * ops.bmm64(A64, K_mm_inv)).sum()                                   # :136-137
        KL = 0.5 * (ldK - S_log_det - m + (K_mm_inv * A64.transpose(-1, -2)).sum((-1, -2)) + quirk)   # :134-137
        return L3.to(self.dtype), KL.to(self.dtype)
