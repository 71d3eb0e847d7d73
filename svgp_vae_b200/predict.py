"""Prediction-time entry points of the SVGP object, all latent channels at once (no gradients).

Reference call sites (the per-channel Python loops these replace):

  precompute_GP_params_SVGPVAE            SVGPVAE_model.py:989-1023   (L x m) mean terms, (L x m x m) Sigma_l^-1,
                                                                      built from ALL training encodings; note :1014 inverts
                                                                      Sigma_l WITHOUT jitter and without the N_train/b factor
  predict_from_precomputed                :610-635 called per channel at :1165-1168
  posterior_predict                       :1048-1050 (bacthing_predict_SVGPVAE_rotated_mnist): approximate_posterior_params
                                          (:303-343) with test index points against the full training set

Same kernels as the training step (K1 builder, K2 SYRK on tcgen05, float64 Cholesky stage, K4 row quadratic forms).
"""
import torch

from . import ops, step
from .backend import get_backend


def _recip_no_nan(x):
    safe = torch.where(x == 0, torch.ones_like(x), x)
    return torch.where(x == 0, torch.zeros_like(x), 1.0 / safe)


def _operands(svgp, aux_data):
    be = get_backend()
    spec = svgp._spec()
    hyp = svgp._hyp().detach().float().contiguous()
    Fx = svgp._features(aux_data, False).detach().float().contiguous()
    Fz = svgp._features(svgp.inducing_index_points, True).detach().float().contiguous()
    kop = be.kernel_fwd(spec, Fx, Fz, hyp, tc=be.want_tc(Fx.shape[0], Fz.shape[0]))
    return be, spec, hyp, Fx, Fz, kop


@torch.no_grad()
def precompute_GP_params_SVGPVAE(means, vars, aux_data, svgp):
    """(mean_terms (L, m), inv_Sigma_l (L, m, m)) -- SVGPVAE_model.py:989-1023, every channel in one pass."""
    be, spec, hyp, Fx, Fz, kop = _operands(svgp, aux_data)
    K_mm = be.kernel_fwd_f64(spec, Fz, Fz, hyp)
    p = _recip_no_nan(vars.detach().float()).contiguous()
    A = step.syrk_fwd(kop, p)                                             # K_mn diag(1/var_l) K_nm          :1013
    V = be.gemm_tn(kop, (p * means.detach().float()).contiguous())        # K_mn (means_l / var_l)           :1015-1016
    Sigma_inv, _, _ = ops.spd_inverse_logdet(K_mm.unsqueeze(0) + A)       # :1014 -- no jitter
    mean_terms = ops.bmv64(Sigma_inv, V)
    return mean_terms.to(svgp.dtype), Sigma_inv.to(svgp.dtype)


@torch.no_grad()
def predict_from_precomputed(svgp, index_points, mean_terms, sigma_terms, K_mm_inv=None):
    """All channels of approximate_posterior_params_precomputed_GP_posterior_params (:610-635):
    mean (b, L) = K_bm mean_terms_l,  B (b, L) = K_bb - diag(K_bm K_mm^-1 K_mb) + diag(K_bm sigma_term_l K_mb).

    The two quadratic forms are taken as one, k^T (sigma_term_l - K_mm^-1) k, with the difference formed in float64: the
    large entries the two matrices share cancel there and not in the products.  On the integer tensor-core path (>= 2048
    test rows) the forms are the row dots of the exact integer products K_bm (sigma_term_l - K_mm^-1), as in the step's
    pass D; the SIMT kernels multiply by the float64 difference directly.  sigma_term_l need not be definite."""
    be, spec, hyp, Fx, Fz, kop = _operands(svgp, index_points)
    if K_mm_inv is None:
        K_mm_inv = step.mm_shared(be.kernel_fwd_f64(spec, Fz, Fz, hyp), svgp.jitter)[0]     # :623-625 (with jitter)
    D = sigma_terms.detach().double() - K_mm_inv.detach().double().reshape(1, *K_mm_inv.shape[-2:])
    D = (0.5 * (D + D.transpose(-1, -2))).contiguous()
    L = D.shape[0]
    K_bb = be.kernel_diag_fwd(spec, Fx, Fx, hyp)
    mean = be.gemm_nn(kop, mean_terms.detach().float().contiguous())
    if getattr(kop, "i8", False):
        W = torch.zeros((kop.N, L), dtype=torch.float32, device=D.device)
        _, q = be.scaled_gemm_i8(kop, W, be.planes_i8(D), ndot=L)
    else:
        q = be.rowquad(kop, D)
    B = K_bb[:, None] + q
    return mean.to(svgp.dtype), B.to(svgp.dtype)


@torch.no_grad()
def posterior_predict(svgp, index_points_test, index_points_train, means, vars):
    """(p_m (x, L), p_v (x, L)): approximate_posterior_params (:303-343) for every channel, test points against the
    given training encodings -- the body of the L-loop of bacthing_predict_SVGPVAE_rotated_mnist (:1048-1050).

    The training step's computation with other rows: K_mm in float64 (kernel_fwd_f64), the step's forward SYRK, its
    M x M stage (step.mm_shared, ops.spd_inverse_logdet) and its quadratic forms through the inverse Cholesky factors,
    p_v = K_xx - |LinvK k|^2 + |Linv_l k|^2.  With the training rows as test rows this is the step's p_m / p_v."""
    be, spec, hyp, Fn, Fz, kop_n = _operands(svgp, index_points_train)
    Fx = svgp._features(index_points_test, False).detach().float().contiguous()
    kop_x = be.kernel_fwd(spec, Fx, Fz, hyp, tc=be.want_tc(Fx.shape[0], Fz.shape[0]))
    K_mm = be.kernel_fwd_f64(spec, Fz, Fz, hyp)
    eye = torch.eye(K_mm.shape[0], dtype=K_mm.dtype, device=K_mm.device)
    c = svgp.N_train / float(index_points_train.shape[0])                 # :316, :328
    p = _recip_no_nan(vars.detach().float()).contiguous()
    A = step.syrk_fwd(kop_n, p)
    V = be.gemm_tn(kop_n, (p * means.detach().float()).contiguous())
    _, _, LinvK = step.mm_shared(K_mm, svgp.jitter)                                           # :319
    S, _, Linv = ops.spd_inverse_logdet(K_mm.unsqueeze(0) + c * A + svgp.jitter * eye)       # :328-331
    w = c * ops.bmv64(S, V)
    K_xx = be.kernel_diag_fwd(spec, Fx, Fx, hyp)
    p_m = be.gemm_nn(kop_x, w.float().contiguous())                                          # :332-334
    h = be.rowquad(kop_x, LinvK, tri=True).squeeze(1)
    p_v, _, _ = be.predictive(K_xx, h, be.rowquad(kop_x, Linv, tri=True), None)              # :336-337
    return p_m.to(svgp.dtype), p_v.to(svgp.dtype)
