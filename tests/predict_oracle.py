"""float64 restatement of the three prediction entry points of svgp_vae_b200/predict.py -- TEST INFRASTRUCTURE ONLY.

Device-agnostic torch float64, every latent channel at once.  The formulas are those of the literal oracle:

  posterior_predict            oracle/svgp_literal.py:158-178 (approximate_posterior_params, :303-343 of the reference)
                               with test rows x and training rows n; c = N_train / n; jitter on K_mm^-1 and on Sigma_l
  precompute                   SVGPVAE_model.py:989-1023 (tests/golden/make_reference_golden.py feeds it): Sigma_l =
                               K_mm + K_mn diag(1 / var_l) K_nm, inverted WITHOUT jitter and without the N_train / b factor
  predict_from_precomputed     oracle/svgp_literal.py:312-322 (:610-635): K_mm^-1 with jitter unless the caller passes it

The kernel matrices come from a callable ``kern(x, y, diag=False)``.  ``spec_kernel`` gives it for the continuous
productSVGP specs from tests/ard_oracle.kernel_value (SE, Matern, linear, cosine, with or without ARD), evaluated block
by block of rows so that no (N, M, d) tensor of the whole problem is formed.  Each block is the exact pairwise
difference of the oracle, so no squared-distance expansion (and its cancellation) is involved.
"""
import torch

from ard_oracle import kernel_value

F64 = torch.float64


def recip_no_nan(x):
    """tf.math.reciprocal_no_nan: 1 / x, 0 where x == 0."""
    return torch.where(x == 0, torch.zeros_like(x), 1.0 / torch.where(x == 0, torch.ones_like(x), x))


def spec_kernel(spec, hyp, rows=2048):
    """kern(x, y, diag=False) of a productSVGP spec: float64 K(x, y), or k(x_i, y_i) with diag=True."""
    hyp = torch.as_tensor(hyp).to(F64)

    def kern(x, y, diag=False):
        x, y = x.to(F64), y.to(F64)
        h = hyp.to(x.device)
        if diag:
            return kernel_value(spec, x, y, h, pairwise=False)
        return torch.cat([kernel_value(spec, x[i:i + rows], y, h) for i in range(0, x.shape[0], rows)], 0)

    return kern


def _eye(M, like):
    return torch.eye(M, dtype=F64, device=like.device)


def _quad(K_xm, S):
    """diag(K_xm S K_xm^T) for every channel of S (L, M, M) -> (x, L)."""
    return torch.stack([((K_xm @ S_l) * K_xm).sum(1) for S_l in S], 1)


def _weighted_gram(K_nm, p):
    """A_l = K_mn diag(p_l) K_nm for every column l of p (n, L) -> (L, M, M)."""
    return torch.stack([K_nm.T @ (p[:, l:l + 1] * K_nm) for l in range(p.shape[1])])


def posterior_predict(kern, Z, X_test, X_train, means, vars_, jitter, N_train):
    """-> (p_m, p_v) (x, L): approximate_posterior_params of every channel, test rows against the training rows."""
    Z, Xt, Xn = Z.to(F64), X_test.to(F64), X_train.to(F64)
    means, vars_ = means.to(F64), vars_.to(F64)
    M = Z.shape[0]
    c = float(N_train) / float(Xn.shape[0])
    K_mm, K_nm, K_xm = kern(Z, Z), kern(Xn, Z), kern(Xt, Z)
    K_xx = kern(Xt, Xt, diag=True)
    eye = _eye(M, K_mm)
    p = recip_no_nan(vars_)
    K_mm_inv = torch.linalg.inv(K_mm + jitter * eye)
    S = torch.linalg.inv(K_mm + c * _weighted_gram(K_nm, p) + jitter * eye)
    v = (p * means).T @ K_nm                                                    # (L, M) = K_mn (means_l / var_l)
    w = c * (S @ v.unsqueeze(-1)).squeeze(-1)
    p_m = K_xm @ w.T
    p_v = K_xx[:, None] - ((K_xm @ K_mm_inv) * K_xm).sum(1)[:, None] + _quad(K_xm, S)
    return p_m, p_v


def precompute(kern, Z, X, means, vars_):
    """-> (mean_terms (L, M), inv_Sigma (L, M, M)) of precompute_GP_params_SVGPVAE (no jitter, no N_train / b)."""
    Z, X, means, vars_ = Z.to(F64), X.to(F64), means.to(F64), vars_.to(F64)
    K_mm, K_nm = kern(Z, Z), kern(X, Z)
    p = recip_no_nan(vars_)
    inv_Sigma = torch.linalg.inv(K_mm + _weighted_gram(K_nm, p))
    v = (p * means).T @ K_nm
    return (inv_Sigma @ v.unsqueeze(-1)).squeeze(-1), inv_Sigma


def predict_from_precomputed(kern, Z, X, mean_terms, sigma_terms, jitter, K_mm_inv=None):
    """-> (mean, B) (b, L): approximate_posterior_params_precomputed_GP_posterior_params of every channel."""
    Z, X = Z.to(F64), X.to(F64)
    mean_terms, sigma_terms = mean_terms.to(F64), sigma_terms.to(F64)
    if K_mm_inv is None:
        K_mm = kern(Z, Z)
        K_mm_inv = torch.linalg.inv(K_mm + jitter * _eye(Z.shape[0], K_mm))
    K_bm = kern(X, Z)
    K_bb = kern(X, X, diag=True)
    mean = K_bm @ mean_terms.T
    B = K_bb[:, None] - ((K_bm @ K_mm_inv.to(F64)) * K_bm).sum(1)[:, None] + _quad(K_bm, sigma_terms)
    return mean, B
