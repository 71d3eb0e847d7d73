"""The batched SVGP step: all L latent channels of one (sharded) mini-batch in one call.

Replaces the per-channel Python loop of forward_pass_SVGPVAE (SVGPVAE_model.py:865-898) and the
two methods it calls per channel (approximate_posterior_params :303-343, variational_loss
:220-301, gauss_cross_entropy utils.py:483-504).  Same mathematics, reorganised (DESIGN.md):

  pass A   K1 builds K_nm (scaled fp16 hi/lo planes when large), K_mm, kappa; row stats; the only reductions
           over datapoints: A_l = sum_i p_il k_i k_i^T (K2, tcgen05 SYRK) and v_l = sum_i p_il y_il k_i
           -> all-reduce over the N-shards -> replicated float64 M x M stage (K3)
  pass B   per-row predictive moments p_m = K_nm w_l, p_v = kappa - h + |R_l^-1 k_i|^2 (K4)
  [decoder / caller]
  pass C   adjoints of p_m, p_v: weighted SYRK + skinny GEMM -> all-reduce -> hand-written adjoint of the
           M x M stage (mm_channels_bwd / mm_shared_bwd: batched float64 products, no autograd graph)
  pass D   dK_nm = sum_s diag(w_s) K_nm G_s over the 2L stacked matrices [dA+dA^T ; S - Kinv] and the
           row-dots k_i^T dA_l k_i from the same tcgen05 products (weights and dots live in the epilogue),
           then K1's adjoint into features / inducing points / hypers.

Every sum over datapoints inside L3 and the cross entropy is taken against A_l / v_l (e.g.
sum_i p_il k_i^T W_l k_i = <W_l, A_l>), so the (b, m, m) tensor of :286-294 never exists and the
catastrophic cancellation between sum L3 and ce_term (SURVEY F11) happens in float64.
"""
import math

import torch

from . import ops
from ._lib import IMPL_AUTO, IMPL_TC_I8_D3, IMPL_TC_I8_O4
from .backend import Planes, PlanesI8, get_backend

LOG_2PI = 1.8378770664093453      # utils.py:498
LOG_2PI_RT = math.log(2.0 * math.pi)


_COLL = None        # bench.py: [(kind, bytes, start event, end event)] while a collective profile is running


def start_coll_profile():
    global _COLL
    _COLL = []


def stop_coll_profile():
    """-> {"all_reduce" / "all_gather": {"ms", "calls", "bytes"}} (CUDA events on the launch stream around every collective)."""
    global _COLL
    torch.cuda.synchronize()
    out = {}
    for kind, nbytes, e0, e1 in _COLL or []:
        d = out.setdefault(kind, {"ms": 0.0, "calls": 0, "bytes": 0})
        d["ms"] += e0.elapsed_time(e1)
        d["calls"] += 1
        d["bytes"] += nbytes
    _COLL = None
    return out


class _timed_coll:
    def __init__(self, kind, t):
        self.kind, self.nbytes = kind, t.numel() * t.element_size()

    def __enter__(self):
        if _COLL is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *a):
        if _COLL is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            _COLL.append((self.kind, self.nbytes, self.e0, e1))


def _allreduce(t, group):
    if group is not None:
        with _timed_coll("all_reduce", t):
            torch.distributed.all_reduce(t, group=group)
    return t


def _world(group):
    return 1 if group is None else torch.distributed.get_world_size(group)


def _allgather0(t, group):
    """Concatenate the ranks' equally shaped tensors along dim 0 (rank order)."""
    t = t.contiguous()
    W = _world(group)
    out = torch.empty((W * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    with _timed_coll("all_gather", out):
        try:
            torch.distributed.all_gather_into_tensor(out, t, group=group)
        except (RuntimeError, NotImplementedError):          # backends without the flat variant
            torch.distributed.all_gather(list(out.chunk(W, 0)), t, group=group)
    return out


def _own_channels(L, group, enabled=True):
    """Channel ownership of the float64 M x M stage when the datapoints are sharded over `group`: rank r runs K3 for
    channels [r L / W, (r + 1) L / W) and the results are all-gathered (K3 is channel-parallel: per-channel
    factorisations and products; SURVEY 8e).  Needs L % W == 0, otherwise the stage stays replicated."""
    W = _world(group)
    if not enabled or W == 1 or L % W != 0:
        return slice(0, L), False
    r = torch.distributed.get_rank(group)
    return slice(r * (L // W), (r + 1) * (L // W)), True


def syrk_fwd(kop, p, chunk_rows=0):
    """A_l = sum_i p_il k_i k_i^T, the forward SYRK of the step and of the prediction entry points (predict.py).

    Above M = 2048 the integer path multiplies the three digit-plane pairs of order 4 as well (thirteen pairs): what the ten
    leave out is what holds the inducing-point gradient at the tolerance there (DESIGN section 7)."""
    o4 = getattr(kop, "i8", False) and kop.M > 2048
    return get_backend().syrk(kop, p, impl=IMPL_TC_I8_O4 if o4 else IMPL_AUTO, chunk_rows=chunk_rows)


def mm_shared(K, jitter):
    """Channel-independent part of the M x M stage: (K + jI)^-1, its log-det and inverse Cholesky factor (:318-319)."""
    M = K.shape[-1]
    eye = torch.eye(M, dtype=K.dtype, device=K.device)
    return ops.spd_inverse_logdet(K.unsqueeze(0) + jitter * eye)


def mm_channels(A, V, sums, K, Kinv_b, ldK, jitter, c, b_total):
    """Per-channel part of the M x M stage for the channels held by A (Lc, M, M), V (Lc, M), sums (3, Lc)
    (SVGPVAE_model.py:328-331, 339-341, 264-279).  Differentiable w.r.t. A, V, sums, K, Kinv_b, ldK."""
    L, M, _ = A.shape
    eye = torch.eye(M, dtype=A.dtype, device=A.device)
    Kb = K.unsqueeze(0)
    Sigma = Kb + c * A + jitter * eye
    S, _, Linv = ops.spd_inverse_logdet(Sigma)
    w = c * ops.bmv64(S, V)                                   # p_m = K_nm w
    mu_hat = ops.bmm64(w.unsqueeze(0), Kb).squeeze(0)         # K w   (K symmetric)
    a = ops.bmm64(mu_hat.unsqueeze(0), Kinv_b).squeeze(0)     # Kinv mu_hat
    KS = ops.bmm64(Kb, S)
    A_hat = ops.bmm64(KS, Kb)
    ld_Ahat = ops.spd_logdet(A_hat + jitter * eye)
    tr_KinvAhat = (Kinv_b * A_hat).sum((-1, -2))
    kl = 0.5 * (ldK - ld_Ahat - M + tr_KinvAhat + (mu_hat * a).sum(-1))
    Wm = ops.bmm64(ops.bmm64(Kinv_b, A_hat), Kinv_b)          # Kinv A_hat Kinv
    s_pk, s_pyy, s_log = sums[0], sums[1], sums[2]
    s_ph = (Kinv_b * A).sum((-1, -2))
    s_t = (Wm * A).sum((-1, -2))
    Aa = ops.bmv64(A, a)
    recon = -0.5 * (s_pk - s_ph + s_t + s_log + b_total * LOG_2PI_RT + s_pyy - 2.0 * (a * V).sum(-1)
                    + (a * Aa).sum(-1))
    Aw = ops.bmv64(A, w)
    s_ppv = s_pk - s_ph + (S * A).sum((-1, -2))
    ce = -0.5 * (b_total * LOG_2PI + s_log + s_ppv + (w * Aw).sum(-1) - 2.0 * (w * V).sum(-1) + s_pyy)
    return dict(S=S, w=w, Linv=Linv, recon=recon, kl=kl, ce=ce, mu_hat=mu_hat, A_hat=A_hat)


def mm_stage(A, V, sums, K, jitter, c, b_total):
    """Replicated float64 M x M stage (SVGPVAE_model.py:318-319, 328-331, 339-341, 264-279).

    A (L,M,M), V (L,M), sums (3,L) = [sum p kappa, sum p y^2, sum log noise], K (M,M).
    Differentiable w.r.t. all four.  The jitter placement is the reference's: Sigma is built from the
    un-jittered K and jittered before inversion; mu_hat / A_hat use the un-jittered K; Kinv is the
    inverse of K + jI.
    """
    Kinv_b, ldK, LinvK = mm_shared(K, jitter)
    mm = mm_channels(A, V, sums, K, Kinv_b, ldK, jitter, c, b_total)
    mm.update(Kinv=Kinv_b, LinvK=LinvK)
    return mm


# ---- the same stage with a hand-written adjoint -------------------------------------------------------------------------
# mm_channels above is the readable definition (torch autograd chains ops.bmm64 / spd_inverse_logdet / spd_logdet; the
# per-channel API of svgp.py and the tests use it as the cross-check).  The batched step runs the two functions below
# instead: no autograd graph, 4 + 8 batched float64 products per step instead of 4 + ~14, and the state kept between the
# forward and the backward is five (L, M, M) tensors (S, A_hat, its inverse Cholesky factor, Kinv A_hat, Kinv A_hat Kinv)
# next to A instead of the ~16 the graph holds.
def mm_channels_fwd(A, V, sums, K, Kinv_b, ldK, jitter, c, b_total):
    """Values of mm_channels (same formulas, same jitter placement), no graph.  -> (out dict as mm_channels, saved state)."""
    be = get_backend()
    L, M, _ = A.shape
    eye = torch.eye(M, dtype=A.dtype, device=A.device)
    Kb = K.unsqueeze(0)
    Lf, status = be.chol((Kb + c * A + jitter * eye).contiguous())
    ops._check_status(status, "mm_channels_fwd(Sigma)")
    Linv = be.trinv(Lf)
    S = be.ltl(Linv)
    del Lf
    mv = lambda X, x: be.bmm64(X, x.unsqueeze(-1).contiguous()).squeeze(-1)
    w = c * mv(S, V)
    mu_hat = mv(Kb, w)
    a = mv(Kinv_b, mu_hat)
    KS = be.bmm64(Kb, S)
    A_hat = be.bmm64(KS, Kb)
    del KS
    LfA, status = be.chol((A_hat + jitter * eye).contiguous())
    ops._check_status(status, "mm_channels_fwd(A_hat)")
    ld_Ahat = 2.0 * torch.log(torch.diagonal(LfA, dim1=-2, dim2=-1)).sum(-1)
    T = be.bmm64(Kinv_b, A_hat)                               # Kinv A_hat
    tr_KinvAhat = torch.diagonal(T, dim1=-2, dim2=-1).sum(-1)
    kl = 0.5 * (ldK - ld_Ahat - M + tr_KinvAhat + (mu_hat * a).sum(-1))
    Wm = be.bmm64(T, Kinv_b)                                  # Kinv A_hat Kinv
    s_pk, s_pyy, s_log = sums[0], sums[1], sums[2]
    s_ph = (Kinv_b * A).sum((-1, -2))
    s_t = (Wm * A).sum((-1, -2))
    Aa = mv(A, a)
    recon = -0.5 * (s_pk - s_ph + s_t + s_log + b_total * LOG_2PI_RT + s_pyy - 2.0 * (a * V).sum(-1) + (a * Aa).sum(-1))
    Aw = mv(A, w)
    s_ppv = s_pk - s_ph + (S * A).sum((-1, -2))
    ce = -0.5 * (b_total * LOG_2PI + s_log + s_ppv + (w * Aw).sum(-1) - 2.0 * (w * V).sum(-1) + s_pyy)
    out = dict(S=S, w=w, Linv=Linv, recon=recon, kl=kl, ce=ce, mu_hat=mu_hat, A_hat=A_hat)
    saved = dict(A=A, V=V, S=S, w=w, mu_hat=mu_hat, a=a, A_hat=A_hat, LfA=LfA, T=T, Wm=Wm, Aa=Aa, Aw=Aw, c=c)
    return out, saved


def mm_channels_bwd(sv, K, Kinv_b, G_S, G_w, g_recon, g_kl, g_ce):
    """Adjoint of mm_channels_fwd for the channels in `sv`.  G_S (Lc, M, M) / G_w (Lc, M): adjoints of S_l / w_l; g_recon,
    g_kl, g_ce (Lc,): adjoints of the three per-channel scalars.  -> dict(gA, gV, gsums (3, Lc), gK (M, M), gKinv (1, M, M),
    gldK scalar): gK is the DIRECT dependence on K only (Sigma_l, mu_hat, A_hat); what flows through Kinv and ldK is
    returned as their adjoints (mm_shared_bwd turns the sum over all channels into dK once).

    With r, k, e the three scalar adjoints, bars for adjoints (every matrix below is symmetric or used symmetrised):
      w_bar   = G_w - e A w + e V + K mu_bar            a_bar = r V - r A a + k/2 mu          mu_bar = k/2 a + Kinv a_bar
      Ahat_bar = -k/2 (A_hat + jI)^-1 + k/2 Kinv - r/2 Kinv A Kinv
      S_bar   = G_S - e/2 A + c w_bar V^T + K Ahat_bar K               Sigma_bar = -S sym(S_bar) S
      A_bar   = (e + r)/2 Kinv - e/2 S - e/2 w w^T - r/2 Wm - r/2 a a^T + c Sigma_bar
      K_bar   = Ahat_bar K S + (Ahat_bar K S)^T + mu_bar w^T + Sigma_bar
      Kinv_bar = (e + r)/2 A + k/2 A_hat - r/2 (A T + (A T)^T) + a_bar mu^T,   T = Kinv A_hat"""
    be = get_backend()
    A, V, S, w, mu, a, A_hat, T, Wm, c = (sv[k_] for k_ in ("A", "V", "S", "w", "mu_hat", "a", "A_hat", "T", "Wm", "c"))
    Kb = K.unsqueeze(0)
    r, k, e = g_recon, g_kl, g_ce
    r3, k3, e3 = r[:, None, None], k[:, None, None], e[:, None, None]
    mv = lambda X, x: be.bmm64(X, x.unsqueeze(-1).contiguous()).squeeze(-1)
    outer = lambda x, y: x.unsqueeze(-1) * y.unsqueeze(-2)
    # vectors
    a_bar = r[:, None] * (V - sv["Aa"]) + 0.5 * k[:, None] * mu
    mu_bar = 0.5 * k[:, None] * a + mv(Kinv_b, a_bar)
    w_bar = G_w + e[:, None] * (V - sv["Aw"]) + mv(Kb, mu_bar)
    gV = e[:, None] * w + r[:, None] * a + c * mv(S, w_bar)
    gsums = (-0.5 * (e + r)).unsqueeze(0).expand(3, -1).contiguous()
    # adjoint of A_hat
    AhatInv = be.ltl(be.trinv(sv["LfA"]))
    KinvA = be.bmm64(Kinv_b, A)
    Ahat_bar = -0.5 * k3 * AhatInv + 0.5 * k3 * Kinv_b - 0.5 * r3 * be.bmm64(KinvA, Kinv_b)
    del AhatInv, KinvA
    # adjoint of Kinv (this chunk's share)
    Y = be.bmm64(A, T)
    gKinv = (0.5 * (e3 + r3) * A + 0.5 * k3 * A_hat - 0.5 * r3 * (Y + Y.transpose(-1, -2)) + outer(a_bar, mu)).sum(0, keepdim=True)
    del Y
    # through A_hat = K S K
    Pm = be.bmm64(Ahat_bar, Kb)
    Q = be.bmm64(Pm, S)
    S_bar = G_S - 0.5 * e3 * A + c * outer(w_bar, V) + be.bmm64(Kb, Pm)
    del Pm
    Sig_bar = -be.bmm64(be.bmm64(S, (0.5 * (S_bar + S_bar.transpose(-1, -2))).contiguous()), S)
    del S_bar
    gK = (Q + Q.transpose(-1, -2) + outer(mu_bar, w) + Sig_bar).sum(0)
    del Q
    gA = 0.5 * (e3 + r3) * Kinv_b - 0.5 * e3 * (S + outer(w, w)) - 0.5 * r3 * (Wm + outer(a, a)) + c * Sig_bar
    return dict(gA=gA, gV=gV, gsums=gsums, gK=gK, gKinv=gKinv, gldK=0.5 * k.sum())


def mm_shared_bwd(Kinv_b, gKinv, gldK):
    """dK through Kinv = (K + jI)^-1 and ldK = logdet(K + jI) (adjoint of mm_shared)."""
    be = get_backend()
    Gs = (0.5 * (gKinv + gKinv.transpose(-1, -2))).contiguous()
    return (gldK * Kinv_b - be.bmm64(be.bmm64(Kinv_b, Gs), Kinv_b)).squeeze(0)


# state of the stage: about this many (M, M) float64 matrices per channel are alive at the peak of its backward (saved: A, S,
# A_hat, its Cholesky factor, Kinv A_hat, Wm; temporaries of mm_channels_bwd: dS, dA_hat and two products, dSigma, dA)
_MM_LIVE_MATRICES = 12


def mm_chunk_channels(L, M, device, override=None):
    """Channels per chunk of the M x M stage.  One chunk (= the whole stage, fastest) whenever its saved state
    fits the budget; otherwise the stage runs chunk by chunk -- forward without a graph, re-materialised chunk by
    chunk in the backward -- so that L x M x M float64 state is bounded (configs[4]: M = 4096, L = 128 is 17 GB per
    (L, M, M) tensor)."""
    if override:
        return max(1, min(L, int(override)))
    budget = 48e9
    if device.type == "cuda":
        budget = min(budget, 0.2 * torch.cuda.get_device_properties(device).total_memory)
    per_channel = _MM_LIVE_MATRICES * 8.0 * M * M
    if per_channel * L <= budget:
        return L
    lc = max(1, int(budget // per_channel))
    nchunk = -(-L // lc)
    return -(-L // nchunk)


class _SVGPStep(torch.autograd.Function):
    @staticmethod
    def forward(ctx, Fx, Fz, hyp, y, noise, cfg):
        be = get_backend()
        spec, jitter, N_train = cfg["spec"], cfg["jitter"], cfg["N_train"]
        group, clip = cfg.get("group"), cfg.get("clip_pv")
        Fx32, Fz32, hyp32 = Fx.float().contiguous(), Fz.float().contiguous(), hyp.float().contiguous()
        y32, n32 = y.float().contiguous(), noise.float().contiguous()
        N, L = y32.shape
        M = Fz32.shape[0]
        tc = cfg.get("tc")
        # the tensor-core kernels need tensor-core sized problems (backend.want_tc is the library's own predicate)
        tc = be.want_tc(N, M) if tc is None else (bool(tc) and be.want_tc(N, M))
        b_total = float(N)
        if group is not None:
            # one K_nm format on every rank: the chunked, channel-sharded backward gathers the adjoint operand planes in that
            # format, so one shard below the tensor-core size takes the whole group to the SIMT kernels.  [rows, 1 - tc]
            # summed over the ranks: the batch size and the format in one all-reduce and one host read
            count = torch.tensor([float(N), 0.0 if tc else 1.0], dtype=torch.float64, device=y32.device)
            _allreduce(count, group)
            b_total, n_simt = count.tolist()
            tc = n_simt == 0

        # pass A
        kop = be.kernel_fwd(spec, Fx32, Fz32, hyp32, tc=tc)
        # K_mm in float64 arithmetic: the M x M stage amplifies its entries' errors by cond(K + J) and more
        K64 = be.kernel_fwd_f64(spec, Fz32, Fz32, hyp32)
        kappa = be.kernel_diag_fwd(spec, Fx32, Fx32, hyp32)
        p, py, sums = be.rowstats(y32, n32, kappa)
        A = syrk_fwd(kop, p, chunk_rows=cfg.get("chunk_rows", 0))
        V = be.gemm_tn(kop, py)
        if group is not None:
            for t in (A, V, sums):
                _allreduce(t, group)
        c = N_train / b_total

        tri = cfg.get("tri", True)
        own, sharded = _own_channels(L, group, cfg.get("shard_k3", True))
        lc = mm_chunk_channels(own.stop - own.start, M, y32.device, cfg.get("mm_chunk"))
        one_chunk = lc >= own.stop - own.start
        if one_chunk:
            Kinv, ldK, LinvK = mm_shared(K64, jitter)
            mm, saved = mm_channels_fwd(A[own].contiguous(), V[own].contiguous(), sums[:, own].contiguous(), K64, Kinv, ldK, jitter, c, b_total)
            # pass B
            S, w, Linv = mm["S"], mm["w"], mm["Linv"]
            if sharded:                      # every rank needs all channels' S_l, w_l and factors for ITS rows
                S, w, Linv = _allgather0(S, group), _allgather0(w, group), _allgather0(Linv, group)
            # quadratic forms through the Cholesky factors: |R^-1 k|^2 is a sum of squares (half the MMA work and
            # no cancellation between the large entries of S_l / Kinv)
            if tri:
                h = be.rowquad(kop, LinvK, tri=True).squeeze(1)
                q1 = be.rowquad(kop, Linv, tri=True)
            else:
                h = be.rowquad(kop, Kinv).squeeze(1)
                q1 = be.rowquad(kop, S)
            recon, kl, ce0 = mm["recon"].clone(), mm["kl"].clone(), mm["ce"]
            mu_hat, A_hat = mm["mu_hat"], mm["A_hat"]
            if sharded:
                recon, kl, ce0, mu_hat = (_allgather0(t, group) for t in (recon, kl, ce0, mu_hat))
                A_hat = _allgather0(A_hat, group) if cfg.get("return_A_hat", True) else None
            del Linv, LinvK, mm
        else:
            # chunked M x M stage: no graph in the forward (the backward re-materialises it chunk by chunk); S is
            # the only (L, M, M) result that stays (pass D reads it), the factors feed the row quads chunk by chunk
            saved = None
            want_Ahat = cfg.get("return_A_hat", True)
            S = torch.empty_like(A)
            A_hat = torch.empty_like(A) if want_Ahat else None
            w = torch.empty_like(V)
            mu_hat = torch.empty_like(V)
            recon, kl, ce0 = (torch.empty(L, dtype=torch.float64, device=A.device) for _ in range(3))
            q1 = torch.empty((N, L), dtype=torch.float32, device=A.device)
            W_, L_own = _world(group) if sharded else 1, own.stop - own.start
            with torch.no_grad():
                Kinv, ldK, LinvK = mm_shared(K64, jitter)
                h = (be.rowquad(kop, LinvK, tri=True) if tri else be.rowquad(kop, Kinv)).squeeze(1)
                for l0 in range(own.start, own.stop, lc):
                    sl = slice(l0, min(own.stop, l0 + lc))
                    mc, _ = mm_channels_fwd(A[sl], V[sl], sums[:, sl].contiguous(), K64, Kinv, ldK, jitter, c, b_total)
                    S[sl], w[sl], mu_hat[sl] = mc["S"], mc["w"], mc["mu_hat"]
                    recon[sl], kl[sl], ce0[sl] = mc["recon"], mc["kl"], mc["ce"]
                    if want_Ahat:
                        A_hat[sl] = mc["A_hat"]
                    F = mc["Linv"] if tri else mc["S"]
                    if sharded:
                        # every rank needs every channel's factor for the quadratic forms of ITS rows: gather this
                        # chunk of all ranks (same chunking everywhere) and scatter the pieces to their columns
                        n, off = sl.stop - sl.start, sl.start - own.start
                        Fall = _allgather0(F, group)
                        for r in range(W_):
                            be.rowquad(kop, Fall[r * n:(r + 1) * n], tri=tri, out=q1[:, r * L_own + off:r * L_own + off + n])
                        del Fall
                    else:
                        be.rowquad(kop, F, tri=tri, out=q1[:, sl])
                    del mc, F
                if sharded:
                    S = _allgather0(S[own], group)
                    w, mu_hat = _allgather0(w[own], group), _allgather0(mu_hat[own], group)
                    recon, kl, ce0 = (_allgather0(t[own], group) for t in (recon, kl, ce0))
                    if want_Ahat:
                        A_hat = _allgather0(A_hat[own], group)
        pm = be.gemm_nn(kop, w.float().contiguous())
        pv, clipsum, mask = be.predictive(kappa, h, q1, p, clip)
        ce = ce0.clone()
        if clip:
            _allreduce(clipsum, group)
            ce = ce - 0.5 * clipsum

        ctx.cfg, ctx.kop, ctx.mm_saved, ctx.lc = cfg, kop, saved, lc
        ctx.mm_in = (A, V, sums, K64, ldK)
        ctx.own, ctx.sharded, ctx.one_chunk = own, sharded, one_chunk
        ctx.b_total, ctx.c = b_total, c
        cfg["_b_total"] = b_total                      # read back by svgp_step (a host number, not a tensor)
        ctx.save_for_backward(Fx32, Fz32, hyp32, y32, n32, p, kappa, h, pv, q1 if clip else pv, mask if clip else pv, S, w, Kinv)
        ctx.in_dtypes = (Fx.dtype, Fz.dtype, hyp.dtype, y.dtype, noise.dtype)
        out_dt = y.dtype
        if A_hat is None:
            ctx.mark_non_differentiable(mu_hat)
        else:
            ctx.mark_non_differentiable(mu_hat, A_hat)
        return pm.to(out_dt), pv.to(out_dt), recon, kl, ce, mu_hat, A_hat

    @staticmethod
    def backward(ctx, g_pm, g_pv, g_recon, g_kl, g_ce, _g_mu, _g_Ahat):
        be = get_backend()
        cfg, kop = ctx.cfg, ctx.kop
        spec, group, clip = cfg["spec"], cfg.get("group"), cfg.get("clip_pv")
        Fx, Fz, hyp, y, noise, p, kappa, h, pv, q1raw, mask, S, w, Kinv = ctx.saved_tensors
        N, L = y.shape
        M = Fz.shape[0]
        dev = y.device
        zeros_L = torch.zeros(L, dtype=torch.float64, device=dev)
        g_recon = zeros_L if g_recon is None else g_recon.double()
        g_kl = zeros_L if g_kl is None else g_kl.double()
        g_ce = zeros_L if g_ce is None else g_ce.double()
        g_pm = torch.zeros_like(y) if g_pm is None else g_pm.float().contiguous()
        g_pv = torch.zeros_like(y) if g_pv is None else g_pv.float().contiguous()
        # scalar adjoints are per-rank shares of the same global scalars: total = sum over ranks
        sc = torch.stack([g_recon, g_kl, g_ce])
        _allreduce(sc, group)
        g_recon, g_kl, g_ce = sc[0], sc[1], sc[2]

        # ---- pass C: row-local adjoints of the predictive moments --------------------------------
        # one fused pass (svgp_rowterms_bwd_pre): dObjective/dq1 (clipped entries only see the clip correction of the
        # collapsed CE sum), the stacked row weights [p | 2 dq1] and [p y | g_pm] of pass D, sum_l dq1 = d/d kappa_i (= -d/d h_i)
        clip_args = (mask, pv, kappa, h, q1raw, g_ce.float().contiguous()) if clip else None
        G_q1, Wstack, PYstack, G_p_clip, G_kappa = be.rowterms_bwd_pre(g_pv if g_pv is not None else None, g_pm, p, y, clip_args)
        # the adjoint SYRK and the S_l - Kinv family of pass D tolerate the three leading digits of both operands (8 of the 10
        # digit-plane pairs) up to M = 2048: they enter the parameter gradients only, not the values (DESIGN section 7; at
        # M = 4096, where dZ sits at the tolerance, the operand-format model shows 7.5e-5 -> 8.2e-5: all ten pairs there)
        d3 = getattr(kop, "i8", False) and M <= 2048
        G_S = be.syrk(kop, G_q1, impl=IMPL_TC_I8_D3 if d3 else IMPL_AUTO, chunk_rows=cfg.get("chunk_rows", 0))
        G_w = be.gemm_tn(kop, g_pm)
        for t in (G_S, G_w):
            _allreduce(t, group)
        if getattr(kop, "i8", False):
            # last use of the column-scaled K^T planes and of the fp16 row planes: pass D reads the row-scaled digit planes
            # only (configs[4]: 33 GB per GPU at N = 1e6, M = 4096 returned before the adjoint of the M x M stage allocates)
            kop.Kc = kop.cscale = kop.Kh = kop.Kl = None
        # d/d Kinv of h_i = k_i^T Kinv k_i is sum_i (-G_kappa_i) k_i k_i^T = -sum_l G_S,l.  Taking it from G_S (instead
        # of a separate single-channel SYRK) is not only free: both adjoints are amplified by the squared inverses
        # downstream (-Kinv G Kinv and -S_l G S_l, |Kinv|, |S_l| ~ 1 / jitter in the directions the data does not
        # see) and only cancel there if they carry the SAME rounding noise.  (Formed below from this rank's channels.)

        # ---- adjoint of the replicated M x M stage -----------------------------------------------
        A_, V_, sums_, K_, ldK_ = ctx.mm_in
        lc = ctx.lc
        own, sharded = ctx.own, ctx.sharded
        if ctx.one_chunk:
            # (channel-sharded K3: this rank differentiates its own channels; dKinv likewise is its channels' share)
            g = mm_channels_bwd(ctx.mm_saved, K_, Kinv, G_S[own], G_w[own], g_recon[own], g_kl[own], g_ce[own])
            gA, gV, gsums = g["gA"], g["gV"], g["gsums"]
            gK = g["gK"] + mm_shared_bwd(Kinv, g["gKinv"] - G_S[own].sum(0, keepdim=True), g["gldK"])
            # the saved state of the stage, A_l and dS_l are dead from here on (17 GB each at M = 4096, L = 128)
            ctx.mm_saved = ctx.mm_in = None
            del A_, G_S, g
            if sharded:
                gA, gV = _allgather0(gA, group), _allgather0(gV, group)
                gsums = _allgather0(gsums.t().contiguous(), group).t().contiguous()
                _allreduce(gK, group)
            # ---- pass D: back to the rows --------------------------------------------------------
            # dK_nm and k^T (dA + dA^T) k from ONE pass over the products K G_s: stacked matrices
            # [dA + dA^T ; S - Kinv] with per-row weights [p | 2 dq1] applied in the epilogue.  p_v = kappa - k^T (Kinv - S_l) k:
            # the difference is formed in float64 BEFORE the fp16 split, so the 1 / jitter-sized components that
            # Kinv and S_l share never enter the tensor-core products
            if kop.tc and getattr(kop, "i8", False):
                # both families as four int8 digit planes each for the exact integer products: K (dA + dA^T) cancels by
                # 10^2..10^3 against the entries of dA (the truncating fp16 accumulation of round 1 left 3e-4 in dZ at
                # M = 1024), and at M = 2048 the S - Kinv family does not tolerate it either (6e-5 of dZ, measured with
                # tests/probes/ablate_i8_probe.py)
                Gstack = be.planes_i8_alloc(2 * L, M, M, dev)
                for l0 in range(0, L, 16):
                    be.planes_i8_into(gA[l0:l0 + 16] + gA[l0:l0 + 16].transpose(-1, -2), Gstack, l0)
                    be.planes_i8_into(S[l0:l0 + 16] - Kinv, Gstack, L + l0)
            elif kop.tc:
                # operand planes filled in pieces of 16 channels: no (2L, M, M) float64 copy next to gA and S
                hi = torch.empty((2 * L, M, M), dtype=torch.float16, device=dev)
                lo = torch.empty_like(hi)
                inv = torch.empty(2 * L, dtype=torch.float32, device=dev)
                for l0 in range(0, L, 16):
                    be.planes_into(gA[l0:l0 + 16] + gA[l0:l0 + 16].transpose(-1, -2), hi, lo, inv, l0)
                    be.planes_into(S[l0:l0 + 16] - Kinv, hi, lo, inv, L + l0)
                Gstack = Planes(hi, lo, inv)
            else:
                Gstack = torch.cat([gA + gA.transpose(-1, -2), S - Kinv], dim=0).contiguous()
            del gA
        else:
            # re-materialise the stage chunk by chunk; every chunk's dA_l + dA_l^T goes straight into the operand
            # planes of pass D, so no second (L, M, M) float64 tensor is alive next to A, S and G_S
            jitter, c, b_total = cfg["jitter"], ctx.c, ctx.b_total
            use_i8 = kop.tc and getattr(kop, "i8", False)
            if use_i8:
                GA = be.planes_i8_alloc(2 * L, M, M, dev)
                put = lambda X, at: be.planes_i8_into(X, GA, at)
            elif kop.tc:
                hi = torch.empty((2 * L, M, M), dtype=torch.float16, device=dev)
                lo = torch.empty_like(hi)
                inv = torch.empty(2 * L, dtype=torch.float32, device=dev)
                put = lambda X, at: be.planes_into(X, hi, lo, inv, at)
            else:
                G64 = torch.empty((2 * L, M, M), dtype=torch.float64, device=dev)

                def put(X, at):
                    G64[at:at + X.shape[0]] = X
            gV, gsums = torch.empty_like(V_), torch.empty_like(sums_)
            gK = torch.zeros_like(K_)
            gKinv = -G_S[own].sum(0, keepdim=True)          # this rank's channels' share of dKinv (all of it when not sharded)
            gldK = torch.zeros((), dtype=torch.float64, device=dev)
            for l0 in range(own.start, own.stop, lc):
                sl = slice(l0, min(own.stop, l0 + lc))
                _, sv = mm_channels_fwd(A_[sl], V_[sl], sums_[:, sl].contiguous(), K_, Kinv, ldK_, jitter, c, b_total)
                g = mm_channels_bwd(sv, K_, Kinv, G_S[sl], G_w[sl], g_recon[sl], g_kl[sl], g_ce[sl])
                del sv
                put(g["gA"] + g["gA"].transpose(-1, -2), l0)
                gV[sl] = g["gV"]
                gsums[:, sl] = g["gsums"]
                gK += g["gK"]
                gKinv += g["gKinv"]
                gldK += g["gldK"]
                del g
            gK += mm_shared_bwd(Kinv, gKinv, gldK)
            del G_S, gKinv
            if sharded:
                # the other ranks' dA_l + dA_l^T (operand planes / float64), dv_l and row-sum adjoints; dK_mm summed
                if use_i8:
                    pl = GA.planes.view(GA.planes.shape[0], 2 * L, M, -1)
                    for d in range(pl.shape[0]):
                        pl[d][:L] = _allgather0(pl[d][own], group)
                    GA.scale.view(2 * L, M)[:L] = _allgather0(GA.scale.view(2 * L, M)[own], group)
                elif kop.tc:
                    hi[:L] = _allgather0(hi[own], group)
                    lo[:L] = _allgather0(lo[own], group)
                    inv[:L] = _allgather0(inv[own], group)
                else:
                    G64[:L] = _allgather0(G64[own], group)
                gV = _allgather0(gV[own], group)
                gsums = _allgather0(gsums[:, own].t().contiguous(), group).t().contiguous()
                _allreduce(gK, group)
            for l0 in range(0, L, lc):
                put(S[l0:l0 + lc] - Kinv, L + l0)
            Gstack = GA if use_i8 else (Planes(hi, lo, inv) if kop.tc else G64)
        if isinstance(Gstack, PlanesI8):
            # the S_l - Kinv family (second half of the stack) with the three leading digits: 8 instead of 10 pairs
            G_K, kGk = be.scaled_gemm_i8(kop, Wstack, Gstack, ndot=L, nfull=L if d3 else 2 * L)
        else:
            G_K, kGk = be.scaled_gemm(kop, Wstack, Gstack, ndot=L)
        del Wstack, Gstack
        # rank-2L part of dK_nm in one pass over it: [p*y | g_pm] (N, 2L) @ [dV ; w] (2L, M)   (via v_l and via p_m)
        be.gemm_f32(PYstack, torch.cat([gV.float(), w.float()], dim=0).contiguous(), out=G_K)
        del PYstack
        # dy, dnoise and the rest of d/d kappa, fused (svgp_rowterms_bwd_post): kGk / 2 = k^T dA k
        G_py = be.gemm_nn(kop, gV.float().contiguous())
        G_y, G_noise, G_kappa = be.rowterms_bwd_post(y, noise, p, kappa, kGk, G_py, gsums.contiguous(), G_p_clip, G_kappa)

        # ---- K1 adjoint ----------------------------------------------------------------------------
        need_x = ctx.needs_input_grad[0]
        Gk = G_K if G_K.shape[1] == M else G_K[:, :M].contiguous()
        dFx, dFz, dhyp = be.kernel_bwd(spec, Fx, Fz, hyp, Gk, need_x=need_x, need_z=True)
        dkx, dky, dhyp_d = be.kernel_diag_bwd(spec, Fx, Fx, hyp, G_kappa.contiguous())
        dhyp = dhyp + dhyp_d
        if need_x:
            dFx = dFx + dkx + dky
        # replicated K_mm: every rank holds the full adjoint -> give each rank a 1/world share so that the
        # caller's sum over ranks (parameters are replicated) counts it once
        share = 1.0 / _world(group)
        gKf = (share * gK).float().contiguous()
        dZa, dZb, dhyp_m = be.kernel_bwd(spec, Fz, Fz, hyp, gKf, need_x=True, need_z=True)
        dFz = dFz + dZa.double() + dZb
        dhyp = dhyp + dhyp_m
        ctx.mm_saved = ctx.mm_in = None
        dx, dz, dh, dy, dn = ctx.in_dtypes
        return (dFx.to(dx) if need_x else None, dFz.to(dz), dhyp.to(dh), G_y.to(dy), G_noise.to(dn), None)


def svgp_step(spec, Fx, Fz, hyp, y, noise, *, N_train, jitter, clip_pv=None, group=None, tc=None, tri=True,
              chunk_rows=0, mm_chunk=None, return_A_hat=True, shard_k3=True):
    """All-channel SVGP step on one shard of datapoints.

    Fx (N, d) data features, Fz (M, d) inducing features, hyp (4,) kernel hypers, y / noise (N, L)
    encoder means / variances.  ``group``: torch.distributed group over which the datapoints are
    sharded (None = single process); A_l, v_l and the scalar sums are all-reduced over it.

    Returns dict(p_m, p_v (N, L); recon_l, kl_l, ce_l (L,) float64 -- GLOBAL sums, identical on all
    ranks; mu_hat (L, M), A_hat (L, M, M) float64, detached; b_total = the all-reduced number of datapoints).
    ``shard_k3``: with a group of W ranks and L % W == 0, every rank runs the float64 M x M stage for L / W channels and
    the results are all-gathered (default); False keeps the stage replicated.
    ``mm_chunk``: channels per chunk of the float64 M x M stage (default: one chunk while its state fits, see
    mm_chunk_channels); ``return_A_hat=False`` skips the (L, M, M) A_hat output on the chunked path.
    Gradient convention when sharded: make each rank's loss ``local terms + global terms / world``;
    gradients of replicated parameters then come out as per-rank partial sums (sum them).
    """
    cfg = dict(spec=spec, N_train=float(N_train), jitter=float(jitter), clip_pv=clip_pv, group=group, tc=tc, tri=tri,
               chunk_rows=chunk_rows, mm_chunk=mm_chunk, return_A_hat=return_A_hat, shard_k3=shard_k3)
    pm, pv, recon, kl, ce, mu_hat, A_hat = _SVGPStep.apply(Fx, Fz, hyp, y, noise, cfg)
    return dict(p_m=pm, p_v=pv, recon_l=recon, kl_l=kl, ce_l=ce, mu_hat=mu_hat, A_hat=A_hat, b_total=cfg["_b_total"])


def elbo_terms(res, b, N_train):
    """SVGPVAE_model.py:880-898 on the per-channel sums: inside_elbo, ce_term, KL_term (Hensman branch)."""
    recon, kl, ce = res["recon_l"].sum(), res["kl_l"].sum(), res["ce_l"].sum()
    inside = recon - (b / N_train) * kl
    return dict(inside_elbo_recon=recon, inside_elbo_kl=kl, inside_elbo=inside, ce_term=ce, KL_term=-ce + inside)
