"""Tensor-level wrappers around the C ABI (one method per entry point of include/svgp_b200.h).

``CudaBackend`` is the only backend the product ships: PyTorch supplies device memory and the
current stream, every FLOP runs in libsvgp_b200.so.  The host logic in ops.py / step.py talks to
``get_backend()`` so that the CPU test-suite can exercise that logic against a float64 oracle
backend (tests/oracle_backend.py, injected with ``set_backend_for_tests``) -- the package itself
never imports the oracle and never falls back to it.
"""
import ctypes
import os

import torch

from . import _lib
from ._lib import IMPL_AUTO, IMPL_SIMT, IMPL_TC, IMPL_TC_I8, IMPL_TC_I8_D3, IMPL_TC_I8_O4, KopStruct


class Kop:
    """K_nm (N x M) in the storage the GEMM-class kernels read.

    SIMT: one fp32 matrix ``K``.  TC: scaled fp16 (hi, lo) planes of K_nm (``Kh``/``Kl``) and of its transpose
    (``Kth``/``Ktl``) plus the device scale record ``kscale`` = {scale, 1/scale, ...} (see tc_engine.cu);
    ``value()`` reassembles (hi + lo) / scale when a plain matrix is asked for.
    """

    def __init__(self, K=None, Kh=None, Kl=None, Kth=None, Ktl=None, kscale=None, N=None, M=None):
        self.K, self.Kh, self.Kl, self.Kth, self.Ktl, self.kscale = K, Kh, Kl, Kth, Ktl, kscale
        ref = K if K is not None else Kh
        self.N = ref.shape[0] if N is None else N
        self.M = ref.shape[1] if M is None else M
        # int8 digit planes of the exact integer tensor-core products (svgp_kernel_fwd_i8): Kr (4, N, ldkr) row-scaled,
        # Kc (4, ceil(N / 128), M, 128) column-scaled and datapoint-blocked, with their scales
        self.Kr = self.rscale = self.Kc = self.cscale = None
        self.Kr_bias = None              # svgp_i8_pair_bias of Kr, formed on first use

    @property
    def tc(self):
        return self.Kh is not None or self.Kr is not None

    @property
    def i8(self):
        return self.Kr is not None

    def value_i8(self, which="r"):
        """K_nm reassembled from the digit planes (float64): which = "r" row-scaled planes, "c" column-scaled ones."""
        if which == "r":
            d = self.Kr.double()
            return ((((d[0] * 256.0 + d[1]) * 256.0 + d[2]) * 256.0 + d[3]) * self.rscale.double()[:, None])[:, : self.M]
        d = self.Kc.double()                                             # (4, nblk, M, 128)
        v = (((d[0] * 256.0 + d[1]) * 256.0 + d[2]) * 256.0 + d[3]) * self.cscale.double()[None, :, None]
        return v.permute(0, 2, 1).reshape(-1, self.M)[: self.N]

    @property
    def device(self):
        return (self.K if self.K is not None else (self.Kh if self.Kh is not None else self.Kr)).device

    def value(self):
        if self.K is not None:
            return self.K[: self.N, : self.M]
        return (self.Kh[: self.N, : self.M].float() + self.Kl[: self.N, : self.M].float()) * self.kscale[1]

    def value_t(self):
        """K_nm^T (M x N) reassembled from the datapoint-blocked transposed planes."""
        t = (self.Kth.float() + self.Ktl.float()) * self.kscale[1]            # (nblk, M, 64)
        return t.permute(1, 0, 2).reshape(self.M, -1)[:, : self.N]

    def struct(self):
        s = KopStruct()
        s.K = self.K.data_ptr() if self.K is not None else None
        s.Kh = self.Kh.data_ptr() if self.Kh is not None else None
        s.Kl = self.Kl.data_ptr() if self.Kl is not None else None
        s.Kth = self.Kth.data_ptr() if self.Kth is not None else None
        s.Ktl = self.Ktl.data_ptr() if self.Ktl is not None else None
        s.kscale = self.kscale.data_ptr() if self.kscale is not None else None
        s.N, s.M = self.N, self.M
        s.ldk = self.K.stride(0) if self.K is not None else 0
        s.ldkh = self.Kh.stride(0) if self.Kh is not None else 0
        s.ldkt = self.Kth.stride(0) if self.Kth is not None else 0
        s.Kr = self.Kr.data_ptr() if self.Kr is not None else None
        s.rscale = self.rscale.data_ptr() if self.rscale is not None else None
        s.Kc = self.Kc.data_ptr() if self.Kc is not None else None
        s.cscale = self.cscale.data_ptr() if self.cscale is not None else None
        s.ldkr = self.Kr.stride(1) if self.Kr is not None else 0
        return s


class Planes:
    """fp16 (hi, lo) operand planes of a (B, M, M) float64 batch with per-matrix 1/scale (svgp_split_f16)."""

    def __init__(self, hi, lo, inv):
        self.hi, self.lo, self.inv = hi, lo, inv


class PlanesI8:
    """int8 digit planes of a (B, R, C) float64 batch with one scale per row (svgp_split_i8): planes (S, B * R, ldp),
    scale (B * R,); x[b, r, c] ~= scale[b R + r] * sum_s planes[s, b R + r, c] 256^(S - 1 - s)."""

    def __init__(self, planes, scale, B, R, C):
        self.planes, self.scale, self.B, self.R, self.C = planes, scale, B, R, C

    def value(self):
        S = self.planes.shape[0]
        d = self.planes.double()
        v = sum(d[s] * 256.0 ** (S - 1 - s) for s in range(S)) * self.scale.double()[:, None]
        return v[:, : self.C].reshape(self.B, self.R, self.C)


_PROFILE = None


def _call(name, *args):
    """_lib.call, optionally bracketed by CUDA events on the launch stream (bench.py's per-kernel times)."""
    if _PROFILE is None:
        return _lib.call(name, *args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = _lib.call(name, *args)
    e1.record()
    _PROFILE.append((name, e0, e1))
    return rc


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t):
    assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous(), (t.dtype, t.shape, t.is_contiguous())
    return t


def _f64c(t):
    assert t.is_cuda and t.dtype == torch.float64 and t.is_contiguous(), (t.dtype, t.shape)
    return t


def _pad(n, m):
    return (n + m - 1) // m * m


class CudaBackend:
    name = "cuda-sm100a"

    def __init__(self):
        _lib.load()
        if not torch.cuda.is_available():
            raise _lib.SvgpLibraryError("svgp_vae_b200 needs a CUDA device (no CPU fallback)")
        if not _lib.load().svgp_device_ok():
            raise _lib.SvgpLibraryError("svgp_vae_b200 kernels are built for sm_100a only (B200)")
        self.launches = 0          # kernels launched through this backend (bench reports it)
        self.tc_min_rows = max(2048, int(os.environ.get("SVGP_TC_MIN_ROWS", "2048")))    # the library needs N >= 2048 (tc_shape_ok)
        self.use_i8 = os.environ.get("SVGP_TC_I8", "1") != "0"
        # expected value of the dropped digit-plane pairs added inside the integer scaled GEMM: from M = 2048 up by default (the
        # coherent 1e-9 per entry it removes costs the hyper-parameter gradients 2e-5 at M = 2048 and 7e-4 at M = 4096, nothing
        # measurable at M = 1024, and the two extra adds per column cost pass D 2.5 % there); SVGP_I8_DEBIAS=1 / 0: always / never
        self.i8_debias = {"0": 1 << 62, "1": 0}.get(os.environ.get("SVGP_I8_DEBIAS", ""), 2048)

    def start_profile(self):
        global _PROFILE
        _PROFILE = []

    def stop_profile(self):
        """-> {entry point: {"ms": total device time, "calls": n, "max_ms": longest call}} since start_profile()."""
        global _PROFILE
        torch.cuda.synchronize()
        out = {}
        for name, e0, e1 in _PROFILE or []:
            d = out.setdefault(name, {"ms": 0.0, "calls": 0, "max_ms": 0.0})
            t = e0.elapsed_time(e1)
            d["ms"] += t
            d["calls"] += 1
            d["max_ms"] = max(d["max_ms"], t)
        _PROFILE = None
        return out

    # ---- K1 --------------------------------------------------------------------------------
    def want_tc(self, N, M):
        return N >= self.tc_min_rows and M >= 128

    def want_i8(self, N, M):
        """Exact integer tensor-core products (SYRK, dA + dA^T part of the scaled GEMM) for tensor-core sized problems."""
        return self.use_i8 and self.want_tc(N, M)

    def kernel_fwd(self, spec, Fx, Fz, hyp, tc=False, i8=None):
        Fx, Fz, hyp = _f32c(Fx), _f32c(Fz), _f32c(hyp)
        N, M = Fx.shape[0], Fz.shape[0]
        ta, da, tb, db = spec
        dev = Fx.device
        if i8 is None:
            i8 = bool(tc) and self.want_i8(N, M)
        if tc and i8:
            # fp16 hi/lo row planes + the int8 digit planes of the integer tensor-core products, straight from fp32 values
            ldkh, ldkr, nblk = _pad(M, 8), _pad(M, 16), (N + 127) // 128
            Kh = torch.empty((N, ldkh), device=dev, dtype=torch.float16)
            Kl = torch.empty((N, ldkh), device=dev, dtype=torch.float16)
            kscale = torch.empty(8, device=dev, dtype=torch.float32)
            kop = Kop(None, Kh, Kl, None, None, kscale, N, M)
            kop.Kr = torch.empty((4, N, ldkr), device=dev, dtype=torch.int8)
            kop.rscale = torch.empty(N, device=dev, dtype=torch.float32)
            kop.Kc = torch.empty((4, nblk, M, 128), device=dev, dtype=torch.int8)
            kop.cscale = torch.empty(M, device=dev, dtype=torch.float32)
            scratch = torch.empty(N + M, device=dev, dtype=torch.float32)
            _call("svgp_kernel_fwd_i8", _ptr(Fx), Fx.stride(0), N, _ptr(Fz), Fz.stride(0), M, ta, da, tb, db, _ptr(hyp),
                  _ptr(Kh), _ptr(Kl), ldkh, _ptr(kop.Kr), ldkr, _ptr(kop.rscale), _ptr(kop.Kc), _ptr(kop.cscale), _ptr(scratch),
                  _ptr(kscale), _stream())
            self.launches += 2
        elif tc:
            ldkh = _pad(M, 8)
            alloc = torch.zeros if (ldkh != M) else torch.empty
            Kh = alloc((N, ldkh), device=dev, dtype=torch.float16)
            Kl = alloc((N, ldkh), device=dev, dtype=torch.float16)
            # transposed planes, blocked by 64 datapoints: [ceil(N / 64)][M][64] (the kernel zeroes the ragged tail)
            nblk = (N + 63) // 64
            Kth = torch.empty((nblk, M, 64), device=dev, dtype=torch.float16)
            Ktl = torch.empty((nblk, M, 64), device=dev, dtype=torch.float16)
            ldkt = M * 64
            kscale = torch.empty(8, device=dev, dtype=torch.float32)
            kop = Kop(None, Kh, Kl, Kth, Ktl, kscale, N, M)
            _call("svgp_kernel_fwd", _ptr(Fx), Fx.stride(0), N, _ptr(Fz), Fz.stride(0), M, ta, da, tb, db, _ptr(hyp),
                  None, 0, _ptr(Kh), _ptr(Kl), ldkh, _ptr(Kth), _ptr(Ktl), ldkt, _ptr(kscale), _stream())
        else:
            K = torch.empty((N, M), device=dev, dtype=torch.float32)
            kop = Kop(K)
            _call("svgp_kernel_fwd", _ptr(Fx), Fx.stride(0), N, _ptr(Fz), Fz.stride(0), M, ta, da, tb, db, _ptr(hyp),
                  _ptr(K), K.stride(0), None, None, 0, None, None, 0, None, _stream())
        self.launches += 1
        return kop

    def kernel_fwd_f64(self, spec, Fx, Fz, hyp):
        """K(Fx, Fz) evaluated and stored in float64 (fp32 features): K_mm of the M x M stage."""
        Fx, Fz, hyp = _f32c(Fx), _f32c(Fz), _f32c(hyp)
        N, M = Fx.shape[0], Fz.shape[0]
        ta, da, tb, db = spec
        K = torch.empty((N, M), device=Fx.device, dtype=torch.float64)
        _call("svgp_kernel_fwd_f64", _ptr(Fx), Fx.stride(0), N, _ptr(Fz), Fz.stride(0), M, ta, da, tb, db, _ptr(hyp), _ptr(K), M, _stream())
        self.launches += 1
        return K

    def kernel_bwd(self, spec, Fx, Fz, hyp, G, need_x=True, need_z=True):
        Fx, Fz, hyp, G = _f32c(Fx), _f32c(Fz), _f32c(hyp), _f32c(G)
        N, M, d = Fx.shape[0], Fz.shape[0], Fx.shape[1]
        ta, da, tb, db = spec
        dFx = torch.empty((N, d), device=Fx.device, dtype=torch.float32) if need_x else None
        dFz = torch.zeros((M, d), device=Fx.device, dtype=torch.float64) if need_z else None
        dhyp = torch.zeros(hyp.numel(), device=Fx.device, dtype=torch.float64)     # 4 + d for ARD specs
        _call("svgp_kernel_bwd", _ptr(Fx), Fx.stride(0), N, _ptr(Fz), Fz.stride(0), M, ta, da, tb, db, _ptr(hyp),
                  _ptr(G), G.stride(0), _ptr(dFx), _ptr(dFz), _ptr(dhyp), _stream())
        self.launches += int(need_x) + int(need_z)
        return dFx, dFz, dhyp

    def kernel_diag_fwd(self, spec, Fx, Fy, hyp):
        Fx, Fy, hyp = _f32c(Fx), _f32c(Fy), _f32c(hyp)
        ta, da, tb, db = spec
        kd = torch.empty(Fx.shape[0], device=Fx.device, dtype=torch.float32)
        _call("svgp_kernel_diag_fwd", _ptr(Fx), Fx.stride(0), _ptr(Fy), Fy.stride(0), Fx.shape[0], ta, da, tb, db,
                  _ptr(hyp), _ptr(kd), _stream())
        self.launches += 1
        return kd

    def kernel_diag_bwd(self, spec, Fx, Fy, hyp, g):
        Fx, Fy, hyp, g = _f32c(Fx), _f32c(Fy), _f32c(hyp), _f32c(g)
        ta, da, tb, db = spec
        dFx, dFy = torch.empty_like(Fx), torch.empty_like(Fy)
        dhyp = torch.zeros(hyp.numel(), device=Fx.device, dtype=torch.float64)
        _call("svgp_kernel_diag_bwd", _ptr(Fx), Fx.stride(0), _ptr(Fy), Fy.stride(0), Fx.shape[0], ta, da, tb, db,
                  _ptr(hyp), _ptr(g), _ptr(dFx), _ptr(dFy), _ptr(dhyp), _stream())
        self.launches += 1
        return dFx, dFy, dhyp

    def gather_rows(self, table, ids):
        table = _f32c(table)
        assert ids.dtype == torch.int64 and ids.is_contiguous()
        out = torch.empty((ids.shape[0], table.shape[1]), device=table.device, dtype=torch.float32)
        _call("svgp_gather_rows", _ptr(table), table.stride(0), table.shape[0], _ptr(ids), ids.shape[0],
                  table.shape[1], _ptr(out), out.stride(0), _stream())
        self.launches += 1
        return out

    def scatter_add_rows(self, g, ids, rows):
        g = _f32c(g)
        dt = torch.zeros((rows, g.shape[1]), device=g.device, dtype=torch.float64)
        _call("svgp_scatter_add_rows", _ptr(g), g.stride(0), _ptr(ids), ids.shape[0], g.shape[1], rows, _ptr(dt),
                  dt.stride(0), _stream())
        self.launches += 1
        return dt

    # ---- GEMM class ------------------------------------------------------------------------
    def planes(self, S64):
        """(B, M, M) float64 -> scaled fp16 (hi, lo) planes + per-matrix 1/scale (the TC operand format)."""
        S64 = _f64c(S64)
        nb = S64.shape[0]
        hi = torch.empty(S64.shape, device=S64.device, dtype=torch.float16)
        lo = torch.empty_like(hi)
        inv = torch.empty(2 * nb, device=S64.device, dtype=torch.float32)
        _call("svgp_split_f16", _ptr(S64), nb, S64[0].numel(), _ptr(hi), _ptr(lo), _ptr(inv), _stream())
        self.launches += 2
        return Planes(hi, lo, inv)

    def planes_into(self, S64, hi, lo, inv, at):
        """svgp_split_f16 of a (b, M, M) float64 batch into rows [at, at + b) of preallocated plane buffers."""
        S64 = _f64c(S64 if S64.is_contiguous() else S64.contiguous())
        nb = S64.shape[0]
        tmp = torch.empty(2 * nb, device=S64.device, dtype=torch.float32)      # [1/scale | abs-max scratch]
        _call("svgp_split_f16", _ptr(S64), nb, S64[0].numel(), _ptr(hi[at:at + nb]), _ptr(lo[at:at + nb]), _ptr(tmp), _stream())
        inv[at:at + nb] = tmp[:nb]
        self.launches += 2

    def planes_i8(self, X64, nslices=4):
        """(B, R, C) float64 -> int8 digit planes with one scale per row (svgp_split_i8)."""
        X64 = _f64c(X64 if X64.is_contiguous() else X64.contiguous())
        B, R, C = X64.shape
        ldp = _pad(C, 16)
        planes = torch.empty((nslices, B * R, ldp), device=X64.device, dtype=torch.int8)
        scale = torch.empty(B * R, device=X64.device, dtype=torch.float32)
        _call("svgp_split_i8", _ptr(X64), B * R, C, C, nslices, _ptr(planes), ldp, _ptr(scale), _stream())
        self.launches += 1
        return PlanesI8(planes, scale, B, R, C)

    def planes_i8_alloc(self, B, R, C, device, nslices=4):
        ldp = _pad(C, 16)
        return PlanesI8(torch.empty((nslices, B * R, ldp), device=device, dtype=torch.int8),
                        torch.empty(B * R, device=device, dtype=torch.float32), B, R, C)

    def planes_i8_into(self, X64, P, at):
        """svgp_split_i8 of a (b, R, C) float64 batch into matrices [at, at + b) of the preallocated PlanesI8 ``P``."""
        X64 = _f64c(X64 if X64.is_contiguous() else X64.contiguous())
        b, R, C = X64.shape
        assert R == P.R and C == P.C and at + b <= P.B
        S, _, ldp = P.planes.shape
        # the planes of a row range are not contiguous across digit planes: the library takes the base of plane 0 and
        # the plane stride is implied by nrows -- so split plane by plane range through a temporary of the piece
        tmp = torch.empty((S, b * R, ldp), device=X64.device, dtype=torch.int8)
        _call("svgp_split_i8", _ptr(X64), b * R, C, C, S, _ptr(tmp), ldp, _ptr(P.scale[at * R:(at + b) * R]), _stream())
        P.planes[:, at * R:(at + b) * R] = tmp
        self.launches += 2

    def pair_bias_i8(self, planes):
        """(4, R, ld) int8 digit planes -> (2, R) fp32: this operand's share of the expected value of the digit-plane pairs the
        integer products drop (svgp_i8_pair_bias; row 0: ten pairs kept, row 1: eight)."""
        S, R, ld = planes.shape
        assert S == 4 and planes.is_contiguous()
        bias = torch.empty((2, R), device=planes.device, dtype=torch.float32)
        _call("svgp_i8_pair_bias", _ptr(planes), R, ld, _ptr(bias), _stream())
        self.launches += 1
        return bias

    def scaled_gemm_i8(self, kop, W, G, out=None, ndot=0, nfull=None, debias=None):
        """scaled_gemm on the integer tensor-core path; G: PlanesI8 of L stacked (Mc, M) matrices (4 digit planes).
        ``nfull``: the matrices from this index on are multiplied with the three leading digits of both operands only
        (8 instead of 10 digit-plane pairs; default: all matrices at full precision).  ``debias``: add the expected value of
        the dropped pairs to every entry before it is rounded (default: on; the digits have mean -1/2, see svgp_b200.h)."""
        assert kop.i8 and isinstance(G, PlanesI8) and G.planes.shape[0] == 4 and G.C == kop.M
        L, Mc = G.B, G.R
        if W is not None:
            W = _f32c(W)
            assert W.shape == (kop.N, L)
        accumulate = out is not None
        if out is None:
            out = torch.empty((kop.N, Mc), device=kop.device, dtype=torch.float32)
        dots = torch.zeros((kop.N, ndot), device=kop.device, dtype=torch.float32) if ndot else None
        s = kop.struct()
        kb = gb = None
        if (kop.M >= self.i8_debias) if debias is None else debias:
            if getattr(kop, "Kr_bias", None) is None:
                kop.Kr_bias = self.pair_bias_i8(kop.Kr)                  # once per kernel matrix
            kb, gb = kop.Kr_bias, self.pair_bias_i8(G.planes)
        _call("svgp_scaled_gemm_i8", ctypes.byref(s), _ptr(W), W.stride(0) if W is not None else 0, _ptr(G.planes), G.planes.stride(1),
              _ptr(G.scale), L, Mc, _ptr(out), out.stride(0), int(accumulate), _ptr(dots), ndot, ndot,
              L if nfull is None else int(nfull), _ptr(kb), _ptr(gb), _stream())
        self.launches += 1
        return (out, dots) if ndot else out

    def syrk(self, kop, W, impl=IMPL_AUTO, chunk_rows=0):
        W = _f32c(W)
        L = W.shape[1]
        A = torch.zeros((L, kop.M, kop.M), device=W.device, dtype=torch.float64)
        use_tc = kop.tc and impl != IMPL_SIMT
        use_i8 = use_tc and kop.i8 and impl in (IMPL_AUTO, IMPL_TC_I8, IMPL_TC_I8_D3, IMPL_TC_I8_O4)
        # D3: the adjoint SYRK (eight digit-plane pairs); O4: the forward SYRK above M = 2048 (thirteen)
        i8_impl = impl if impl in (IMPL_TC_I8_D3, IMPL_TC_I8_O4) else IMPL_TC_I8
        ws = None
        if use_tc:
            ws = torch.empty(int(_lib.load().svgp_syrk_ws_floats(kop.N, kop.M, L)), device=W.device, dtype=torch.float32)
        s = kop.struct()
        _call("svgp_syrk", ctypes.byref(s), _ptr(W), W.stride(0), L, _ptr(A),
              i8_impl if use_i8 else (IMPL_TC if use_tc else IMPL_SIMT), chunk_rows, _ptr(ws), _stream())
        self.launches += 4 if use_tc else 1
        return A

    def gemm_tn(self, kop, X):
        X = _f32c(X)
        L = X.shape[1]
        V = torch.zeros((L, kop.M), device=X.device, dtype=torch.float64)
        s = kop.struct()
        _call("svgp_gemm_tn", ctypes.byref(s), _ptr(X), X.stride(0), L, _ptr(V), _stream())
        self.launches += 1
        return V

    def gemm_nn(self, kop, Wm, impl=IMPL_AUTO):
        L = Wm.shape[0]
        out = torch.empty((kop.N, L), device=Wm.device, dtype=torch.float32)
        s = kop.struct()
        if kop.i8 and impl in (IMPL_AUTO, IMPL_TC_I8):
            # exact integer products: K_nm w_l cancels heavily at large M (p_m, dy at M = 2048)
            return self.scaled_gemm_i8(kop, None, self.planes_i8(Wm.double().contiguous().unsqueeze(0)))
        if kop.tc and impl != IMPL_SIMT and kop.M >= 128 and kop.N >= self.tc_min_rows:
            pl = self.planes(Wm.double().contiguous().unsqueeze(0))          # (1, L, M) -> one scale for the whole matrix
            _call("svgp_gemm_nn_tc", ctypes.byref(s), _ptr(pl.hi), _ptr(pl.lo), _ptr(pl.inv), L, _ptr(out), out.stride(0), _stream())
            self.launches += 1
            return out
        Wm = _f32c(Wm.float().contiguous())
        _call("svgp_gemm_nn", ctypes.byref(s), _ptr(Wm), Wm.stride(0), L, _ptr(out), out.stride(0), _stream())
        self.launches += 1
        return out

    def _operand(self, S64, use_tc):
        """-> (hi ptr, lo ptr, inv ptr, keep-alive) of a float64 batch in the format the chosen implementation reads."""
        if use_tc:
            pl = S64 if isinstance(S64, Planes) else self.planes(S64)
            return _ptr(pl.hi), _ptr(pl.lo), _ptr(pl.inv), pl
        S64 = _f64c(S64 if S64.is_contiguous() else S64.contiguous())      # SIMT kernels read the float64 matrices directly
        return _ptr(S64), None, None, S64

    def rowquad(self, kop, S64, tri=False, impl=IMPL_AUTO, out=None):
        """q[i, l] = k_i^T S_l k_i (or |T_l k_i|^2 for a triangular factor T_l); ``out``: an (N, L) fp32 view
        with unit column stride to write into (e.g. a column slice of a wider matrix)."""
        L = (S64.hi if isinstance(S64, Planes) else S64).shape[0]
        use_tc = kop.tc and impl != IMPL_SIMT
        hi, lo, inv, keep = self._operand(S64, use_tc)
        if out is None:
            q = torch.empty((kop.N, L), device=kop.device, dtype=torch.float32)
        else:
            q = out
            assert q.is_cuda and q.dtype == torch.float32 and q.shape == (kop.N, L) and q.stride(1) == 1, (q.shape, q.stride())
        s = kop.struct()
        _call("svgp_rowquad", ctypes.byref(s), hi, lo, inv, L, int(bool(tri)), _ptr(q), q.stride(0),
              IMPL_TC if use_tc else IMPL_SIMT, _stream())
        self.launches += 1
        del keep
        return q

    def scaled_gemm(self, kop, W, G64, out=None, ndot=0, impl=IMPL_AUTO):
        """out (+)= sum_l diag(W[:, l]) K G_l; with ndot > 0 also returns dots[i, l] = k_i^T G_l k_i for l < ndot."""
        W = _f32c(W)
        L = W.shape[1]
        use_tc = kop.tc and impl != IMPL_SIMT
        hi, lo, inv, keep = self._operand(G64, use_tc)
        accumulate = out is not None
        if out is None:
            out = torch.empty((kop.N, kop.M), device=W.device, dtype=torch.float32)
        dots = torch.zeros((kop.N, ndot), device=W.device, dtype=torch.float32) if ndot else None
        s = kop.struct()
        _call("svgp_scaled_gemm", ctypes.byref(s), _ptr(W), W.stride(0), hi, lo, inv, L, _ptr(out), out.stride(0),
              int(accumulate), _ptr(dots), ndot, ndot, IMPL_TC if use_tc else IMPL_SIMT, _stream())
        self.launches += 1 + (0 if use_tc or not ndot else 1)
        del keep
        return (out, dots) if ndot else out

    def gemm_f32(self, A, B, out=None):
        A, B = _f32c(A), _f32c(B)
        accumulate = out is not None
        if out is None:
            out = torch.empty((A.shape[0], B.shape[1]), device=A.device, dtype=torch.float32)
        _call("svgp_gemm_f32", A.shape[0], B.shape[1], A.shape[1], _ptr(A), A.stride(0), _ptr(B), B.stride(0),
                  _ptr(out), out.stride(0), int(accumulate), _stream())
        self.launches += 1
        return out

    # ---- K3 --------------------------------------------------------------------------------
    def chol(self, X):
        """Lower Cholesky factors of a (B, M, M) float64 batch; returns (Lf, status int32[B])."""
        X = _f64c(X)
        B, M, _ = X.shape
        Lf = X.clone()
        status = torch.zeros(B, device=X.device, dtype=torch.int32)
        ws = torch.empty(B * 32 * 32, device=X.device, dtype=torch.float64)
        _call("svgp_chol_f64", _ptr(Lf), M, M, M * M, B, _ptr(status), _ptr(ws), _stream())
        self.launches += 3 * ((M + 31) // 32)
        return Lf, status

    def trinv(self, Lf):
        Lf = _f64c(Lf)
        B, M, _ = Lf.shape
        nblk = (M + 31) // 32
        Linv = torch.empty_like(Lf)
        ws = torch.empty(B * nblk * 32 * 32 + B * 32 * M, device=Lf.device, dtype=torch.float64)
        _call("svgp_trinv_f64", _ptr(Lf), _ptr(Linv), M, M, M * M, B, _ptr(ws), _stream())
        self.launches += 2 * nblk + 2
        return Linv

    def ltl(self, T):
        """T^T T for a batch of lower-triangular float64 matrices (X^-1 from the inverse Cholesky factor)."""
        T = _f64c(T)
        B, M, _ = T.shape
        S = torch.empty_like(T)
        _call("svgp_ltl_f64", _ptr(T), _ptr(S), M, M, M * M, B, _stream())
        self.launches += 2
        return S

    def bmm64(self, A, B, transA=False, transB=False):
        """C[b] = op(A[b]) op(B[b]); a leading batch of 1 broadcasts against the other operand."""
        A, B = _f64c(A), _f64c(B)
        nb = max(A.shape[0], B.shape[0])
        Mr = A.shape[2] if transA else A.shape[1]
        Kd = A.shape[1] if transA else A.shape[2]
        Nc = B.shape[1] if transB else B.shape[2]
        assert Kd == (B.shape[2] if transB else B.shape[1]), (A.shape, B.shape, transA, transB)
        C = torch.empty((nb, Mr, Nc), device=A.device, dtype=torch.float64)
        sA = 0 if (A.shape[0] == 1 and nb > 1) else A.shape[1] * A.shape[2]
        sB = 0 if (B.shape[0] == 1 and nb > 1) else B.shape[1] * B.shape[2]
        _call("svgp_gemm_f64", int(transA), int(transB), Mr, Nc, Kd, 1.0, _ptr(A), A.shape[2], sA, _ptr(B),
                  B.shape[2], sB, 0.0, _ptr(C), Nc, Mr * Nc, nb, _stream())
        self.launches += 1
        return C

    # ---- K4 row terms ----------------------------------------------------------------------
    def rowstats(self, y, noise, kappa):
        y, noise, kappa = _f32c(y), _f32c(noise), _f32c(kappa)
        N, L = y.shape
        p, py = torch.empty_like(y), torch.empty_like(y)
        sums = torch.zeros((3, L), device=y.device, dtype=torch.float64)
        _call("svgp_rowstats_fwd", _ptr(y), _ptr(noise), _ptr(kappa), N, L, _ptr(p), _ptr(py), _ptr(sums), _stream())
        self.launches += 1
        return p, py, sums

    def predictive(self, kappa, h, q1, p, clip=None):
        kappa, h, q1 = _f32c(kappa), _f32c(h), _f32c(q1)
        N, L = q1.shape
        pv = q1.clone()
        clipsum = torch.zeros(L, device=q1.device, dtype=torch.float64)
        mask = torch.zeros((N, L), device=q1.device, dtype=torch.uint8) if clip else None
        lo, hi = clip if clip else (0.0, 0.0)
        _call("svgp_predictive_fwd", _ptr(kappa), _ptr(h), _ptr(pv), _ptr(_f32c(p)) if clip else None, N, L,
                  int(bool(clip)), lo, hi, _ptr(clipsum), _ptr(mask), _stream())
        self.launches += 1
        return pv, clipsum, mask


    def rowterms_bwd_pre(self, g_pv, g_pm, p, y, clip=None):
        """-> G_q1 (N, L), Wst = [p | 2 G_q1], PYst = [p y | g_pm] (N, 2L), G_p_clip (N, L) or None, G_kappa (N,).
        clip = (mask uint8, pv, kappa, h, q1raw, gce (L,) fp32) on the SPRITES clip branch."""
        g_pm, p, y = _f32c(g_pm), _f32c(p), _f32c(y)
        N, L = y.shape
        dev = y.device
        G_q1 = torch.empty((N, L), device=dev, dtype=torch.float32)
        Wst = torch.empty((N, 2 * L), device=dev, dtype=torch.float32)
        PYst = torch.empty((N, 2 * L), device=dev, dtype=torch.float32)
        G_kappa = torch.empty(N, device=dev, dtype=torch.float32)
        G_p_clip = torch.empty((N, L), device=dev, dtype=torch.float32) if clip else None
        mask, pv, kappa, h, q1raw, gce = clip if clip else (None,) * 6
        _call("svgp_rowterms_bwd_pre", _ptr(None if g_pv is None else _f32c(g_pv)), _ptr(g_pm), _ptr(p), _ptr(y), _ptr(mask),
              _ptr(pv), _ptr(kappa), _ptr(h), _ptr(q1raw), _ptr(gce), N, L, _ptr(G_q1), _ptr(Wst), _ptr(PYst), _ptr(G_p_clip),
              _ptr(G_kappa), _stream())
        self.launches += 1
        return G_q1, Wst, PYst, G_p_clip, G_kappa

    def rowterms_bwd_post(self, y, noise, p, kappa, kGk, G_py, gsums, G_p_clip, G_kappa):
        """-> G_y, G_noise (N, L); G_kappa (N,) is updated in place."""
        N, L = y.shape
        G_y, G_noise = torch.empty_like(y), torch.empty_like(y)
        _call("svgp_rowterms_bwd_post", _ptr(_f32c(y)), _ptr(_f32c(noise)), _ptr(_f32c(p)), _ptr(_f32c(kappa)), _ptr(_f32c(kGk)),
              _ptr(_f32c(G_py)), _ptr(_f64c(gsums)), _ptr(G_p_clip), N, L, _ptr(G_y), _ptr(G_noise), _ptr(G_kappa), _stream())
        self.launches += 1
        return G_y, G_noise, G_kappa


_BACKEND = None


def get_backend():
    global _BACKEND
    if _BACKEND is None:
        _BACKEND = CudaBackend()          # raises if the library / device is missing: no fallback
    return _BACKEND


def set_backend_for_tests(backend):
    """Test hook (tests/ only): run the host logic against a float64 CPU oracle backend."""
    global _BACKEND
    old = _BACKEND
    _BACKEND = backend
    return old
