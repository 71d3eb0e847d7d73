"""tcgen05 engine (3 x FP16 split) against float64 on the device and against the SIMT kernels."""
import pytest
import torch

from conftest import rel_err
from svgp_vae_b200.backend import IMPL_SIMT, Kop

pytestmark = pytest.mark.gpu
SPEC = (1, 4, 1, 4)
# LINEAR x COSINE on [16 | 16]: K has negative entries (kscale[6] = 0: no one-signed truncation-bias correction)
SIGNED = (3, 16, 4, 16)


def _setup(be, N, M, L, seed=0, spec=SPEC, i8=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    Fx = torch.randn(N, spec[1] + spec[3], generator=g, device="cuda")
    Fz = torch.randn(M, spec[1] + spec[3], generator=g, device="cuda")
    hyp = torch.ones(4, device="cuda")
    kop = be.kernel_fwd(spec, Fx, Fz, hyp, tc=True, i8=i8)
    assert float(kop.kscale[6]) == (0.0 if spec == SIGNED else 1.0)
    K64 = kop.value().double()
    W = torch.randn(N, L, generator=g, device="cuda")
    return kop, K64, W, g


@pytest.mark.parametrize("shape", [(4096, 256, 3), (3000, 200, 2), (8192, 384, 2), (2500, 1024, 1)])
def test_tc_syrk(cuda_backend, shape, spec=SPEC):
    be = cuda_backend
    N, M, L = shape
    kop, K64, W, g = _setup(be, N, M, L, spec=spec)
    ref = torch.einsum('il,ia,ib->lab', W.double(), K64, K64)
    # the tensor core accumulates with truncation: the bias grows ~2.7e-8 per MMA of a chain (measured,
    # profiles/r01_accuracy.md), so short chains (chunk_rows=128 -> 24 MMAs) reach fp32-level accuracy and
    # the default chain (2048 rows -> 384 MMAs) stays ~1e-5
    assert rel_err(be.syrk(kop, W, chunk_rows=128), ref) < 3e-6
    A = be.syrk(kop, W)
    assert rel_err(A, ref) < 3e-5
    assert rel_err(A, A.transpose(1, 2)) == 0.0
    A2 = be.syrk(Kop(kop.value().contiguous()), W, impl=IMPL_SIMT)
    assert rel_err(A2, ref) < 1e-6 and rel_err(A, A2) < 3e-5
    # weights spanning six decades (p = 1/noise with the reference's clip [1e-3, 10]): per-channel power-of-two scaling
    Wp = torch.exp(torch.empty(N, L, device="cuda").uniform_(-4.6, 9.2, generator=g))
    refp = torch.einsum('il,ia,ib->lab', Wp.double(), K64, K64)
    assert rel_err(be.syrk(kop, Wp), refp) < 3e-5


@pytest.mark.parametrize("shape", [(4096, 256, 3), (2500, 1024, 1)])
def test_tc_syrk_signed(cuda_backend, shape):
    test_tc_syrk(cuda_backend, shape, SIGNED)


@pytest.mark.parametrize("shape", [(9000, 256, 1), (20000, 384, 3), (20000, 384, 4), (70000, 1024, 2)])
def test_tc_syrk_superchunks(cuda_backend, shape, monkeypatch):
    """Datapoints are walked in L2-sized super-chunks; different CTAs add different super-chunks of one tile into the
    float64 accumulator under a lock.  Force many small super-chunks (L = 1: same-tile items run concurrently)."""
    be = cuda_backend
    N, M, L = shape
    kop, K64, W, g = _setup(be, N, M, L, seed=5)
    ref = torch.einsum('il,ia,ib->lab', W.double(), K64, K64)
    monkeypatch.setenv("SVGP_SYRK_SC", "512")
    for _ in range(3):
        A = be.syrk(kop, W, chunk_rows=256)
        assert rel_err(A, ref) < 3e-6
    monkeypatch.setenv("SVGP_SYRK_SC", "4096")
    assert rel_err(be.syrk(kop, W), ref) < 3e-5


@pytest.mark.parametrize("shape", [(4096, 256, 3), (3000, 200, 2), (2304, 1024, 2)])
def test_tc_rowquad_scaled(cuda_backend, shape, spec=SPEC, i8=False):
    be = cuda_backend
    N, M, L = shape
    kop, K64, W, g = _setup(be, N, M, L, seed=1, spec=spec, i8=i8)
    S = torch.randn(L, M, M, generator=g, device="cuda", dtype=torch.float64)
    S = (S + S.transpose(1, 2)).contiguous()
    S[0] *= 1e4                                      # per-matrix scaling of the fp16 planes
    Lt = torch.tril(torch.randn(L, M, M, generator=g, device="cuda", dtype=torch.float64)).contiguous()
    Lt[-1] *= 1e-3
    ref = torch.einsum('ia,lab,ib->il', K64, S, K64)
    assert rel_err(be.rowquad(kop, S), ref) < 3e-5
    T = torch.einsum('ia,lca->ilc', K64, Lt)
    for l in range(L):
        assert rel_err(be.rowquad(kop, Lt, tri=True)[:, l], (T * T).sum(-1)[:, l]) < 3e-5
    refo = torch.einsum('il,ia,lac->ic', W.double(), K64, S)
    out, dots = be.scaled_gemm(kop, W, S, ndot=L)
    assert rel_err(out, refo) < 3e-5
    for l in range(L):
        assert rel_err(dots[:, l], ref[:, l]) < 3e-5
    be.scaled_gemm(kop, W, S, out=out)
    assert rel_err(out, 2 * refo) < 3e-5
    out1, dots1 = be.scaled_gemm(kop, W, S, ndot=1)
    assert rel_err(out1, refo) < 3e-5 and rel_err(dots1[:, 0], ref[:, 0]) < 3e-5


@pytest.mark.parametrize("shape", [(4096, 256, 3), (2304, 1024, 2)])
def test_tc_rowquad_scaled_signed(cuda_backend, shape):
    """The row quads and the scaled GEMM on the fp16 row planes of the integer builder (the step's default format)."""
    test_tc_rowquad_scaled(cuda_backend, shape, SIGNED, i8=True)


@pytest.mark.parametrize("shape", [(4096, 256, 3), (3000, 200, 64), (2304, 1024, 70), (2500, 384, 300)])
def test_tc_gemm_nn(cuda_backend, shape):
    """out = K Wm^T on the tensor cores (SCALED mode with L output columns) against float64 and the SIMT kernel."""
    be = cuda_backend
    N, M, L = shape
    kop, K64, _, g = _setup(be, N, M, 1, seed=7)
    Wm = torch.randn(L, M, generator=g, device="cuda") * torch.exp(torch.randn(L, 1, generator=g, device="cuda") * 3)
    ref = K64 @ Wm.double().t()
    out = be.gemm_nn(kop, Wm)
    assert out.shape == (N, L) and rel_err(out, ref) < 3e-5
    assert rel_err(be.gemm_nn(Kop(kop.value().contiguous()), Wm, impl=IMPL_SIMT), ref) < 1e-5


def test_tc_planes_roundtrip(cuda_backend):
    be = cuda_backend
    g = torch.Generator(device="cuda").manual_seed(3)
    X = torch.randn(3, 64, 64, generator=g, device="cuda", dtype=torch.float64)
    X[1] *= 1e-6
    X[2] = 0
    pl = be.planes(X)
    back = (pl.hi.double() + pl.lo.double()) * pl.inv[:3, None, None].double()
    assert rel_err(back[0], X[0]) < 1e-6 and rel_err(back[1], X[1]) < 1e-6 and float(back[2].abs().max()) == 0.0
    assert float(pl.hi.abs().max()) <= 2 ** 14
