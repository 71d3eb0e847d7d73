// K1: kernel-matrix builder, its adjoint, the element-wise (diag) form and the embedding
// gather / scatter.  Replaces mnistSVGP.kernel_matrix (SVGPVAE_model.py:427-476),
// spritesSVGP.kernel_matrix (:550-600), the ball's kernel.matrix calls (:81-86, :152-157)
// and the tfp.math.psd_kernels arithmetic under them (formulas: oracle/tfp_kernels.py).
//
// k(x, z) = kA(xA, zA) * kB(xB, zB), each factor one of NONE / SE / EXPSIN / LINEAR / COSINE / MATERN12 / MATERN32 /
// MATERN52.
// The builder is HBM-bound: every output element is written once (coalesced, through a
// padded shared-memory tile so that both K (N x M) and its transpose Kt (M x N) leave the SM
// as full row segments), optionally as a scaled fp16 hi/lo pair for the tcgen05 consumers.
#include <cuda_fp16.h>
#include <stdarg.h>

#include "common.cuh"

namespace svgp {

// ------------------------------------------------------------------------------------------
// error plumbing (shared by every translation unit)
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return SVGP_ERR_CUDA;
  }
  return SVGP_OK;
}
const char* last_error() { return g_err; }

// ------------------------------------------------------------------------------------------
// factor arithmetic
// ------------------------------------------------------------------------------------------
// ta / tb are the base type codes: the SVGP_K_ARD flag is stripped at the ABI boundary into ard_a / ard_b
struct Spec {
  int ta, da, tb, db;
  bool ard_a, ard_b;
};

struct Hyp {
  float amp_a, len_a, amp_b, len_b;
};

__device__ __forceinline__ Hyp load_hyp(const float* hyp) {
  Hyp h;
  h.amp_a = hyp[0]; h.len_a = hyp[1]; h.amp_b = hyp[2]; h.len_b = hyp[3];
  return h;
}

// Matern factors: k = a^2 p(u) e^-u with u = c r / l, r = |x - z| over the block, c = 1, sqrt 3, sqrt 5 and
// p(u) = 1, 1 + u, 1 + u + u^2 / 3 for nu = 1/2, 3/2, 5/2
__host__ __device__ __forceinline__ bool is_matern(int type) {
  return type == SVGP_K_MATERN12 || type == SVGP_K_MATERN32 || type == SVGP_K_MATERN52;
}
__device__ __forceinline__ float matern_c(int type) {
  return type == SVGP_K_MATERN12 ? 1.0f : (type == SVGP_K_MATERN32 ? 1.7320508075688772f : 2.2360679774997897f);
}
__device__ __forceinline__ float matern_poly(int type, float u) {
  if (type == SVGP_K_MATERN12) return 1.0f;
  if (type == SVGP_K_MATERN32) return 1.0f + u;
  return fmaf(u, u * (1.0f / 3.0f), 1.0f + u);
}

// value of one factor.  nx / nz are the Euclidean norms of the feature blocks (COSINE only).
// ARD: the SE and Matern distances take every difference times il[f], the inverse length scale of feature f (1 on the
// features of an isotropic block, whose len is its own; len = 1 for an ARD block)
template <bool ARD = false>
__device__ __forceinline__ float factor_value(int type, const float* x, const float* z, int d, float amp,
                                              float len, float nx, float nz, const float* il = nullptr) {
  if (type == SVGP_K_NONE) return 1.0f;
  if (type == SVGP_K_SE) {
    float r2 = 0.f;
    for (int f = 0; f < d; ++f) { float t = x[f] - z[f]; if (ARD) t *= il[f]; r2 = fmaf(t, t, r2); }
    return amp * amp * expf(-0.5f * r2 / (len * len));
  }
  if (type == SVGP_K_EXPSIN) {
    float u = 0.f;
    for (int f = 0; f < d; ++f) { float s = sinf(0.5f * fabsf(x[f] - z[f])); u = fmaf(s, s, u); }
    return amp * amp * expf(-2.0f * u / (len * len));
  }
  if (is_matern(type)) {
    float r2 = 0.f;
    for (int f = 0; f < d; ++f) { float t = x[f] - z[f]; if (ARD) t *= il[f]; r2 = fmaf(t, t, r2); }
    const float u = matern_c(type) * sqrtf(r2) / len;
    return amp * amp * matern_poly(type, u) * expf(-u);
  }
  float dot = 0.f;
  for (int f = 0; f < d; ++f) dot = fmaf(x[f], z[f], dot);
  if (type == SVGP_K_COSINE) dot = dot / (nx * nz);
  return dot;
}

// the same in float64 arithmetic on the fp32 features (the integer tensor-core operands and the M x M stage's K_mm:
// an fp32 evaluation carries ~|exponent| 2^-24 ~ 5e-7 of relative error per entry, which the ill-conditioned M x M
// stage turns into 1e-4 of the inducing-point gradient at M = 2048 -- tools/numerics/sim_parity.py, SIM_KNOISE)
// (ARD: the exact float64 difference times the float64 inverse length scale -- no rounding of x_f / l_f to fp32)
template <bool ARD = false>
__device__ __forceinline__ double factor_value_f64(int type, const float* x, const float* z, int d, double amp,
                                                   double len, double nx, double nz, const double* il = nullptr) {
  if (type == SVGP_K_NONE) return 1.0;
  if (type == SVGP_K_SE) {
    double r2 = 0.0;
    for (int f = 0; f < d; ++f) { double t = (double)x[f] - (double)z[f]; if (ARD) t *= il[f]; r2 = fma(t, t, r2); }
    return amp * amp * exp(-0.5 * r2 / (len * len));
  }
  if (type == SVGP_K_EXPSIN) {
    double u = 0.0;
    for (int f = 0; f < d; ++f) { const double s = sin(0.5 * fabs((double)x[f] - (double)z[f])); u = fma(s, s, u); }
    return amp * amp * exp(-2.0 * u / (len * len));
  }
  if (is_matern(type)) {
    double r2 = 0.0;
    for (int f = 0; f < d; ++f) { double t = (double)x[f] - (double)z[f]; if (ARD) t *= il[f]; r2 = fma(t, t, r2); }
    const double c = type == SVGP_K_MATERN12 ? 1.0 : (type == SVGP_K_MATERN32 ? 1.7320508075688772 : 2.23606797749979);
    const double u = c * sqrt(r2) / len;
    const double p = type == SVGP_K_MATERN12 ? 1.0 : (type == SVGP_K_MATERN32 ? 1.0 + u : fma(u, u * (1.0 / 3.0), 1.0 + u));
    return amp * amp * p * exp(-u);
  }
  double dot = 0.0;
  for (int f = 0; f < d; ++f) dot = fma((double)x[f], (double)z[f], dot);
  if (type == SVGP_K_COSINE) dot = dot / (nx * nz);
  return dot;
}
__device__ __forceinline__ double block_norm_f64(const float* v, int d) {
  double s = 0.0;
  for (int f = 0; f < d; ++f) s = fma((double)v[f], (double)v[f], s);
  return sqrt(s);
}

// adjoint coefficients of one factor for one (row, col) pair, given gk = g * (other factor):
//   d/dz_f = c1 * x_f + c2z * z_f (+ e for EXPSIN on its single feature, sign + for z, - for x)
//   d/dx_f = c1 * z_f + c2x * x_f
//   d/d amp, d/d len returned through damp / dlen
// ARD: the coefficients are those of the scaled coordinates x_f il_f, z_f il_f (len = 1 for an ARD block): on the
// unscaled features d/dz_f = il_f^2 (c1 x_f + c2z z_f), d/dl_f = il_f^3 c1 (x_f - z_f)^2, and dlen means nothing
struct FactorAdj {
  float c1, c2z, c2x, e, damp, dlen;
};
template <bool ARD = false>
__device__ __forceinline__ FactorAdj factor_adjoint(int type, const float* x, const float* z, int d, float amp,
                                                    float len, float nx, float nz, float kval, float gk,
                                                    const float* il = nullptr) {
  FactorAdj a = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (type == SVGP_K_SE) {
    float r2 = 0.f;
    for (int f = 0; f < d; ++f) { float t = x[f] - z[f]; if (ARD) t *= il[f]; r2 = fmaf(t, t, r2); }
    float il2 = 1.0f / (len * len);
    a.c1 = gk * kval * il2;      // dk/dz_f = k (x_f - z_f)/l^2
    a.c2z = -a.c1;
    a.c2x = -a.c1;               // dk/dx_f = k (z_f - x_f)/l^2
    a.damp = gk * 2.0f * kval / amp;
    a.dlen = gk * kval * r2 * il2 / len;
  } else if (type == SVGP_K_EXPSIN) {
    float dd = x[0] - z[0];
    float s = sinf(0.5f * dd);
    float il2 = 1.0f / (len * len);
    a.e = gk * kval * sinf(dd) * il2;          // dk/dz = k sin(x - z)/l^2 ; dk/dx = -that
    a.damp = gk * 2.0f * kval / amp;
    a.dlen = gk * kval * 4.0f * s * s * il2 / len;
  } else if (type == SVGP_K_LINEAR) {
    a.c1 = gk;
  } else if (type == SVGP_K_COSINE) {
    a.c1 = gk / (nx * nz);
    a.c2z = -gk * kval / (nz * nz);
    a.c2x = -gk * kval / (nx * nx);
  } else if (is_matern(type)) {
    // dk/dz_f = C (x_f - z_f) with C = -(dk/du) c / (l r); written with e = a^2 e^-u = kval / p(u), C stays finite at r = 0
    // for nu = 3/2, 5/2 and no division by r appears.  nu = 1/2 has C = k / (l r): 0 at r = 0 (the symmetric subgradient,
    // which gives the exact total derivative of k(z, z) = a^2 when both sides are summed, as the K_mm adjoint does)
    float r2 = 0.f;
    for (int f = 0; f < d; ++f) { float t = x[f] - z[f]; if (ARD) t *= il[f]; r2 = fmaf(t, t, r2); }
    const float r = sqrtf(r2), u = matern_c(type) * r / len;
    const float il2 = 1.0f / (len * len);
    float C, dl;
    if (type == SVGP_K_MATERN12) {
      C = r > 0.f ? kval / (len * r) : 0.f;
      dl = kval * u / len;                                    // dk/dl = k u / l
    } else if (type == SVGP_K_MATERN32) {
      const float e = kval / (1.0f + u);
      C = 3.0f * e * il2;
      dl = e * u * u / len;                                   // dk/dl = a^2 u^2 e^-u / l
    } else {
      const float p1 = 1.0f + u, e = kval / fmaf(u, u * (1.0f / 3.0f), p1);
      C = (5.0f / 3.0f) * p1 * e * il2;
      dl = e * (u * u * (1.0f / 3.0f)) * p1 / len;            // dk/dl = a^2 e^-u (u^2 / 3)(1 + u) / l
    }
    a.c1 = gk * C;
    a.c2z = -a.c1;
    a.c2x = -a.c1;
    a.damp = gk * 2.0f * kval / amp;
    a.dlen = gk * dl;
  }
  return a;
}

constexpr int TILE = 64;        // rows and columns per shared tile
constexpr int THREADS = 256;
constexpr int MAXD = 32;        // max total feature count

__device__ __forceinline__ float block_norm(const float* v, int d) {
  float s = 0.f;
  for (int f = 0; f < d; ++f) s = fmaf(v[f], v[f], s);
  return sqrtf(s);
}

// load `rows` feature rows (d floats, leading dim ld) starting at row r0 into sm[TILE][dp],
// plus the two block norms; rows beyond `total` are zero-filled
__device__ __forceinline__ void load_features(const float* F, int64_t ld, int64_t r0, int64_t total, int d, int dp,
                                              Spec sp, float* sm, float* na, float* nb) {
  for (int idx = threadIdx.x; idx < TILE * d; idx += THREADS) {
    int r = idx / d, f = idx - r * d;
    int64_t gr = r0 + r;
    sm[r * dp + f] = (gr < total) ? F[gr * ld + f] : 0.f;
  }
  __syncthreads();
  if (threadIdx.x < TILE) {
    int r = threadIdx.x;
    bool valid = (r0 + r) < total;    // padding rows get norm 1 so that 0/0 never appears
    na[r] = (valid && sp.ta == SVGP_K_COSINE) ? block_norm(sm + r * dp, sp.da) : 1.f;
    nb[r] = (valid && sp.tb == SVGP_K_COSINE) ? block_norm(sm + r * dp + sp.da, sp.db) : 1.f;
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------
// ARD (SVGP_K_ARD): one length scale l_f per feature column of a block, at hyp[4 + f].  The ARD instantiations of the
// generic kernels keep the inverse length scales in ARD_SMEM bytes behind their own shared-memory layout (float il[MAXD]
// for the fp32 passes, double il[MAXD] for the float64 evaluations) and evaluate an ARD factor with len = 1; the
// features of an isotropic block get il = 1 (exact), so its factor keeps its own len.  Every kernel without ARD is
// the same code as without the flag.
// ------------------------------------------------------------------------------------------
constexpr size_t ARD_SMEM = MAXD * (sizeof(float) + sizeof(double));
__device__ __forceinline__ bool ard_feature(Spec sp, int f) { return f < sp.da ? sp.ard_a : sp.ard_b; }
// written by the first d threads: callers synchronise before the first read (load_features does)
__device__ __forceinline__ void load_ard(const float* hyp, Spec sp, float* ilf, double* ild) {
  for (int f = threadIdx.x; f < sp.da + sp.db; f += blockDim.x) {
    const double il = ard_feature(sp, f) ? 1.0 / (double)hyp[4 + f] : 1.0;
    if (ilf) ilf[f] = (float)il;
    if (ild) ild[f] = il;
  }
}
__device__ __forceinline__ Hyp ard_hyp(Hyp h, Spec sp) {
  if (sp.ard_a) h.len_a = 1.f;
  if (sp.ard_b) h.len_b = 1.f;
  return h;
}
// length scale of feature f (SE44 kernels: the eight of them live in registers)
__device__ __forceinline__ float ard_len(const float* hyp, Spec sp, Hyp h, int f) {
  return ard_feature(sp, f) ? hyp[4 + f] : (f < sp.da ? h.len_a : h.len_b);
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
// Power-of-two scale of the fp16 planes: the kernel's upper bound (amplitude^2 for the stationary factors,
// max|x| max|z| for LINEAR, 1 for COSINE) is brought just below 2^14, so that value * scale = hi + lo keeps
// 22 significand bits for every entry larger than 2^-17 of the bound and never overflows fp16.
__device__ __forceinline__ float factor_bound(int type, float amp, float nx, float nz) {
  if (type == SVGP_K_LINEAR) return nx * nz;
  if (type == SVGP_K_NONE || type == SVGP_K_COSINE) return 1.0f;
  return amp * amp;                    // SE, EXPSIN and the Matern factors
}
__device__ __forceinline__ float plane_scale(Spec sp, Hyp h, const float* ks) {
  float b = factor_bound(sp.ta, h.amp_a, ks[2], ks[4]) * factor_bound(sp.tb, h.amp_b, ks[3], ks[5]);
  if (!(b > 0.f) || !isfinite(b)) return 1.0f;
  int e;
  frexpf(b, &e);                       // b = m 2^e, m in [0.5, 1)
  e = 14 - e;
  if (e > 100) e = 100;
  if (e < -100) e = -100;
  return ldexpf(1.0f, e);
}

// every entry of K is >= 0 (stationary factors only): recorded in kscale[6] for the SYRK's truncation-bias correction
__device__ __forceinline__ bool kernel_nonneg(Spec sp) {
  auto ok = [](int t) { return t != SVGP_K_LINEAR && t != SVGP_K_COSINE; };   // (check_spec admits nothing else)
  return ok(sp.ta) && ok(sp.tb);
}

// max Euclidean norms of the two feature blocks over the rows of F -> ks[slot], ks[slot + 1] (float bits, >= 0)
__global__ void feature_norm_kernel(const float* __restrict__ F, int64_t ld, int64_t rows, Spec sp, float* ks, int slot) {
  float ma = 0.f, mb = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < rows; i += (int64_t)gridDim.x * blockDim.x) {
    float sa = 0.f, sb = 0.f;
    for (int f = 0; f < sp.da; ++f) { float v = F[i * ld + f]; sa = fmaf(v, v, sa); }
    for (int f = 0; f < sp.db; ++f) { float v = F[i * ld + sp.da + f]; sb = fmaf(v, v, sb); }
    ma = fmaxf(ma, sqrtf(sa)); mb = fmaxf(mb, sqrtf(sb));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ma = fmaxf(ma, __shfl_xor_sync(0xffffffffu, ma, o));
    mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(reinterpret_cast<int*>(ks + slot), __float_as_int(ma));
    atomicMax(reinterpret_cast<int*>(ks + slot + 1), __float_as_int(mb));
  }
}

template <bool ARD = false>
__global__ void __launch_bounds__(THREADS) kernel_fwd_kernel(
    const float* __restrict__ Fx, int64_t ldx, int64_t N, const float* __restrict__ Fz, int64_t ldz, int64_t M,
    Spec sp, const float* __restrict__ hyp, float* __restrict__ K, int64_t ldk, __half* __restrict__ Kh,
    __half* __restrict__ Kl, int64_t ldkh, __half* __restrict__ Kth, __half* __restrict__ Ktl, int64_t ldkt,
    float* __restrict__ kscale) {
  extern __shared__ float smem[];
  const int d = sp.da + sp.db, dp = d | 1;
  float* xs = smem;                    // [TILE][dp]
  float* zs = xs + TILE * dp;          // [TILE][dp]
  float* tile = zs + TILE * dp;        // [TILE][TILE+1]
  float* nxa = tile + TILE * (TILE + 1);
  float* nxb = nxa + TILE;
  float* nza = nxb + TILE;
  float* nzb = nza + TILE;
  float* il = nzb + TILE;              // ARD: [MAXD]
  const Hyp h = ARD ? ard_hyp(load_hyp(hyp), sp) : load_hyp(hyp);
  if (ARD) load_ard(hyp, sp, il, nullptr);
  const int64_t col0 = (int64_t)blockIdx.x * TILE;
  const int64_t ntiles_r = (N + TILE - 1) / TILE;
  float scale = 1.0f;
  if (Kh || Kth) {
    scale = plane_scale(sp, h, kscale);
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
      kscale[0] = scale; kscale[1] = 1.0f / scale; kscale[6] = kernel_nonneg(sp) ? 1.0f : 0.0f;
    }
  }

  load_features(Fz, ldz, col0, M, d, dp, sp, zs, nza, nzb);
  const int c = threadIdx.x % TILE, rg = threadIdx.x / TILE;   // 4 row groups
  for (int64_t rt = blockIdx.y; rt < ntiles_r; rt += gridDim.y) {
    const int64_t row0 = rt * TILE;
    load_features(Fx, ldx, row0, N, d, dp, sp, xs, nxa, nxb);
#pragma unroll 4
    for (int j = 0; j < TILE / 4; ++j) {
      int r = rg + 4 * j;
      float ka = factor_value<ARD>(sp.ta, xs + r * dp, zs + c * dp, sp.da, h.amp_a, h.len_a, nxa[r], nza[c], il);
      float kb = factor_value<ARD>(sp.tb, xs + r * dp + sp.da, zs + c * dp + sp.da, sp.db, h.amp_b, h.len_b, nxb[r], nzb[c],
                                   il + sp.da);
      tile[r * (TILE + 1) + c] = ka * kb;
    }
    __syncthreads();
    if (K || Kh) {
#pragma unroll 4
      for (int j = 0; j < TILE / 4; ++j) {
        int r = rg + 4 * j;
        int64_t gr = row0 + r, gc = col0 + c;
        if (gr < N && gc < M) {
          float v = tile[r * (TILE + 1) + c];
          if (K) K[gr * ldk + gc] = v;
          if (Kh) {
            float vs = v * scale;
            __half hi = __float2half_rn(vs);
            Kh[gr * ldkh + gc] = hi;
            Kl[gr * ldkh + gc] = __float2half_rn(vs - __half2float(hi));
          }
        }
      }
    }
    if (Kth) {
      // transposed, datapoint-blocked write  Kt[n / 64][m][n % 64]  (block stride ldkt): this 64 x 64 tile is one
      // contiguous 8 KB run, and the SYRK's TMA boxes (rows x 64 datapoints) are contiguous too -- a plain M x N
      // transpose puts every row of a box on its own 2 MB page.  Datapoints past N in the last block are zeroed.
      static_assert(TILE == 64, "the blocked transpose is laid out in 64-datapoint blocks");
      const int r = threadIdx.x % TILE, cg = threadIdx.x / TILE;
#pragma unroll 4
      for (int j = 0; j < TILE / 4; ++j) {
        int cc = cg + 4 * j;
        int64_t gr = row0 + r, gc = col0 + cc;
        if (gc < M) {
          float vs = gr < N ? tile[r * (TILE + 1) + cc] * scale : 0.f;
          __half hi = __float2half_rn(vs);
          const int64_t o = rt * ldkt + gc * TILE + r;
          Kth[o] = hi;
          Ktl[o] = __float2half_rn(vs - __half2float(hi));
        }
      }
    }
    __syncthreads();
  }
}

// Planes-only builder (the tcgen05 consumers' operand format: scaled fp16 hi/lo of K and of its datapoint-blocked
// transpose).  HBM-write bound: 8 bytes leave the SM per kernel entry.  The 64 x 64 tile is kept in shared memory as
// packed {hi, lo} words (pitch 65: conflict-free for the column-per-lane writes and for both read-outs below) and
// every thread leaves with 16-byte stores -- 8 consecutive columns of a row of Kh / Kl, 8 consecutive datapoints of
// a row of Kth / Ktl.  SE44 = product of two 4-feature SE factors (the SWEEP kernel): inducing features live in
// registers, datapoint features are broadcast float4 loads, both factors share one ex2.  ARD specs take the generic form.
template <bool SE44, bool ARD = false>
__global__ void __launch_bounds__(THREADS) kernel_fwd_planes_kernel(
    const float* __restrict__ Fx, int64_t ldx, int64_t N, const float* __restrict__ Fz, int64_t ldz, int64_t M,
    Spec sp, const float* __restrict__ hyp, __half* __restrict__ Kh, __half* __restrict__ Kl, int64_t ldkh,
    __half* __restrict__ Kth, __half* __restrict__ Ktl, int64_t ldkt, float* __restrict__ kscale) {
  extern __shared__ float smem[];
  const int d = sp.da + sp.db;
  const int dpx = SE44 ? 8 : (d | 1), dpz = d | 1;
  float* xs = smem;                                   // [TILE][dpx]   (16-byte aligned rows when SE44)
  float* zs = xs + TILE * (SE44 ? 8 : dpz);           // [TILE][dpz]
  uint32_t* tile = reinterpret_cast<uint32_t*>(zs + TILE * dpz);   // [TILE][TILE + 1] packed {hi | lo << 16}
  float* nxa = reinterpret_cast<float*>(tile + TILE * (TILE + 1));
  float* nxb = nxa + TILE;
  float* nza = nxb + TILE;
  float* nzb = nza + TILE;
  float* il = nzb + TILE;                             // ARD: [MAXD]
  constexpr int P = TILE + 1;
  static_assert(!(SE44 && ARD), "ARD specs take the generic planes builder");
  const Hyp h = ARD ? ard_hyp(load_hyp(hyp), sp) : load_hyp(hyp);
  if (ARD) load_ard(hyp, sp, il, nullptr);
  const int64_t col0 = (int64_t)blockIdx.x * TILE;
  const int64_t ntiles_r = (N + TILE - 1) / TILE;
  const float scale = plane_scale(sp, h, kscale);
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
    kscale[0] = scale; kscale[1] = 1.0f / scale; kscale[6] = kernel_nonneg(sp) ? 1.0f : 0.0f;
  }

  load_features(Fz, ldz, col0, M, d, dpz, sp, zs, nza, nzb);
  const int c = threadIdx.x % TILE, rg = threadIdx.x / TILE;   // compute phase: one column, 16 rows per thread
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k4 = lane & 3, sub = lane >> 2;                   // read-out phase: 4 lanes x 8 entries = 32 entries
  float zr[8];
  float ca = 0.f, cb = 0.f, amp2s = 0.f;
  if (SE44) {
#pragma unroll
    for (int f = 0; f < 8; ++f) zr[f] = zs[c * dpz + f];
    const float LOG2E = 1.4426950408889634f;
    ca = -0.5f * LOG2E / (h.len_a * h.len_a);
    cb = -0.5f * LOG2E / (h.len_b * h.len_b);
    amp2s = h.amp_a * h.amp_a * h.amp_b * h.amp_b * scale;
  }
  const bool vec_rows = (ldkh % 8) == 0 && ((reinterpret_cast<uintptr_t>(Kh) | reinterpret_cast<uintptr_t>(Kl)) & 15) == 0;
  const bool vec_cols = (ldkt % 8) == 0 && ((reinterpret_cast<uintptr_t>(Kth) | reinterpret_cast<uintptr_t>(Ktl)) & 15) == 0;

  for (int64_t rt = blockIdx.y; rt < ntiles_r; rt += gridDim.y) {
    const int64_t row0 = rt * TILE;
    load_features(Fx, ldx, row0, N, d, dpx, sp, xs, nxa, nxb);
#pragma unroll 4
    for (int j = 0; j < TILE / 4; ++j) {
      const int r = rg + 4 * j;
      float vs;
      if (SE44) {
        const float4 xa = *reinterpret_cast<const float4*>(xs + r * 8);
        const float4 xb = *reinterpret_cast<const float4*>(xs + r * 8 + 4);
        float t, ra, rb;
        t = xa.x - zr[0]; ra = t * t;
        t = xa.y - zr[1]; ra = fmaf(t, t, ra);
        t = xa.z - zr[2]; ra = fmaf(t, t, ra);
        t = xa.w - zr[3]; ra = fmaf(t, t, ra);
        t = xb.x - zr[4]; rb = t * t;
        t = xb.y - zr[5]; rb = fmaf(t, t, rb);
        t = xb.z - zr[6]; rb = fmaf(t, t, rb);
        t = xb.w - zr[7]; rb = fmaf(t, t, rb);
        vs = amp2s * exp2f(fmaf(ca, ra, cb * rb));
      } else {
        const float ka = factor_value<ARD>(sp.ta, xs + r * dpx, zs + c * dpz, sp.da, h.amp_a, h.len_a, nxa[r], nza[c], il);
        const float kb = factor_value<ARD>(sp.tb, xs + r * dpx + sp.da, zs + c * dpz + sp.da, sp.db, h.amp_b, h.len_b, nxb[r],
                                           nzb[c], il + sp.da);
        vs = ka * kb * scale;
      }
      if (row0 + r >= N) vs = 0.f;                    // datapoints past N are zero in the blocked transpose
      const __half hi = __float2half_rn(vs);
      const __half lo = __float2half_rn(vs - __half2float(hi));
      tile[r * P + c] = (uint32_t)__half_as_ushort(hi) | ((uint32_t)__half_as_ushort(lo) << 16);
    }
    __syncthreads();
    // read-out: a warp covers 8 tile rows (or columns) x 32 entries; bank = (line + 8 k4 + i) mod 32 -> conflict-free
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      uint32_t w[8];
      {   // Kh / Kl: row r, columns e0 .. e0 + 7
        const int r = warp * 8 + sub, e0 = half * 32 + k4 * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = tile[r * P + e0 + i];
        const int64_t gr = row0 + r, gc = col0 + e0;
        if (gr < N && gc < M) {
          const int64_t o = gr * ldkh + gc;
          if (vec_rows && gc + 8 <= M) {
            *reinterpret_cast<uint4*>(Kh + o) = make_uint4(__byte_perm(w[0], w[1], 0x5410), __byte_perm(w[2], w[3], 0x5410),
                                                           __byte_perm(w[4], w[5], 0x5410), __byte_perm(w[6], w[7], 0x5410));
            *reinterpret_cast<uint4*>(Kl + o) = make_uint4(__byte_perm(w[0], w[1], 0x7632), __byte_perm(w[2], w[3], 0x7632),
                                                           __byte_perm(w[4], w[5], 0x7632), __byte_perm(w[6], w[7], 0x7632));
          } else {
            for (int i = 0; i < 8 && gc + i < M; ++i) {
              Kh[o + i] = __ushort_as_half((unsigned short)(w[i] & 0xffffu));
              Kl[o + i] = __ushort_as_half((unsigned short)(w[i] >> 16));
            }
          }
        }
      }
      {   // Kth / Ktl: column cc, datapoints e0 .. e0 + 7 of this 64-datapoint block (block stride ldkt)
        const int cc = warp * 8 + sub, e0 = half * 32 + k4 * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = tile[(e0 + i) * P + cc];
        const int64_t gc = col0 + cc;
        if (gc < M) {
          const int64_t o = rt * ldkt + gc * TILE + e0;
          if (vec_cols) {
            *reinterpret_cast<uint4*>(Kth + o) = make_uint4(__byte_perm(w[0], w[1], 0x5410), __byte_perm(w[2], w[3], 0x5410),
                                                            __byte_perm(w[4], w[5], 0x5410), __byte_perm(w[6], w[7], 0x5410));
            *reinterpret_cast<uint4*>(Ktl + o) = make_uint4(__byte_perm(w[0], w[1], 0x7632), __byte_perm(w[2], w[3], 0x7632),
                                                            __byte_perm(w[4], w[5], 0x7632), __byte_perm(w[6], w[7], 0x7632));
          } else {
            for (int i = 0; i < 8; ++i) {
              Kth[o + i] = __ushort_as_half((unsigned short)(w[i] & 0xffffu));
              Ktl[o + i] = __ushort_as_half((unsigned short)(w[i] >> 16));
            }
          }
        }
      }
    }
    __syncthreads();
  }
}

// float64 kernel matrix (fp32 features, float64 arithmetic): OutT = double is K_mm of the M x M stage; OutT = float is the plain
// K_nm of the small (SIMT-path) problems, ONE rounding of the float64 value -- the fp32 evaluation of the exponential carries
// ~5e-7 of relative error (rounding of its argument), which e.g. the (b x b) solve of the Titsias bound amplifies to 1.2e-4 in dy
// ARD: launched with MAXD doubles of dynamic shared memory for the inverse length scales
template <typename OutT, bool ARD = false>
__global__ void kernel_fwd_f64_kernel(const float* __restrict__ Fx, int64_t ldx, int64_t N, const float* __restrict__ Fz, int64_t ldz,
                                      int64_t M, Spec sp, const float* __restrict__ hyp, OutT* __restrict__ K, int64_t ldk) {
  extern __shared__ double il_f64[];
  const Hyp h = ARD ? ard_hyp(load_hyp(hyp), sp) : load_hyp(hyp);
  if (ARD) {
    load_ard(hyp, sp, nullptr, il_f64);
    __syncthreads();
  }
  const int64_t total = N * M;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = idx / M, j = idx - i * M;
    const float* x = Fx + i * ldx;
    const float* z = Fz + j * ldz;
    const double ka = factor_value_f64<ARD>(sp.ta, x, z, sp.da, h.amp_a, h.len_a, sp.ta == SVGP_K_COSINE ? block_norm_f64(x, sp.da) : 1.0,
                                            sp.ta == SVGP_K_COSINE ? block_norm_f64(z, sp.da) : 1.0, il_f64);
    const double kb = factor_value_f64<ARD>(sp.tb, x + sp.da, z + sp.da, sp.db, h.amp_b, h.len_b,
                                            sp.tb == SVGP_K_COSINE ? block_norm_f64(x + sp.da, sp.db) : 1.0,
                                            sp.tb == SVGP_K_COSINE ? block_norm_f64(z + sp.da, sp.db) : 1.0, il_f64 + sp.da);
    K[i * ldk + j] = (OutT)(ka * kb);
  }
}

// Builder of the integer tensor-core operand format (tc_i8_engine.cu, i8_planes.cu): every entry of K_nm as a 32-bit
// fixed-point integer against the largest entry of its ROW (Kr: products that reduce over the inducing points) and of
// its COLUMN (Kc, datapoint-blocked transpose: the SYRK), cut into four balanced base-256 digit planes each -- written
// straight from the fp32 kernel values, so the planes carry fp32 accuracy (a plane derived from the fp16 hi/lo pair
// would stop at 22 bits; the M = 2048 sweep point needs more: tools/numerics/sim_parity.py) -- plus the fp16 hi/lo row
// planes the remaining fp16 consumers read.  Two passes over the same tiles: MAXPASS = true only reduces the row and
// column maxima (float bits, atomicMax), MAXPASS = false writes.
// ARD: the generic form reads the inverse length scales from shared memory (ARD_SMEM behind the layout); SE44 keeps the
// per-feature exponent factors -log2(e) / (2 l_f^2) in registers, in fp32 for the maxima and in float64 for the write
template <bool SE44, bool MAXPASS, bool ARD = false>
__global__ void __launch_bounds__(THREADS) kernel_fwd_i8_kernel(
    const float* __restrict__ Fx, int64_t ldx, int64_t N, const float* __restrict__ Fz, int64_t ldz, int64_t M,
    Spec sp, const float* __restrict__ hyp, __half* __restrict__ Kh, __half* __restrict__ Kl, int64_t ldkh,
    int8_t* __restrict__ Kr, int64_t ldkr, float* __restrict__ rscale, int8_t* __restrict__ Kc, float* __restrict__ cscale,
    float* __restrict__ rmax, float* __restrict__ cmax, float* __restrict__ kscale) {
  extern __shared__ float smem[];
  const int d = sp.da + sp.db;
  const int dpx = SE44 ? 8 : (d | 1), dpz = d | 1;
  float* xs = smem;
  float* zs = xs + TILE * (SE44 ? 8 : dpz);
  float* tile = zs + TILE * dpz;                      // [TILE][TILE + 1] kernel values (fp32)
  float* nxa = tile + TILE * (TILE + 1);
  float* nxb = nxa + TILE;
  float* nza = nxb + TILE;
  float* nzb = nza + TILE;
  float* il = nzb + TILE;                             // ARD, generic: float[MAXD], then double[MAXD]
  double* ild = reinterpret_cast<double*>(il + MAXD);
  constexpr int P = TILE + 1;
  // POWER-OF-TWO fixed-point grids: max = m 2^e (m in [0.5, 1)) -> integer = value * 2^(31 - e) (2^(30 - e) when m > 0.99).  The
  // product with a power of two is exact in fp32 and a 24-bit mantissa within 2^-7 of the maximum fits the grid whole, so
  // the row-scaled and the column-scaled planes hold THE SAME number wherever it matters.  (With max / (127 2^24) as the
  // unit the two grids rounded every entry independently at the 2^-24 level; that inconsistency between the K_nm of the
  // SYRK and the K_nm of everything else alone cost 1e-4 of the inducing-point gradient at M = 2048.)
  auto pow2_q = [](float m) -> float {
    if (!(m > 0.f)) return 0.f;
    int e;
    const float f = frexpf(m, &e);                      // m = f 2^e, f in [0.5, 1)
    e = (f <= 0.99f ? 31 : 30) - e;                     // largest integer <= 127 2^24 = 0.992 2^31 (the top digit is signed)
    e = e > 120 ? 120 : (e < -120 ? -120 : e);
    return ldexpf(1.0f, e);
  };
  const Hyp h = ARD ? ard_hyp(load_hyp(hyp), sp) : load_hyp(hyp);
  if (ARD && !SE44) load_ard(hyp, sp, il, ild);
  const int64_t col0 = (int64_t)blockIdx.x * TILE;
  const int64_t ntiles_r = (N + TILE - 1) / TILE;
  const float scale = plane_scale(sp, h, kscale);
  if (!MAXPASS && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
    kscale[0] = scale; kscale[1] = 1.0f / scale; kscale[6] = kernel_nonneg(sp) ? 1.0f : 0.0f;
  }
  load_features(Fz, ldz, col0, M, d, dpz, sp, zs, nza, nzb);
  const int c = threadIdx.x % TILE, rg = threadIdx.x / TILE;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k4 = lane & 3, sub = lane >> 2;
  float zr[8];
  float ca = 0.f, cb = 0.f, amp2 = 0.f;
  float cf[ARD ? 8 : 1];                              // SE44 + ARD: -log2(e) / (2 l_f^2), fp32 (maxima) ...
  double cfd[ARD ? 8 : 1];                            // ... and float64 (write pass)
  if (SE44) {
#pragma unroll
    for (int f = 0; f < 8; ++f) zr[f] = zs[c * dpz + f];
    const float LOG2E = 1.4426950408889634f;
    ca = -0.5f * LOG2E / (h.len_a * h.len_a);
    cb = -0.5f * LOG2E / (h.len_b * h.len_b);
    amp2 = h.amp_a * h.amp_a * h.amp_b * h.amp_b;
    if (ARD) {
#pragma unroll
      for (int f = 0; f < 8; ++f) {
        const double l = ard_len(hyp, sp, h, f);
        if (MAXPASS) cf[f] = -0.5f * LOG2E / (float)(l * l);
        else cfd[f] = -0.5 * 1.4426950408889634 / (l * l);
      }
    }
  }
  const double LOG2E_D = 1.4426950408889634;
  const double cad = -0.5 * LOG2E_D / ((double)h.len_a * (double)h.len_a), cbd = -0.5 * LOG2E_D / ((double)h.len_b * (double)h.len_b);
  const double amp2d = (double)h.amp_a * (double)h.amp_a * (double)h.amp_b * (double)h.amp_b;
  const int64_t nb128 = (N + 127) / 128;
  const int64_t rplane = N * ldkr, cplane = nb128 * M * 128;
  float colmax = 0.f;                                 // MAXPASS: this thread's column over all its row tiles
  float qc = 0.f;                                     // write pass: quantisation factor of the read-out column
  if (!MAXPASS) {
    const int64_t gc = col0 + warp * 8 + sub;
    const float m = gc < M ? cmax[gc] : 0.f;
    qc = pow2_q(m);
    if (blockIdx.y == 0 && k4 == 0 && gc < M) cscale[gc] = qc > 0.f ? 1.0f / qc : 0.f;
  }

  for (int64_t rt = blockIdx.y; rt < ntiles_r; rt += gridDim.y) {
    const int64_t row0 = rt * TILE;
    load_features(Fx, ldx, row0, N, d, dpx, sp, xs, nxa, nxb);
#pragma unroll 4
    for (int j = 0; j < TILE / 4; ++j) {
      const int r = rg + 4 * j;
      float v;
      if (SE44 && ARD) {
        // exponent sum_f c_f (x_f - z_f)^2: fp32 for the maxima; for the write pass the float64 difference times the
        // float64 c_f (one DMUL per feature on top of the isotropic form) and one rounding at the end
        const float4 xa = *reinterpret_cast<const float4*>(xs + r * 8);
        const float4 xb = *reinterpret_cast<const float4*>(xs + r * 8 + 4);
        const float xv[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
        if (MAXPASS) {
          float e = 0.f;
#pragma unroll
          for (int f = 0; f < 8; ++f) { const float t = xv[f] - zr[f]; e = fmaf(cf[f] * t, t, e); }
          v = amp2 * exp2f(e);
        } else {
          double e = 0.0;
#pragma unroll
          for (int f = 0; f < 8; ++f) { const double t = (double)xv[f] - (double)zr[f]; e = fma(cfd[f] * t, t, e); }
          v = (float)(amp2d * exp2(e));
        }
      } else if (SE44 && MAXPASS) {
        const float4 xa = *reinterpret_cast<const float4*>(xs + r * 8);
        const float4 xb = *reinterpret_cast<const float4*>(xs + r * 8 + 4);
        float t, ra, rb;
        t = xa.x - zr[0]; ra = t * t;
        t = xa.y - zr[1]; ra = fmaf(t, t, ra);
        t = xa.z - zr[2]; ra = fmaf(t, t, ra);
        t = xa.w - zr[3]; ra = fmaf(t, t, ra);
        t = xb.x - zr[4]; rb = t * t;
        t = xb.y - zr[5]; rb = fmaf(t, t, rb);
        t = xb.z - zr[6]; rb = fmaf(t, t, rb);
        t = xb.w - zr[7]; rb = fmaf(t, t, rb);
        v = amp2 * exp2f(fmaf(ca, ra, cb * rb));
      } else if (SE44) {
        // write pass: float64 evaluation (the maxima above only position the fixed-point grid)
        const float4 xa = *reinterpret_cast<const float4*>(xs + r * 8);
        const float4 xb = *reinterpret_cast<const float4*>(xs + r * 8 + 4);
        double t, ra, rb;
        t = (double)xa.x - (double)zr[0]; ra = t * t;
        t = (double)xa.y - (double)zr[1]; ra = fma(t, t, ra);
        t = (double)xa.z - (double)zr[2]; ra = fma(t, t, ra);
        t = (double)xa.w - (double)zr[3]; ra = fma(t, t, ra);
        t = (double)xb.x - (double)zr[4]; rb = t * t;
        t = (double)xb.y - (double)zr[5]; rb = fma(t, t, rb);
        t = (double)xb.z - (double)zr[6]; rb = fma(t, t, rb);
        t = (double)xb.w - (double)zr[7]; rb = fma(t, t, rb);
        v = (float)(amp2d * exp2(fma(cad, ra, cbd * rb)));
      } else if (MAXPASS) {
        const float ka = factor_value<ARD>(sp.ta, xs + r * dpx, zs + c * dpz, sp.da, h.amp_a, h.len_a, nxa[r], nza[c], il);
        const float kb = factor_value<ARD>(sp.tb, xs + r * dpx + sp.da, zs + c * dpz + sp.da, sp.db, h.amp_b, h.len_b, nxb[r],
                                           nzb[c], il + sp.da);
        v = ka * kb;
      } else {
        const double ka = factor_value_f64<ARD>(sp.ta, xs + r * dpx, zs + c * dpz, sp.da, h.amp_a, h.len_a,
                                                sp.ta == SVGP_K_COSINE ? block_norm_f64(xs + r * dpx, sp.da) : 1.0,
                                                sp.ta == SVGP_K_COSINE ? block_norm_f64(zs + c * dpz, sp.da) : 1.0, ild);
        const double kb = factor_value_f64<ARD>(sp.tb, xs + r * dpx + sp.da, zs + c * dpz + sp.da, sp.db, h.amp_b, h.len_b,
                                                sp.tb == SVGP_K_COSINE ? block_norm_f64(xs + r * dpx + sp.da, sp.db) : 1.0,
                                                sp.tb == SVGP_K_COSINE ? block_norm_f64(zs + c * dpz + sp.da, sp.db) : 1.0,
                                                ild + sp.da);
        v = (float)(ka * kb);
      }
      if (row0 + r >= N || col0 + c >= M) v = 0.f;
      if (MAXPASS) colmax = fmaxf(colmax, fabsf(v));
      tile[r * P + c] = v;
    }
    __syncthreads();
    if (MAXPASS) {
      // row maxima of this tile: a warp covers 8 rows x 64 columns (4 lanes x 16 entries per row)
      const int r = warp * 8 + sub;
      float m = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) m = fmaxf(m, fabsf(tile[r * P + k4 * 16 + i]));
      m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
      m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 2));
      if (k4 == 0 && row0 + r < N && m > 0.f) atomicMax(reinterpret_cast<int*>(rmax + row0 + r), __float_as_int(m));
    } else {
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        {   // row r, columns e0 .. e0 + 7: fp16 hi / lo planes and the row-scaled digits
          const int r = warp * 8 + sub, e0 = half * 32 + k4 * 8;
          const int64_t gr = row0 + r, gc = col0 + e0;
          if (gr < N && gc < M) {
            const float qr = pow2_q(rmax[gr]);
            if (blockIdx.x == 0 && e0 == 0) rscale[gr] = qr > 0.f ? 1.0f / qr : 0.f;
            uint32_t hw[4], lw[4], e[8];
#pragma unroll
            for (int i = 0; i < 8; i += 2) {
              const float v0 = tile[r * P + e0 + i], v1 = tile[r * P + e0 + i + 1];
              const __half2 hi = __floats2half2_rn(v0 * scale, v1 * scale);
              const float2 hf = __half22float2(hi);
              const __half2 lo = __floats2half2_rn(v0 * scale - hf.x, v1 * scale - hf.y);
              hw[i >> 1] = *reinterpret_cast<const uint32_t*>(&hi);
              lw[i >> 1] = *reinterpret_cast<const uint32_t*>(&lo);
              e[i] = ((uint32_t)__float2int_rn(v0 * qr) + 0x00808080u) ^ 0x00808080u;
              e[i + 1] = ((uint32_t)__float2int_rn(v1 * qr) + 0x00808080u) ^ 0x00808080u;
            }
            // (columns >= M inside this run are zero in the tile: zero digits)
            *reinterpret_cast<uint4*>(Kh + gr * ldkh + gc) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
            *reinterpret_cast<uint4*>(Kl + gr * ldkh + gc) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
            uint32_t w0[4], w1[4];
            {
              const uint32_t x01 = __byte_perm(e[0], e[1], 0x7362), y01 = __byte_perm(e[0], e[1], 0x5140);
              const uint32_t x23 = __byte_perm(e[2], e[3], 0x7362), y23 = __byte_perm(e[2], e[3], 0x5140);
              w0[0] = __byte_perm(x01, x23, 0x7632); w0[1] = __byte_perm(x01, x23, 0x5410);
              w0[2] = __byte_perm(y01, y23, 0x7632); w0[3] = __byte_perm(y01, y23, 0x5410);
            }
            {
              const uint32_t x01 = __byte_perm(e[4], e[5], 0x7362), y01 = __byte_perm(e[4], e[5], 0x5140);
              const uint32_t x23 = __byte_perm(e[6], e[7], 0x7362), y23 = __byte_perm(e[6], e[7], 0x5140);
              w1[0] = __byte_perm(x01, x23, 0x7632); w1[1] = __byte_perm(x01, x23, 0x5410);
              w1[2] = __byte_perm(y01, y23, 0x7632); w1[3] = __byte_perm(y01, y23, 0x5410);
            }
#pragma unroll
            for (int s = 0; s < 4; ++s) *reinterpret_cast<uint2*>(Kr + s * rplane + gr * ldkr + gc) = make_uint2(w0[s], w1[s]);
          }
        }
        {   // column cc, datapoints e0 .. e0 + 7 of this 64-datapoint half block: column-scaled digits, blocked by 128
          const int cc = warp * 8 + sub, e0 = half * 32 + k4 * 8;
          const int64_t gc = col0 + cc;
          if (gc < M) {
            uint32_t e[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) e[i] = ((uint32_t)__float2int_rn(tile[(e0 + i) * P + cc] * qc) + 0x00808080u) ^ 0x00808080u;
            uint32_t w0[4], w1[4];
            {
              const uint32_t x01 = __byte_perm(e[0], e[1], 0x7362), y01 = __byte_perm(e[0], e[1], 0x5140);
              const uint32_t x23 = __byte_perm(e[2], e[3], 0x7362), y23 = __byte_perm(e[2], e[3], 0x5140);
              w0[0] = __byte_perm(x01, x23, 0x7632); w0[1] = __byte_perm(x01, x23, 0x5410);
              w0[2] = __byte_perm(y01, y23, 0x7632); w0[3] = __byte_perm(y01, y23, 0x5410);
            }
            {
              const uint32_t x01 = __byte_perm(e[4], e[5], 0x7362), y01 = __byte_perm(e[4], e[5], 0x5140);
              const uint32_t x23 = __byte_perm(e[6], e[7], 0x7362), y23 = __byte_perm(e[6], e[7], 0x5140);
              w1[0] = __byte_perm(x01, x23, 0x7632); w1[1] = __byte_perm(x01, x23, 0x5410);
              w1[2] = __byte_perm(y01, y23, 0x7632); w1[3] = __byte_perm(y01, y23, 0x5410);
            }
            const int64_t o = ((row0 >> 7) * M + gc) * 128 + (row0 & 127) + e0;
#pragma unroll
            for (int s = 0; s < 4; ++s) *reinterpret_cast<uint2*>(Kc + s * cplane + o) = make_uint2(w0[s], w1[s]);
          }
        }
      }
    }
    __syncthreads();
  }
  if (MAXPASS) {
    // fold the four row groups of every column, then one atomic per column and block
    __syncthreads();
    tile[rg * P + c] = colmax;
    __syncthreads();
    if (rg == 0) {
      const float m = fmaxf(fmaxf(tile[c], tile[P + c]), fmaxf(tile[2 * P + c], tile[3 * P + c]));
      if (col0 + c < M && m > 0.f) atomicMax(reinterpret_cast<int*>(cmax + col0 + c), __float_as_int(m));
    }
  }
}

// ------------------------------------------------------------------------------------------
// backward.  Two passes over the same tiles so that neither needs float atomics on N-sized data:
//   pass X: one block per row tile walks every column tile      -> dFx rows (plain stores)
//   pass Z: one block per (column tile, row slab) walks its rows -> dFz, dhyp (double atomics,
//           one flush per block)
// ACC64 (pass Z of the Matern factors): the per-tile fp32 partials are folded into double across the row tiles and the
// flush  dz_f = sum c1 x_f + z_f sum c2z  (which cancels: c2z = -c1) is done in double, as in kernel_bwd_z_se44_kernel
// ARD: the coefficients are those of the scaled coordinates (factor_adjoint), the phase-2 sums run on the unscaled
// features, and the flush multiplies by il_f^2.  Pass Z also sums  c1 (x_f - z_f)^2  per entry for every feature of an
// ARD block (fp32 per tile, folded into double): dl_f = il_f^3 times that.  (Per-column moments sum c1 x^2, sum c1 x,
// sum c1 would cancel by orders of magnitude in fp32 for offset features such as time stamps.)
// ------------------------------------------------------------------------------------------
template <bool PASS_X, bool ACC64 = false, bool ARD = false>
__global__ void __launch_bounds__(THREADS) kernel_bwd_kernel(
    const float* __restrict__ Fx, int64_t ldx, int64_t N, const float* __restrict__ Fz, int64_t ldz, int64_t M,
    Spec sp, const float* __restrict__ hyp, const float* __restrict__ G, int64_t ldg, float* __restrict__ dFx,
    double* __restrict__ dFz, double* __restrict__ dhyp) {
  static_assert(!(PASS_X && ACC64), "ACC64 is a Z-pass variant");
  extern __shared__ float smem[];
  const int d = sp.da + sp.db, dp = d | 1;
  float* xs = smem;
  float* zs = xs + TILE * dp;
  float* c1a = zs + TILE * dp;                  // [TILE][TILE+1] coefficient on the other side's features (block A)
  float* c1b = c1a + TILE * (TILE + 1);         // same, block B
  float* nxa = c1b + TILE * (TILE + 1);
  float* nxb = nxa + TILE;
  float* nza = nxb + TILE;
  float* nzb = nza + TILE;
  float* own = nzb + TILE;                      // [TILE][4]: scalar coefficients on own features {c2 A, c2 B, e A, e B}
  float* hred = own + TILE * 4;                 // [4] hyper partials (float atomics in smem)
  float* il = hred + 4;                         // ARD: [MAXD]
  const Hyp h = ARD ? ard_hyp(load_hyp(hyp), sp) : load_hyp(hyp);
  if (ARD) load_ard(hyp, sp, il, nullptr);
  const int c = threadIdx.x % TILE, rg = threadIdx.x / TILE;
  const int64_t ntr = (N + TILE - 1) / TILE, ntc = (M + TILE - 1) / TILE;

  // outer = the tile whose gradient this block owns, inner = the tiles it walks
  const int64_t n_outer = PASS_X ? ntr : ntc;
  const int64_t n_inner = PASS_X ? ntc : ntr;
  for (int64_t ot = blockIdx.x; ot < n_outer; ot += gridDim.x) {
    // accumulators for (own row/col = threadIdx%TILE, features fg, fg+4, ...)
    float acc[MAXD / 4];
#pragma unroll
    for (int q = 0; q < MAXD / 4; ++q) acc[q] = 0.f;
    float own_acc[4] = {0.f, 0.f, 0.f, 0.f};
    double acc64[ACC64 ? MAXD / 4 : 1], own64[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int q = 0; q < (ACC64 ? MAXD / 4 : 1); ++q) acc64[q] = 0.0;
    // hyper-parameter gradients are heavily cancelling sums over all N x M entries: accumulate them in double
    double hy[4] = {0.0, 0.0, 0.0, 0.0};
    double hyl[ARD && !PASS_X ? MAXD / 4 : 1];   // ARD: sum c1 (x_f - z_f)^2 of the owned column, features fg + 4q
#pragma unroll
    for (int q = 0; q < (ARD && !PASS_X ? MAXD / 4 : 1); ++q) hyl[q] = 0.0;
    if (threadIdx.x < 4) hred[threadIdx.x] = 0.f;
    if (PASS_X) load_features(Fx, ldx, ot * TILE, N, d, dp, sp, xs, nxa, nxb);
    else        load_features(Fz, ldz, ot * TILE, M, d, dp, sp, zs, nza, nzb);

    for (int64_t it = (PASS_X ? 0 : blockIdx.y); it < n_inner; it += (PASS_X ? 1 : gridDim.y)) {
      const int64_t row0 = (PASS_X ? ot : it) * TILE, col0 = (PASS_X ? it : ot) * TILE;
      if (PASS_X) load_features(Fz, ldz, col0, M, d, dp, sp, zs, nza, nzb);
      else        load_features(Fx, ldx, row0, N, d, dp, sp, xs, nxa, nxb);
      for (int idx = threadIdx.x; idx < TILE * 4; idx += THREADS) own[idx] = 0.f;
      __syncthreads();
      // phase 1: coefficients for the 64x64 tile (thread: fixed column c, rows rg + 4j)
      float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f;   // PASS_Z: sums over rows for column c
      for (int j = 0; j < TILE / 4; ++j) {
        int r = rg + 4 * j;
        int64_t gr = row0 + r, gc = col0 + c;
        float g = (gr < N && gc < M) ? G[gr * ldg + gc] : 0.f;
        const float* xa = xs + r * dp;
        const float* za = zs + c * dp;
        float ka = factor_value<ARD>(sp.ta, xa, za, sp.da, h.amp_a, h.len_a, nxa[r], nza[c], il);
        float kb = factor_value<ARD>(sp.tb, xa + sp.da, za + sp.da, sp.db, h.amp_b, h.len_b, nxb[r], nzb[c], il + sp.da);
        FactorAdj A = factor_adjoint<ARD>(sp.ta, xa, za, sp.da, h.amp_a, h.len_a, nxa[r], nza[c], ka, g * kb, il);
        FactorAdj B = factor_adjoint<ARD>(sp.tb, xa + sp.da, za + sp.da, sp.db, h.amp_b, h.len_b, nxb[r], nzb[c], kb, g * ka,
                                          il + sp.da);
        if (ARD && sp.ard_a) A.dlen = 0.f;        // an ARD block's isotropic slot gets exactly 0
        if (ARD && sp.ard_b) B.dlen = 0.f;
        c1a[r * (TILE + 1) + c] = A.c1;
        c1b[r * (TILE + 1) + c] = B.c1;
        if (PASS_X) {
          // sums over columns for row r: reduce across the 32 lanes of this warp (same row)
          float s0 = warp_sum(A.c2x), s1 = warp_sum(B.c2x), s2 = warp_sum(-A.e), s3 = warp_sum(-B.e);
          if ((threadIdx.x & 31) == 0) {
            atomicAdd(&own[r * 4 + 0], s0); atomicAdd(&own[r * 4 + 1], s1);
            atomicAdd(&own[r * 4 + 2], s2); atomicAdd(&own[r * 4 + 3], s3);
          }
        } else {
          o0 += A.c2z; o1 += B.c2z; o2 += A.e; o3 += B.e;
          hy[0] += A.damp; hy[1] += A.dlen; hy[2] += B.damp; hy[3] += B.dlen;
        }
      }
      if (!PASS_X) {
        atomicAdd(&own[c * 4 + 0], o0); atomicAdd(&own[c * 4 + 1], o1);
        atomicAdd(&own[c * 4 + 2], o2); atomicAdd(&own[c * 4 + 3], o3);
      }
      __syncthreads();
      // phase 2: own-side gradient. thread: own index o = threadIdx%TILE, features fg + 4q
      {
        const int o = threadIdx.x % TILE, fg = threadIdx.x / TILE;
#pragma unroll
        for (int q = 0; q < MAXD / 4; ++q) {
          const int f = fg + 4 * q;
          if (f < d) {
            const float* cmat = (f < sp.da) ? c1a : c1b;
            float s = 0.f;
            if (PASS_X) {
              for (int k = 0; k < TILE; ++k) s = fmaf(cmat[o * (TILE + 1) + k], zs[k * dp + f], s);
            } else {
              for (int k = 0; k < TILE; ++k) s = fmaf(cmat[k * (TILE + 1) + o], xs[k * dp + f], s);
            }
            if (ACC64) acc64[q] += (double)s;
            else acc[q] += s;
            if (ARD && !PASS_X && ard_feature(sp, f)) {
              const float zf = zs[o * dp + f];
              float s2 = 0.f;
              for (int k = 0; k < TILE; ++k) {
                const float t = xs[k * dp + f] - zf;
                s2 = fmaf(cmat[k * (TILE + 1) + o] * t, t, s2);
              }
              hyl[q] += (double)s2;
            }
          }
        }
        if (ACC64) {          // every thread keeps its own copy: the flush needs no broadcast
          own64[0] += (double)own[o * 4 + 0]; own64[1] += (double)own[o * 4 + 1];
          own64[2] += (double)own[o * 4 + 2]; own64[3] += (double)own[o * 4 + 3];
        } else if (fg == 0) {
          own_acc[0] += own[o * 4 + 0]; own_acc[1] += own[o * 4 + 1];
          own_acc[2] += own[o * 4 + 2]; own_acc[3] += own[o * 4 + 3];
        }
      }
      __syncthreads();
    }
    // flush
    {
      const int o = threadIdx.x % TILE, fg = threadIdx.x / TILE;
      const int64_t go = ot * TILE + o;
      const float* self = (PASS_X ? xs : zs) + o * dp;
      // broadcast the per-own-index scalars from the fg == 0 thread through shared memory
      if (fg == 0) { own[o * 4 + 0] = own_acc[0]; own[o * 4 + 1] = own_acc[1]; own[o * 4 + 2] = own_acc[2]; own[o * 4 + 3] = own_acc[3]; }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < MAXD / 4; ++q) {
        const int f = fg + 4 * q;
        if (f >= d) continue;
        bool inA = f < sp.da;
        if (ACC64) {
          double v = acc64[q] + own64[inA ? 0 : 1] * (double)self[f];
          if (inA && f == 0 && sp.ta == SVGP_K_EXPSIN) v += own64[2];
          if (!inA && f == sp.da && sp.tb == SVGP_K_EXPSIN) v += own64[3];
          if (ARD) v *= (double)il[f] * (double)il[f];
          if (go < M) atomicAdd(&dFz[go * d + f], v);
          continue;
        }
        float v = acc[q] + own[o * 4 + (inA ? 0 : 1)] * self[f];
        // EXPSIN contributes only through its single feature (the first of its block)
        if (inA && f == 0 && sp.ta == SVGP_K_EXPSIN) v += own[o * 4 + 2];
        if (!inA && f == sp.da && sp.tb == SVGP_K_EXPSIN) v += own[o * 4 + 3];
        if (ARD) v *= il[f] * il[f];
        if (PASS_X) {
          if (go < N) dFx[go * d + f] = v;
        } else {
          if (go < M) atomicAdd(&dFz[go * d + f], (double)v);
        }
      }
      if (!PASS_X) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          double s = hy[k];
#pragma unroll
          for (int o2 = 16; o2 > 0; o2 >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o2);
          if ((threadIdx.x & 31) == 0) atomicAdd(&dhyp[k], s);          // one double atomic per warp per owned tile
        }
        if (ARD) {
          // the 32 lanes of a warp share fg: one double atomic per warp and ARD feature
#pragma unroll
          for (int q = 0; q < MAXD / 4; ++q) {
            const int f = fg + 4 * q;
            if (f >= d || !ard_feature(sp, f)) continue;
            const double l = hyp[4 + f];
            double s = hyl[q] / (l * l * l);
#pragma unroll
            for (int o2 = 16; o2 > 0; o2 >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o2);
            if ((threadIdx.x & 31) == 0) atomicAdd(&dhyp[4 + f], s);
          }
        }
      }
      __syncthreads();
    }
  }
}

// Z pass specialised for the product of two 4-feature SE factors (the SWEEP kernel; the generic pass above spends
// ~20 ns per 1000 entries on run-time factor dispatch, a second distance evaluation and four double adds per entry).
// With c = g k:  dz_f = (sum_i c x_if - z_f sum_i c) / l^2,  dl = sum c r2 / l^3,  damp = 2 sum c / amp  per block --
// a thread owns one inducing point (features in registers) and 16 of the 64 datapoints of a tile, the datapoint
// features are broadcast float4 loads, g is read in coalesced 128-byte rows; one float partial per tile, folded into
// double per thread (the hyper-parameter sums cancel heavily), one double atomic per (column, feature) per block.
// ARD (either block): the exponent is sum_f c_f d_f^2 with c_f = -log2(e) / (2 l_f^2), and the eight per-feature sums
// sum c d_f^2 take the place of the two per-block sums sum c r2 (17 partials instead of 11); dz_f = (...) / l_f^2,
// dl_f = sum c d_f^2 / l_f^3, and an isotropic block's dl is the sum of its four.
template <bool ARD = false>
__global__ void __launch_bounds__(THREADS) kernel_bwd_z_se44_kernel(
    const float* __restrict__ Fx, int64_t ldx, int64_t N, const float* __restrict__ Fz, int64_t ldz, int64_t M,
    const float* __restrict__ hyp, const float* __restrict__ G, int64_t ldg, double* __restrict__ dFz,
    double* __restrict__ dhyp, Spec sp) {
  constexpr int NS = ARD ? 17 : 11, NH = ARD ? 12 : 4;   // partials per thread, dhyp slots
  __shared__ __align__(16) float xs[TILE * 8];
  __shared__ double red[4][TILE][NS];            // per row group: 8 feature sums, sum c, sum c r2a, sum c r2b (ARD: 8 x sum c d_f^2)
  const Hyp h = load_hyp(hyp);
  const int c = threadIdx.x % TILE, rg = threadIdx.x / TILE;
  const int64_t ntr = (N + TILE - 1) / TILE;
  const int64_t col0 = (int64_t)blockIdx.x * TILE, gc = col0 + c;
  float z[8];
#pragma unroll
  for (int f = 0; f < 8; ++f) z[f] = gc < M ? Fz[gc * ldz + f] : 0.f;
  const float LOG2E = 1.4426950408889634f;
  const float ca = -0.5f * LOG2E / (h.len_a * h.len_a), cb = -0.5f * LOG2E / (h.len_b * h.len_b);
  const float amp2 = h.amp_a * h.amp_a * h.amp_b * h.amp_b;
  float cf[ARD ? 8 : 1];
  if (ARD) {
#pragma unroll
    for (int f = 0; f < 8; ++f) { const float l = ard_len(hyp, sp, h, f); cf[f] = -0.5f * LOG2E / (l * l); }
  }
  double acc[NS];
#pragma unroll
  for (int q = 0; q < NS; ++q) acc[q] = 0.0;
  for (int64_t rt = blockIdx.y; rt < ntr; rt += gridDim.y) {
    const int64_t row0 = rt * TILE;
    __syncthreads();
    for (int idx = threadIdx.x; idx < TILE * 8; idx += THREADS) {
      const int64_t gr = row0 + (idx >> 3);
      xs[idx] = gr < N ? Fx[gr * ldx + (idx & 7)] : 0.f;
    }
    __syncthreads();
    float t[NS];
#pragma unroll
    for (int q = 0; q < NS; ++q) t[q] = 0.f;
#pragma unroll 4
    for (int j = 0; j < TILE / 4; ++j) {
      const int r = rg + 4 * j;
      const int64_t gr = row0 + r;
      const float g = (gr < N && gc < M) ? __ldg(G + gr * ldg + gc) : 0.f;
      const float4 xa = *reinterpret_cast<const float4*>(xs + r * 8);
      const float4 xb = *reinterpret_cast<const float4*>(xs + r * 8 + 4);
      float d0 = xa.x - z[0], d1 = xa.y - z[1], d2 = xa.z - z[2], d3 = xa.w - z[3];
      float e0 = xb.x - z[4], e1 = xb.y - z[5], e2 = xb.z - z[6], e3 = xb.w - z[7];
      if (ARD) {
        const float sq[8] = {d0 * d0, d1 * d1, d2 * d2, d3 * d3, e0 * e0, e1 * e1, e2 * e2, e3 * e3};
        float ex = 0.f;
#pragma unroll
        for (int f = 0; f < 8; ++f) ex = fmaf(cf[f], sq[f], ex);
        const float ck = g * amp2 * exp2f(ex);
        t[0] = fmaf(ck, xa.x, t[0]); t[1] = fmaf(ck, xa.y, t[1]); t[2] = fmaf(ck, xa.z, t[2]); t[3] = fmaf(ck, xa.w, t[3]);
        t[4] = fmaf(ck, xb.x, t[4]); t[5] = fmaf(ck, xb.y, t[5]); t[6] = fmaf(ck, xb.z, t[6]); t[7] = fmaf(ck, xb.w, t[7]);
        t[8] += ck;
#pragma unroll
        for (int f = 0; f < 8; ++f) t[9 + f] = fmaf(ck, sq[f], t[9 + f]);
        continue;
      }
      const float ra = fmaf(d3, d3, fmaf(d2, d2, fmaf(d1, d1, d0 * d0)));
      const float rb = fmaf(e3, e3, fmaf(e2, e2, fmaf(e1, e1, e0 * e0)));
      const float ck = g * amp2 * exp2f(fmaf(ca, ra, cb * rb));
      t[0] = fmaf(ck, xa.x, t[0]); t[1] = fmaf(ck, xa.y, t[1]); t[2] = fmaf(ck, xa.z, t[2]); t[3] = fmaf(ck, xa.w, t[3]);
      t[4] = fmaf(ck, xb.x, t[4]); t[5] = fmaf(ck, xb.y, t[5]); t[6] = fmaf(ck, xb.z, t[6]); t[7] = fmaf(ck, xb.w, t[7]);
      t[8] += ck; t[9] = fmaf(ck, ra, t[9]); t[10] = fmaf(ck, rb, t[10]);
    }
#pragma unroll
    for (int q = 0; q < NS; ++q) acc[q] += (double)t[q];
  }
#pragma unroll
  for (int q = 0; q < NS; ++q) red[rg][c][q] = acc[q];
  __syncthreads();
  if (ARD && rg == 0 && gc < M) {
    double s[NS], dl[8];
#pragma unroll
    for (int q = 0; q < NS; ++q) s[q] = red[0][c][q] + red[1][c][q] + red[2][c][q] + red[3][c][q];
#pragma unroll
    for (int f = 0; f < 8; ++f) {
      const double l = ard_len(hyp, sp, h, f), il2 = 1.0 / (l * l);
      atomicAdd(&dFz[gc * 8 + f], (s[f] - (double)z[f] * s[8]) * il2);
      dl[f] = s[9 + f] * il2 / l;
    }
    red[0][c][0] = 2.0 * s[8] / h.amp_a; red[0][c][1] = sp.ard_a ? 0.0 : dl[0] + dl[1] + dl[2] + dl[3];
    red[0][c][2] = 2.0 * s[8] / h.amp_b; red[0][c][3] = sp.ard_b ? 0.0 : dl[4] + dl[5] + dl[6] + dl[7];
#pragma unroll
    for (int f = 0; f < 8; ++f) red[0][c][4 + f] = ard_feature(sp, f) ? dl[f] : 0.0;
  } else if (ARD && rg == 0) {
#pragma unroll
    for (int k = 0; k < NH; ++k) red[0][c][k] = 0.0;
  } else if (rg == 0 && gc < M) {
    double s[NS];
#pragma unroll
    for (int q = 0; q < NS; ++q) s[q] = red[0][c][q] + red[1][c][q] + red[2][c][q] + red[3][c][q];
    const double ila = 1.0 / ((double)h.len_a * h.len_a), ilb = 1.0 / ((double)h.len_b * h.len_b);
#pragma unroll
    for (int f = 0; f < 8; ++f) atomicAdd(&dFz[gc * 8 + f], (s[f] - (double)z[f] * s[8]) * (f < 4 ? ila : ilb));
    red[0][c][0] = 2.0 * s[8] / h.amp_a; red[0][c][1] = s[9] * ila / h.len_a;
    red[0][c][2] = 2.0 * s[8] / h.amp_b; red[0][c][3] = s[10] * ilb / h.len_b;
  } else if (rg == 0) {
    red[0][c][0] = red[0][c][1] = red[0][c][2] = red[0][c][3] = 0.0;
  }
  __syncthreads();
  if (threadIdx.x < NH) {
    double s = 0.0;
    for (int k = 0; k < TILE; ++k) s += red[0][k][threadIdx.x];
    atomicAdd(&dhyp[threadIdx.x], s);
  }
}

// ------------------------------------------------------------------------------------------
// element-wise apply (diag_only=True)
// ------------------------------------------------------------------------------------------
// ARD: launched with ARD_SMEM bytes of dynamic shared memory (the inverse length scales; the adjoint also keeps its
// per-feature dl_f partials there)
template <bool ARD = false>
__global__ void kernel_diag_fwd_kernel(const float* __restrict__ Fx, int64_t ldx, const float* __restrict__ Fy,
                                       int64_t ldy, int64_t N, Spec sp, const float* __restrict__ hyp,
                                       float* __restrict__ kd) {
  extern __shared__ float il_diag[];
  const Hyp h = ARD ? ard_hyp(load_hyp(hyp), sp) : load_hyp(hyp);
  if (ARD) {
    load_ard(hyp, sp, il_diag, nullptr);
    __syncthreads();
  }
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    float x[MAXD], y[MAXD];
    const int d = sp.da + sp.db;
    for (int f = 0; f < d; ++f) { x[f] = Fx[i * ldx + f]; y[f] = Fy[i * ldy + f]; }
    float nxa = 1.f, nya = 1.f, nxb = 1.f, nyb = 1.f;
    if (sp.ta == SVGP_K_COSINE) { nxa = block_norm(x, sp.da); nya = block_norm(y, sp.da); }
    if (sp.tb == SVGP_K_COSINE) { nxb = block_norm(x + sp.da, sp.db); nyb = block_norm(y + sp.da, sp.db); }
    float ka = factor_value<ARD>(sp.ta, x, y, sp.da, h.amp_a, h.len_a, nxa, nya, il_diag);
    float kb = factor_value<ARD>(sp.tb, x + sp.da, y + sp.da, sp.db, h.amp_b, h.len_b, nxb, nyb, il_diag + sp.da);
    kd[i] = ka * kb;
  }
}

template <bool ARD = false>
__global__ void kernel_diag_bwd_kernel(const float* __restrict__ Fx, int64_t ldx, const float* __restrict__ Fy,
                                       int64_t ldy, int64_t N, Spec sp, const float* __restrict__ hyp,
                                       const float* __restrict__ g, float* __restrict__ dFx, float* __restrict__ dFy,
                                       double* __restrict__ dhyp) {
  extern __shared__ float il_diag[];
  double* dl = reinterpret_cast<double*>(il_diag + MAXD);       // ARD: this block's sum c1 (x_f - y_f)^2 il_f^3
  const Hyp h = ARD ? ard_hyp(load_hyp(hyp), sp) : load_hyp(hyp);
  if (ARD) {
    load_ard(hyp, sp, il_diag, nullptr);
    for (int f = threadIdx.x; f < MAXD; f += blockDim.x) dl[f] = 0.0;
    __syncthreads();
  }
  double hy[4] = {0.0, 0.0, 0.0, 0.0};
  const int d = sp.da + sp.db;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
    float x[MAXD], y[MAXD];
    for (int f = 0; f < d; ++f) { x[f] = Fx[i * ldx + f]; y[f] = Fy[i * ldy + f]; }
    float nxa = 1.f, nya = 1.f, nxb = 1.f, nyb = 1.f;
    if (sp.ta == SVGP_K_COSINE) { nxa = block_norm(x, sp.da); nya = block_norm(y, sp.da); }
    if (sp.tb == SVGP_K_COSINE) { nxb = block_norm(x + sp.da, sp.db); nyb = block_norm(y + sp.da, sp.db); }
    float ka = factor_value<ARD>(sp.ta, x, y, sp.da, h.amp_a, h.len_a, nxa, nya, il_diag);
    float kb = factor_value<ARD>(sp.tb, x + sp.da, y + sp.da, sp.db, h.amp_b, h.len_b, nxb, nyb, il_diag + sp.da);
    float gi = g[i];
    FactorAdj A = factor_adjoint<ARD>(sp.ta, x, y, sp.da, h.amp_a, h.len_a, nxa, nya, ka, gi * kb, il_diag);
    FactorAdj B = factor_adjoint<ARD>(sp.tb, x + sp.da, y + sp.da, sp.db, h.amp_b, h.len_b, nxb, nyb, kb, gi * ka,
                                      il_diag + sp.da);
    if (ARD && sp.ard_a) A.dlen = 0.f;
    if (ARD && sp.ard_b) B.dlen = 0.f;
    for (int f = 0; f < d; ++f) {
      const FactorAdj& T = (f < sp.da) ? A : B;
      int type = (f < sp.da) ? sp.ta : sp.tb;
      bool first = (f == 0) || (f == sp.da);
      float ex = (type == SVGP_K_EXPSIN && first) ? T.e : 0.f;
      if (ARD) {
        const float il2 = il_diag[f] * il_diag[f];
        dFx[i * d + f] = (T.c1 * y[f] + T.c2x * x[f] - ex) * il2;
        dFy[i * d + f] = (T.c1 * x[f] + T.c2z * y[f] + ex) * il2;
        const float t = x[f] - y[f];
        if (ard_feature(sp, f) && T.c1 * t != 0.f) atomicAdd(&dl[f], (double)(T.c1 * t * t * il2 * il_diag[f]));
        continue;
      }
      dFx[i * d + f] = T.c1 * y[f] + T.c2x * x[f] - ex;
      dFy[i * d + f] = T.c1 * x[f] + T.c2z * y[f] + ex;
    }
    hy[0] += A.damp; hy[1] += A.dlen; hy[2] += B.damp; hy[3] += B.dlen;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    double s = hy[k];
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o2);
    if ((threadIdx.x & 31) == 0 && s != 0.0) atomicAdd(&dhyp[k], s);
  }
  if (ARD) {
    __syncthreads();
    for (int f = threadIdx.x; f < d; f += blockDim.x)
      if (dl[f] != 0.0) atomicAdd(&dhyp[4 + f], dl[f]);
  }
}

// ------------------------------------------------------------------------------------------
// gather / scatter-add
// ------------------------------------------------------------------------------------------
__global__ void gather_rows_kernel(const float* __restrict__ table, int64_t ldt, int64_t rows,
                                   const int64_t* __restrict__ ids, int64_t N, int64_t d, float* __restrict__ out,
                                   int64_t ldo) {
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < N * d; idx += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = idx / d, f = idx - i * d;
    int64_t r = ids[i];
    out[i * ldo + f] = (r >= 0 && r < rows) ? table[r * ldt + f] : 0.f;
  }
}

// Rows arrive grouped by id in practice (16 frames per MNIST digit, 72 action ids for 500 SPRITES rows), so each
// warp first folds runs of equal ids inside its 32 consecutive rows (shuffle segmented sum) and only the run
// heads issue a double atomic: the duplicate factor of the data becomes the atomic-traffic reduction factor.
__global__ void scatter_add_rows_kernel(const float* __restrict__ g, int64_t ldg, const int64_t* __restrict__ ids,
                                        int64_t N, int64_t d, int64_t rows, double* __restrict__ dtable, int64_t ldt) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t base = warp * 32; base < N; base += nwarps * 32) {
    int64_t i = base + lane;
    int64_t id = (i < N) ? ids[i] : -1;
    int64_t prev = __shfl_up_sync(0xffffffffu, id, 1);
    bool head = (lane == 0) || (prev != id);
    unsigned heads = __ballot_sync(0xffffffffu, head);
    // length of the run starting at this lane
    unsigned after = heads & ~((2u << lane) - 1u);     // heads strictly above this lane
    int next = after ? (__ffs(after) - 1) : 32;
    for (int64_t f = 0; f < d; ++f) {
      float v = (i < N) ? g[i * ldg + f] : 0.f;
      // segmented inclusive suffix-sum within runs: fold from the right
      float s = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        float t = __shfl_down_sync(0xffffffffu, s, o);
        if (lane + o < next) s += t;
      }
      if (head && id >= 0 && id < rows) atomicAdd(&dtable[id * ldt + f], (double)s);
    }
  }
}

static size_t fwd_smem(int d) {
  int dp = d | 1;
  return sizeof(float) * (2 * TILE * dp + TILE * (TILE + 1) + 4 * TILE);
}
static size_t bwd_smem(int d) {
  int dp = d | 1;
  return sizeof(float) * (2 * TILE * dp + 2 * TILE * (TILE + 1) + 4 * TILE + 4 * TILE + 4);
}

static int check_spec(int ta, int da, int tb, int db) {
  auto ok = [](int t, int d) {
    if (t >= 0 && (t & SVGP_K_ARD)) {                // ARD: the stationary factors with a length scale per feature
      t &= ~SVGP_K_ARD;
      if (t != SVGP_K_SE && !is_matern(t)) return false;
    }
    if (t < 0 || t > SVGP_K_MATERN52 || d < 0) return false;
    if (t == SVGP_K_NONE) return d == 0;
    if (t == SVGP_K_EXPSIN) return d == 1;
    return d >= 1;
  };
  return ok(ta, da) && ok(tb, db) && (da + db) >= 1 && (da + db) <= MAXD;
}
// (after check_spec) the flag moves into ard_a / ard_b, so that every comparison of ta / tb sees the base type
static Spec make_spec(int ta, int da, int tb, int db) {
  return Spec{ta & ~SVGP_K_ARD, da, tb & ~SVGP_K_ARD, db, (ta & SVGP_K_ARD) != 0, (tb & SVGP_K_ARD) != 0};
}

}  // namespace svgp

using namespace svgp;

extern "C" {

int svgp_version(void) { return 200; }
const char* svgp_last_error(void) { return svgp::last_error(); }
int svgp_device_ok(void) {
  int dev = 0;
  cudaDeviceProp p;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&p, dev) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return p.major == 10 ? 1 : 0;
}

int svgp_kernel_fwd(const float* Fx, int64_t ldx, int64_t N, const float* Fz, int64_t ldz, int64_t M, int type_a,
                    int dim_a, int type_b, int dim_b, const float* hyp, float* K, int64_t ldk, void* Kh, void* Kl,
                    int64_t ldkh, void* Kth, void* Ktl, int64_t ldkt, float* kscale, void* stream) {
  SVGP_REQUIRE(check_spec(type_a, dim_a, type_b, dim_b), "bad kernel spec");
  SVGP_REQUIRE(Fx && Fz && hyp && N >= 0 && M >= 0, "null input");
  SVGP_REQUIRE((K || Kh || Kth), "no output requested");
  SVGP_REQUIRE(!(Kh && !Kl) && !(Kth && !Ktl), "fp16 planes come in hi/lo pairs");
  SVGP_REQUIRE(!(Kh || Kth) || kscale, "fp16 planes need the kscale buffer");
  if (N == 0 || M == 0) return SVGP_OK;
  const Spec sp = make_spec(type_a, dim_a, type_b, dim_b);
  const bool ard = sp.ard_a || sp.ard_b;
  cudaStream_t st = (cudaStream_t)stream;
  if (Kh || Kth) {
    if (cudaMemsetAsync(kscale, 0, 8 * sizeof(float), st) != cudaSuccess) return check_launch("svgp_kernel_fwd(memset)");
    if (sp.ta == SVGP_K_LINEAR || sp.tb == SVGP_K_LINEAR) {
      int64_t bx = ceil_div(N, 256), bz = ceil_div(M, 256);
      if (bx > 148 * 8) bx = 148 * 8;
      if (bz > 148 * 8) bz = 148 * 8;
      feature_norm_kernel<<<(unsigned)bx, 256, 0, st>>>(Fx, ldx, N, sp, kscale, 2);
      feature_norm_kernel<<<(unsigned)bz, 256, 0, st>>>(Fz, ldz, M, sp, kscale, 4);
      int rc = check_launch("svgp_kernel_fwd(norms)");
      if (rc) return rc;
    }
  }
  int64_t ntc = ceil_div(M, TILE), ntr = ceil_div(N, TILE);
  // grid.y strides over row tiles; keep >= ~8 CTAs per SM in flight without exceeding the 65535 limit
  int64_t gy = ntr;
  int64_t cap = (148 * 16 + ntc - 1) / ntc;
  if (gy > cap) gy = cap;
  if (gy < 1) gy = 1;
  if (gy > 65535) gy = 65535;
  dim3 grid((unsigned)ntc, (unsigned)gy);
  if (!K && Kh && Kth) {
    // the tcgen05 consumers' operand format only: vectorised builder
    const bool se44 = sp.ta == SVGP_K_SE && sp.tb == SVGP_K_SE && dim_a == 4 && dim_b == 4;
    if (ard)
      kernel_fwd_planes_kernel<false, true><<<grid, THREADS, fwd_smem(dim_a + dim_b) + ARD_SMEM, st>>>(
          Fx, ldx, N, Fz, ldz, M, sp, hyp, (__half*)Kh, (__half*)Kl, ldkh, (__half*)Kth, (__half*)Ktl, ldkt, kscale);
    else if (se44)
      kernel_fwd_planes_kernel<true><<<grid, THREADS, fwd_smem(dim_a + dim_b), st>>>(
          Fx, ldx, N, Fz, ldz, M, sp, hyp, (__half*)Kh, (__half*)Kl, ldkh, (__half*)Kth, (__half*)Ktl, ldkt, kscale);
    else
      kernel_fwd_planes_kernel<false><<<grid, THREADS, fwd_smem(dim_a + dim_b), st>>>(
          Fx, ldx, N, Fz, ldz, M, sp, hyp, (__half*)Kh, (__half*)Kl, ldkh, (__half*)Kth, (__half*)Ktl, ldkt, kscale);
    return check_launch("svgp_kernel_fwd(planes)");
  }
  if (K && !Kh && !Kth && N * M <= (int64_t)1 << 26) {
    // plain fp32 K_nm of a small problem: float64 evaluation, one rounding (the tiled fp32 builder below serves the large ones)
    int64_t blocks = ceil_div(N * M, 256);
    if (blocks > 148 * 32) blocks = 148 * 32;
    if (ard)
      kernel_fwd_f64_kernel<float, true><<<(unsigned)blocks, 256, MAXD * sizeof(double), st>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, K, ldk);
    else
      kernel_fwd_f64_kernel<float><<<(unsigned)blocks, 256, 0, st>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, K, ldk);
    return check_launch("svgp_kernel_fwd(f64 evaluation)");
  }
  if (ard)
    kernel_fwd_kernel<true><<<grid, THREADS, fwd_smem(dim_a + dim_b) + ARD_SMEM, st>>>(
        Fx, ldx, N, Fz, ldz, M, sp, hyp, K, ldk, (__half*)Kh, (__half*)Kl, ldkh, (__half*)Kth, (__half*)Ktl, ldkt, kscale);
  else
    kernel_fwd_kernel<<<grid, THREADS, fwd_smem(dim_a + dim_b), st>>>(
        Fx, ldx, N, Fz, ldz, M, sp, hyp, K, ldk, (__half*)Kh, (__half*)Kl, ldkh, (__half*)Kth, (__half*)Ktl, ldkt, kscale);
  return check_launch("svgp_kernel_fwd");
}

int svgp_kernel_fwd_f64(const float* Fx, int64_t ldx, int64_t N, const float* Fz, int64_t ldz, int64_t M, int type_a, int dim_a,
                        int type_b, int dim_b, const float* hyp, double* K, int64_t ldk, void* stream) {
  SVGP_REQUIRE(check_spec(type_a, dim_a, type_b, dim_b), "bad kernel spec");
  SVGP_REQUIRE(Fx && Fz && hyp && K && N >= 0 && M >= 0 && ldk >= M, "bad argument");
  if (N == 0 || M == 0) return SVGP_OK;
  const Spec sp = make_spec(type_a, dim_a, type_b, dim_b);
  const bool ard = sp.ard_a || sp.ard_b;
  int64_t blocks = ceil_div(N * M, 256);
  if (blocks > 148 * 32) blocks = 148 * 32;
  if (ard)
    kernel_fwd_f64_kernel<double, true><<<(unsigned)blocks, 256, MAXD * sizeof(double), (cudaStream_t)stream>>>(
        Fx, ldx, N, Fz, ldz, M, sp, hyp, K, ldk);
  else
    kernel_fwd_f64_kernel<double><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, K, ldk);
  return check_launch("svgp_kernel_fwd_f64");
}

int svgp_kernel_fwd_i8(const float* Fx, int64_t ldx, int64_t N, const float* Fz, int64_t ldz, int64_t M, int type_a, int dim_a,
                       int type_b, int dim_b, const float* hyp, void* Kh, void* Kl, int64_t ldkh, void* Kr, int64_t ldkr,
                       float* rscale, void* Kc, float* cscale, float* scratch, float* kscale, void* stream) {
  SVGP_REQUIRE(check_spec(type_a, dim_a, type_b, dim_b), "bad kernel spec");
  SVGP_REQUIRE(Fx && Fz && hyp && Kh && Kl && Kr && rscale && Kc && cscale && scratch && kscale && N >= 0 && M >= 0, "null argument");
  SVGP_REQUIRE(ldkh % 8 == 0 && ldkh >= (M + 7) / 8 * 8 && ldkr % 16 == 0 && ldkr >= (M + 7) / 8 * 8, "row pitches: ldkh multiple of 8, ldkr multiple of 16, both >= M rounded up to 8");
  SVGP_REQUIRE((((uintptr_t)Kh | (uintptr_t)Kl | (uintptr_t)Kr | (uintptr_t)Kc) & 15) == 0, "planes need 16-byte alignment");
  if (N == 0 || M == 0) return SVGP_OK;
  const Spec sp = make_spec(type_a, dim_a, type_b, dim_b);
  const bool ard = sp.ard_a || sp.ard_b;
  cudaStream_t st = (cudaStream_t)stream;
  float* rmax = scratch;
  float* cmax = scratch + N;
  if (cudaMemsetAsync(kscale, 0, 8 * sizeof(float), st) != cudaSuccess) return check_launch("svgp_kernel_fwd_i8(memset)");
  if (cudaMemsetAsync(scratch, 0, (N + M) * sizeof(float), st) != cudaSuccess) return check_launch("svgp_kernel_fwd_i8(memset)");
  // the last 128-datapoint block of Kc and the pad columns of Kr / Kh / Kl must be zeros (TMA boxes read them)
  const int64_t nb128 = (N + 127) / 128;
  if (N % 128) {
    for (int s = 0; s < 4; ++s)
      if (cudaMemsetAsync((int8_t*)Kc + (s * nb128 + (nb128 - 1)) * M * 128, 0, M * 128, st) != cudaSuccess) return check_launch("svgp_kernel_fwd_i8(memset)");
  }
  if (ldkr != M && cudaMemsetAsync(Kr, 0, 4 * N * ldkr, st) != cudaSuccess) return check_launch("svgp_kernel_fwd_i8(memset)");
  if (ldkh != M) {
    if (cudaMemsetAsync(Kh, 0, N * ldkh * 2, st) != cudaSuccess || cudaMemsetAsync(Kl, 0, N * ldkh * 2, st) != cudaSuccess)
      return check_launch("svgp_kernel_fwd_i8(memset)");
  }
  if (sp.ta == SVGP_K_LINEAR || sp.tb == SVGP_K_LINEAR) {
    int64_t bx = ceil_div(N, 256), bz = ceil_div(M, 256);
    if (bx > 148 * 8) bx = 148 * 8;
    if (bz > 148 * 8) bz = 148 * 8;
    feature_norm_kernel<<<(unsigned)bx, 256, 0, st>>>(Fx, ldx, N, sp, kscale, 2);
    feature_norm_kernel<<<(unsigned)bz, 256, 0, st>>>(Fz, ldz, M, sp, kscale, 4);
    int rc = check_launch("svgp_kernel_fwd_i8(norms)");
    if (rc) return rc;
  }
  int64_t ntc = ceil_div(M, TILE), ntr = ceil_div(N, TILE);
  int64_t gy = ntr;
  int64_t cap = (148 * 16 + ntc - 1) / ntc;
  if (gy > cap) gy = cap;
  if (gy < 1) gy = 1;
  if (gy > 65535) gy = 65535;
  dim3 grid((unsigned)ntc, (unsigned)gy);
  const bool se44 = sp.ta == SVGP_K_SE && sp.tb == SVGP_K_SE && dim_a == 4 && dim_b == 4;
  const size_t sm = fwd_smem(dim_a + dim_b) + (ard ? ARD_SMEM : 0);
#define SVGP_LAUNCH_I8(SE, MX, ARD)                                                                                               \
  kernel_fwd_i8_kernel<SE, MX, ARD><<<grid, THREADS, sm, st>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, (__half*)Kh, (__half*)Kl, ldkh,   \
                                                               (int8_t*)Kr, ldkr, rscale, (int8_t*)Kc, cscale, rmax, cmax, kscale)
  if (se44 && ard) { SVGP_LAUNCH_I8(true, true, true); SVGP_LAUNCH_I8(true, false, true); }
  else if (se44) { SVGP_LAUNCH_I8(true, true, false); SVGP_LAUNCH_I8(true, false, false); }
  else if (ard) { SVGP_LAUNCH_I8(false, true, true); SVGP_LAUNCH_I8(false, false, true); }
  else { SVGP_LAUNCH_I8(false, true, false); SVGP_LAUNCH_I8(false, false, false); }
#undef SVGP_LAUNCH_I8
  return check_launch("svgp_kernel_fwd_i8");
}

int svgp_kernel_bwd(const float* Fx, int64_t ldx, int64_t N, const float* Fz, int64_t ldz, int64_t M, int type_a,
                    int dim_a, int type_b, int dim_b, const float* hyp, const float* G, int64_t ldg, float* dFx,
                    double* dFz, double* dhyp, void* stream) {
  SVGP_REQUIRE(check_spec(type_a, dim_a, type_b, dim_b), "bad kernel spec");
  SVGP_REQUIRE(Fx && Fz && hyp && G && N >= 0 && M >= 0, "null input");
  if (N == 0 || M == 0) return SVGP_OK;
  const Spec sp = make_spec(type_a, dim_a, type_b, dim_b);
  const bool ard = sp.ard_a || sp.ard_b;
  size_t sm = bwd_smem(dim_a + dim_b) + (ard ? ARD_SMEM : 0);
  cudaStream_t st = (cudaStream_t)stream;
  int64_t ntc = ceil_div(M, TILE), ntr = ceil_div(N, TILE);
  if (dFx) {
    int64_t gx = ntr < 148 * 8 ? ntr : 148 * 8;
    if (ard)
      kernel_bwd_kernel<true, false, true><<<(unsigned)gx, THREADS, sm, st>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, G, ldg, dFx, nullptr, nullptr);
    else
      kernel_bwd_kernel<true><<<(unsigned)gx, THREADS, sm, st>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, G, ldg, dFx, nullptr, nullptr);
    int rc = check_launch("svgp_kernel_bwd(x)");
    if (rc) return rc;
  }
  if (dFz) {
    SVGP_REQUIRE(dhyp != nullptr, "dhyp required with dFz");
    int64_t gy = (148 * 8 + ntc - 1) / ntc;
    if (gy > ntr) gy = ntr;
    if (gy < 1) gy = 1;
    dim3 grid((unsigned)(ntc < 65535 ? ntc : 65535), (unsigned)gy);
    const bool se44 = sp.ta == SVGP_K_SE && sp.tb == SVGP_K_SE && dim_a == 4 && dim_b == 4 && ntc <= 65535 &&
                      !getenv("SVGP_K1_BWD_GENERIC");
    const bool matern = is_matern(sp.ta) || is_matern(sp.tb);
    if (se44 && ard)
      kernel_bwd_z_se44_kernel<true><<<grid, THREADS, 0, st>>>(Fx, ldx, N, Fz, ldz, M, hyp, G, ldg, dFz, dhyp, sp);
    else if (se44)
      kernel_bwd_z_se44_kernel<<<grid, THREADS, 0, st>>>(Fx, ldx, N, Fz, ldz, M, hyp, G, ldg, dFz, dhyp, sp);
    else if (matern && ard)
      kernel_bwd_kernel<false, true, true><<<grid, THREADS, sm, st>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, G, ldg, nullptr, dFz, dhyp);
    else if (matern)
      kernel_bwd_kernel<false, true><<<grid, THREADS, sm, st>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, G, ldg, nullptr, dFz, dhyp);
    else if (ard)
      kernel_bwd_kernel<false, false, true><<<grid, THREADS, sm, st>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, G, ldg, nullptr, dFz, dhyp);
    else
      kernel_bwd_kernel<false><<<grid, THREADS, sm, st>>>(Fx, ldx, N, Fz, ldz, M, sp, hyp, G, ldg, nullptr, dFz, dhyp);
    int rc = check_launch("svgp_kernel_bwd(z)");
    if (rc) return rc;
  }
  return SVGP_OK;
}

int svgp_kernel_diag_fwd(const float* Fx, int64_t ldx, const float* Fy, int64_t ldy, int64_t N, int type_a, int dim_a,
                         int type_b, int dim_b, const float* hyp, float* kd, void* stream) {
  SVGP_REQUIRE(check_spec(type_a, dim_a, type_b, dim_b), "bad kernel spec");
  SVGP_REQUIRE(Fx && Fy && hyp && kd && N >= 0, "null input");
  if (N == 0) return SVGP_OK;
  const Spec sp = make_spec(type_a, dim_a, type_b, dim_b);
  const bool ard = sp.ard_a || sp.ard_b;
  int64_t blocks = ceil_div(N, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (ard)
    kernel_diag_fwd_kernel<true><<<(unsigned)blocks, 256, ARD_SMEM, (cudaStream_t)stream>>>(Fx, ldx, Fy, ldy, N, sp, hyp, kd);
  else
    kernel_diag_fwd_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(Fx, ldx, Fy, ldy, N, sp, hyp, kd);
  return check_launch("svgp_kernel_diag_fwd");
}

int svgp_kernel_diag_bwd(const float* Fx, int64_t ldx, const float* Fy, int64_t ldy, int64_t N, int type_a, int dim_a,
                         int type_b, int dim_b, const float* hyp, const float* g, float* dFx, float* dFy, double* dhyp,
                         void* stream) {
  SVGP_REQUIRE(check_spec(type_a, dim_a, type_b, dim_b), "bad kernel spec");
  SVGP_REQUIRE(Fx && Fy && hyp && g && dFx && dFy && dhyp && N >= 0, "null input");
  if (N == 0) return SVGP_OK;
  const Spec sp = make_spec(type_a, dim_a, type_b, dim_b);
  const bool ard = sp.ard_a || sp.ard_b;
  int64_t blocks = ceil_div(N, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (ard)
    kernel_diag_bwd_kernel<true><<<(unsigned)blocks, 256, ARD_SMEM, (cudaStream_t)stream>>>(Fx, ldx, Fy, ldy, N, sp, hyp, g, dFx,
                                                                                          dFy, dhyp);
  else
    kernel_diag_bwd_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(Fx, ldx, Fy, ldy, N, sp, hyp, g, dFx, dFy, dhyp);
  return check_launch("svgp_kernel_diag_bwd");
}

int svgp_gather_rows(const float* table, int64_t ldt, int64_t rows, const int64_t* ids, int64_t N, int64_t d, float* out,
                     int64_t ldo, void* stream) {
  SVGP_REQUIRE(table && ids && out && N >= 0 && d >= 1 && rows >= 1, "bad argument");
  if (N == 0) return SVGP_OK;
  int64_t blocks = ceil_div(N * d, 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  gather_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(table, ldt, rows, ids, N, d, out, ldo);
  return check_launch("svgp_gather_rows");
}

int svgp_scatter_add_rows(const float* g, int64_t ldg, const int64_t* ids, int64_t N, int64_t d, int64_t rows,
                          double* dtable, int64_t ldt, void* stream) {
  SVGP_REQUIRE(g && ids && dtable && N >= 0 && d >= 1 && rows >= 1, "bad argument");
  if (N == 0) return SVGP_OK;
  int64_t blocks = ceil_div(N, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  scatter_add_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(g, ldg, ids, N, d, rows, dtable, ldt);
  return check_launch("svgp_scatter_add_rows");
}

}  // extern "C"
