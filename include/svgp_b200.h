/*
 * svgp_b200.h -- C ABI of libsvgp_b200.so: the sm_100a kernels behind the SVGP hot path
 * of ratschlab/SVGP-VAE (the Hensman-style SVGP object in SVGPVAE_model.py).
 *
 * The reference has no FFI: its boundary is a duck-typed Python object (mainSVGP /
 * mnistSVGP / spritesSVGP / SVGP) whose methods expand into stock TensorFlow ops.  Every
 * entry point below replaces one such op chain; the "replaces" line cites it
 * (file:line in the reference tree).  svgp_vae_b200/_lib.py binds exactly these symbols
 * with ctypes; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless it says "host"; matrices are row-major with
 *     an explicit leading dimension (in elements); batches use an element stride
 *   - the caller (PyTorch) allocates all outputs and workspaces; the library never
 *     allocates or frees device memory and keeps no mutable global state except the
 *     thread-local last-error string
 *   - `stream` is a cudaStream_t passed as void*; calls on distinct streams are independent
 *   - return 0 on success; SVGP_ERR_ARG (-1) bad argument; SVGP_ERR_CUDA (-2) CUDA runtime
 *     error (text via svgp_last_error()); SVGP_ERR_UNSUPPORTED (-4) shape not handled by
 *     the requested implementation.  A non-positive-definite pivot in svgp_chol_f64 is
 *     reported on the device: status[b] = 1 + (failing column), never as NaN-propagation only.
 *   - there is no CPU fallback anywhere behind this header.
 */
#ifndef SVGP_B200_H_
#define SVGP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVGP_OK 0
#define SVGP_ERR_ARG (-1)
#define SVGP_ERR_CUDA (-2)
#define SVGP_ERR_UNSUPPORTED (-4)

/* factor kernels of the two-block product kernel  k(x,z) = kA(xA,zA) * kB(xB,zB)            */
#define SVGP_K_NONE 0   /* factor == 1                                                        */
#define SVGP_K_SE 1     /* tfk.ExponentiatedQuadratic: s^2 exp(-|x-z|^2 / (2 l^2))             */
#define SVGP_K_EXPSIN 2 /* tfk.ExpSinSquared, period 2*pi: s^2 exp(-2 sum sin^2((x-z)/2)/l^2)  */
#define SVGP_K_LINEAR 3 /* tfk.Linear(): x . z                                                */
#define SVGP_K_COSINE 4 /* Linear divided by |x||z|  (K_obj_normalize)                        */
/* Matern factors, tfk.MaternOneHalf / MaternThreeHalves / MaternFiveHalves: r = |x-z| over the block, u = c r / l   */
#define SVGP_K_MATERN12 5 /* s^2 exp(-u), c = 1; its gradient in x and z is taken as 0 at r = 0 (symmetric subgradient) */
#define SVGP_K_MATERN32 6 /* s^2 (1 + u) exp(-u), c = sqrt(3)                                                     */
#define SVGP_K_MATERN52 7 /* s^2 (1 + u + u^2/3) exp(-u), c = sqrt(5)                                             */
/* automatic relevance determination: OR'ed into SVGP_K_SE or a Matern code, the factor's distance becomes
 * r^2 = sum_f ((x_f - z_f) / l_f)^2 with one length scale l_f per feature column of its block (hyp layout below)      */
#define SVGP_K_ARD 16

/* implementation selector for the GEMM-class entry points */
#define SVGP_IMPL_AUTO 0
#define SVGP_IMPL_SIMT 1 /* fp32 CUDA-core tiles, any shape                                   */
#define SVGP_IMPL_TC 2   /* tcgen05 / TMEM / TMA, fp32-emulating 3 x FP16 split operands          */
#define SVGP_IMPL_TC_I8 3 /* tcgen05 kind::i8 on base-256 digit planes: exact int32 accumulation (svgp_syrk only;
                             the scaled GEMM has its own entry point svgp_scaled_gemm_i8)            */
#define SVGP_IMPL_TC_I8_O4 5 /* the same with thirteen pairs: the three pairs of order 4 as well, as a second set of work items on the
                                CTA-pair kernel (full form only: both triangles; otherwise as SVGP_IMPL_TC_I8).  The FORWARD SYRK
                                at M > 2048, where the truncation after order 3 holds the inducing-point gradient at 1e-4          */
#define SVGP_IMPL_TC_I8_D3 4 /* the same with the three leading digits of both operands (8 instead of 10 digit-plane
                                pairs): enough for the ADJOINT SYRK dS_l = sum_i dq_il k_i k_i^T, not for the forward one  */

int svgp_version(void);
const char* svgp_last_error(void); /* host string, thread-local */
int svgp_device_ok(void);          /* 1 if the current device is compute capability 10.x      */

/* ---------------------------------------------------------------------------------------
 * K1  kernel-matrix builder
 * replaces: mnistSVGP.kernel_matrix SVGPVAE_model.py:427-476, spritesSVGP.kernel_matrix
 *           :550-600, ball kernel.matrix :81-86/:152-157 and the tfp.math.psd_kernels
 *           .matrix/.apply calls under them.
 * Fx (N x d) / Fz (M x d) are dense fp32 feature rows [block A | block B], d = dim_a+dim_b.
 * hyp = device float[4] = {amplitude_a, length_a, amplitude_b, length_b} (unused entries 1).
 * With SVGP_K_ARD on either factor hyp = device float[4 + dim_a + dim_b]: hyp[4 + f] is the length scale of feature
 * column f of the [A | B] row.  An ARD block reads its l_f there and not its isotropic slot (hyp[1] / hyp[3]); an
 * isotropic block reads its slot and not its hyp[4 + f] (callers put 1 there).  The type codes may carry the flag in
 * every K1 entry point below.
 * Outputs (each group may be NULL):
 *   K   (N x M fp32, ld = ldk)                         plain matrix for the SIMT consumers; requested alone and with
 *                                                      N M <= 2^26 it is the float64 evaluation rounded once to fp32
 *   Kh, Kl   (N x M fp16 planes, ld = ldkh elements)   operand planes of the tcgen05 consumers:
 *   Kth, Ktl (transposed planes, datapoint-blocked:    value * scale = fp16 hi + fp16 lo (22 bits),
 *            element (m, n) at [n / 64] * ldkt + m * 64 + n % 64, ldkt >= 64 M; ceil(N / 64) blocks, the
 *            datapoints past N in the last block are written as zeros)
 *            with scale = the power of two that puts the kernel's upper bound (amplitudes, max
 *            feature norms) just below 2^14; kscale (device float[8], required with the planes)
 *            receives {scale, 1/scale, ...scratch}.  Rows/columns beyond N / M up to ld stay untouched.
 * ------------------------------------------------------------------------------------- */
int svgp_kernel_fwd(const float* Fx, int64_t ldx, int64_t N, const float* Fz, int64_t ldz, int64_t M,
                    int type_a, int dim_a, int type_b, int dim_b, const float* hyp,
                    float* K, int64_t ldk, void* Kh, void* Kl, int64_t ldkh, void* Kth, void* Ktl,
                    int64_t ldkt, float* kscale, void* stream);

/* adjoint of svgp_kernel_fwd.  G (N x M) is dObjective/dK.  dFx (N x d) is overwritten;
 * dFz (M x d, double) and dhyp (double[4], double[4 + dim_a + dim_b] for ARD specs: slot 4 + f takes dObjective/dl_f,
 * and the slots hyp does not read get exactly 0) are ACCUMULATED into (caller zeroes them).  The same for
 * svgp_kernel_diag_bwd.
 * replaces: tf.gradients through kernel_matrix (MNIST_experiment.py:202-208).                */
int svgp_kernel_bwd(const float* Fx, int64_t ldx, int64_t N, const float* Fz, int64_t ldz, int64_t M,
                    int type_a, int dim_a, int type_b, int dim_b, const float* hyp,
                    const float* G, int64_t ldg, float* dFx, double* dFz, double* dhyp, void* stream);

/* element-wise kernel .apply: kd[i] = k(Fx[i], Fy[i])  (diag_only=True, :458-467/:572-583)   */
int svgp_kernel_diag_fwd(const float* Fx, int64_t ldx, const float* Fy, int64_t ldy, int64_t N,
                         int type_a, int dim_a, int type_b, int dim_b, const float* hyp, float* kd,
                         void* stream);
int svgp_kernel_diag_bwd(const float* Fx, int64_t ldx, const float* Fy, int64_t ldy, int64_t N,
                         int type_a, int dim_a, int type_b, int dim_b, const float* hyp,
                         const float* g, float* dFx, float* dFy, double* dhyp, void* stream);

/* embedding gather / scatter-add (tf.gather :451,455,565,570 and its IndexedSlices gradient)
 * out[i, :] = table[ids[i], :];  dtable[ids[i], :] += g[i, :]  (dtable double, caller zeroes) */
int svgp_gather_rows(const float* table, int64_t ldt, int64_t rows, const int64_t* ids, int64_t N,
                     int64_t d, float* out, int64_t ldo, void* stream);
int svgp_scatter_add_rows(const float* g, int64_t ldg, const int64_t* ids, int64_t N, int64_t d,
                          int64_t rows, double* dtable, int64_t ldt, void* stream);

/* ---------------------------------------------------------------------------------------
 * The operand "Kop" of the GEMM-class calls is K_nm (N x M).  SIMT: K (fp32), the planes NULL.
 * TC: the four fp16 planes and kscale written by svgp_kernel_fwd (K may be NULL).
 * ------------------------------------------------------------------------------------- */
typedef struct svgp_kop {
  const float* K;      /* N x M fp32, ld = ldk (SIMT operand; may be NULL when the planes are given) */
  const void* Kh;      /* N x M fp16 hi plane, ld = ldkh                                            */
  const void* Kl;      /* N x M fp16 lo plane                                                       */
  const void* Kth;     /* fp16 hi plane of the transpose, blocked [ceil(N/64)][M][64], block stride ldkt */
  const void* Ktl;     /* fp16 lo plane, same layout                                                */
  const float* kscale; /* device float[8]: {scale, 1/scale, feature norms..., [6] = 1 if K >= 0 element-wise} */
  int64_t N, M, ldk, ldkh, ldkt;
  /* int8 digit planes of svgp_kernel_fwd_i8 (all NULL / 0 when absent): the operands of the exact integer products  */
  const void* Kr;       /* [4][N][ldkr] balanced base-256 digits of rint(K[i, m] / rscale[i]), most significant first */
  const float* rscale;  /* [N]                                                                                        */
  const void* Kc;       /* [4][ceil(N/128)][M][128]: digits of rint(K[n, m] / cscale[m]) at [n / 128][m][n % 128]       */
  const float* cscale;  /* [M]                                                                                        */
  int64_t ldkr;         /* row pitch of Kr in bytes, multiple of 16, >= M                                             */
} svgp_kop;

/* the same kernel matrix in float64 arithmetic and storage (fp32 features): K_mm of the float64 M x M stage.  An fp32
 * evaluation carries ~5e-7 of relative error per entry (rounding of the exponent's argument); the ill-conditioned
 * M x M stage amplifies that into 1e-4 of the inducing-point gradient at M = 2048.                                   */
int svgp_kernel_fwd_f64(const float* Fx, int64_t ldx, int64_t N, const float* Fz, int64_t ldz, int64_t M, int type_a,
                        int dim_a, int type_b, int dim_b, const float* hyp, double* K, int64_t ldk, void* stream);

/* K1 for the exact-accumulation tensor-core products (tcgen05.mma.kind::i8, int32 accumulators): every entry of K_nm
 * becomes a 32-bit fixed-point integer against the largest |entry| of its row (Kr: products that reduce over the inducing
 * points) / of its column (Kc: the SYRK, which reduces over the datapoints), written as four balanced base-256 digits in
 * four int8 planes, from kernel values evaluated in float64 and rounded once to fp32; plus the fp16 hi/lo row planes and kscale of svgp_kernel_fwd
 * for the remaining fp16 consumers (no transposed fp16 planes).  Two passes over the tiles (maxima, then write).
 * scratch: float[N + M].  Rows n >= N of the last 128-datapoint block of Kc and the pad columns of Kr / Kh / Kl are zero.
 * replaces: the same reference lines as svgp_kernel_fwd.                                                              */
int64_t svgp_i8_ldkr(int64_t M);  /* (M + 15) / 16 * 16 */
int64_t svgp_i8_nblk(int64_t N);  /* (N + 127) / 128    */
int svgp_kernel_fwd_i8(const float* Fx, int64_t ldx, int64_t N, const float* Fz, int64_t ldz, int64_t M, int type_a,
                       int dim_a, int type_b, int dim_b, const float* hyp, void* Kh, void* Kl, int64_t ldkh, void* Kr,
                       int64_t ldkr, float* rscale, void* Kc, float* cscale, float* scratch, float* kscale, void* stream);

/* nslices (3 or 4) digit planes of a float64 matrix with one scale per ROW: x[r, c] ~= scale[r] * sum_s d_s[r, c] 256^(S-1-s);
 * planes[s][r][c] (row pitch ldp bytes, multiple of 16; columns >= cols zeroed).  A batch of matrices is its row-stack. */
int svgp_split_i8(const double* x, int64_t nrows, int64_t cols, int64_t ldx, int nslices, void* planes, int64_t ldp,
                  float* scale, void* stream);

/* per-matrix fp16 operand planes of a (nb x rows x cols) float64 batch:  x * s_b = hi + lo with
 * s_b = 2^(14 - e_b), max|x_b| = m 2^e_b (m in [0.5,1));  inv_scale: device float[2*nb] =
 * {1/s_b ..., scratch...}.  replaces nothing in the reference: it is the operand format of the
 * tensor-core calls below (the 3 x FP16 split emulating fp32 products).                        */
int svgp_split_f16(const double* x, int64_t nb, int64_t count, void* hi, void* lo, float* inv_scale,
                   void* stream);

/* K2  batched weighted SYRK   A[l] = sum_i W[i,l] k_i k_i^T   (L x M x M, double, ACCUMULATED:
 * caller zeroes; both triangles written).  W is N x L fp32 (any sign).  The TC path needs the
 * workspace ws (float[svgp_syrk_ws_floats(N, M, L)]): it holds the channel-major copy of W scaled
 * per channel by a power of two (|w s_l| <= 1, so that w * k stays inside fp16 range), 1/s_l, and
 * the lock words guarding the float64 tiles of A (datapoints are walked in L2-sized super-chunks;
 * CTAs working on different super-chunks of one tile add into it under a spin lock).
 * chunk_rows: datapoints per TMEM accumulation chain (0 = default: 512 on the TC path, 2048 on the SIMT path).
 * The tensor core accumulates with truncation; chains whose terms all have one sign (every weight of a channel
 * >= 0 and kop->kscale[6] != 0, i.e. an element-wise non-negative kernel as recorded by svgp_kernel_fwd) get their
 * known relative loss of 0.666 n 2^-24 (n MMAs per chain, measured) added back per chunk.
 * replaces: K_mn (K_nm * 1/sigma^2) SVGPVAE_model.py:328-330 (:160 for the ball) and, as the
 * adjoint of svgp_rowquad, the (b,m,m) trace pattern :286-294.                               */
/* impl = SVGP_IMPL_TC_I8 (needs kop->Kc, cscale): the weighted operand w[n, l] K[n, a] is rebuilt per channel in shared
 * memory as a 32-bit fixed-point integer (4 digit planes) against the 32-bit K^T planes, the 10 digit-plane pairs of
 * order <= 3 run as integer MMAs over windows of <= 16384 datapoints and the exactly recombined window sums are added
 * into A with double atomics: no rounding inside the contraction (the summation ORDER of the window sums in float64 is
 * not fixed).  Same workspace size function.                                                                        */
int64_t svgp_syrk_ws_floats(int64_t N, int64_t M, int64_t L);
int svgp_syrk(const svgp_kop* kop, const float* W, int64_t ldw, int64_t L, double* A, int impl,
              int64_t chunk_rows, float* ws, void* stream);

/* V[l, :] += sum_i X[i,l] k_i          (L x M double, accumulated)  -- K_mn (p*y), :333-334   */
int svgp_gemm_tn(const svgp_kop* kop, const float* X, int64_t ldx, int64_t L, double* V, void* stream);

/* out[i,l] = k_i . Wm[l,:]             (N x L fp32)   -- K_xm (S K_mn p y), :332-334; :264-265 */
int svgp_gemm_nn(const svgp_kop* kop, const float* Wm, int64_t ldwm, int64_t L, float* out,
                 int64_t ldo, void* stream);

/* the same product on the tensor cores: Wm given as the fp16 planes + 1/scale of svgp_split_f16(Wm, nb = 1,
 * count = L * M); needs the fp16 planes of K_nm in kop.                                        */
int svgp_gemm_nn_tc(const svgp_kop* kop, const void* Wm_hi, const void* Wm_lo, const float* Wm_inv, int64_t L,
                    float* out, int64_t ldo, void* stream);

/* K4  row-wise quadratic forms  q[i,l] = k_i^T S_l k_i  (N x L fp32).
 * S (L x M x M, symmetric): SIMT takes the float64 matrices themselves (S_hi = const double*, S_lo and
 * S_inv NULL: fp32 K entries times float64 S entries, float64 accumulation); TC takes the fp16
 * planes + inv_scale of svgp_split_f16.  If `tri` != 0 the planes hold a lower-triangular factor
 * Rinv_l instead and q[i,l] = |Rinv_l k_i|^2 (half the work, a sum of squares: no cancellation).
 * L may be 1 with N x 1 output (h_i = k^T Kinv k).
 * replaces: diag_part(K_xm Sigma_l^-1 K_mx), diag_part(K_xm K_mm^-1 K_mx) :336-337, :284.    */
int svgp_rowquad(const svgp_kop* kop, const void* S_hi, const void* S_lo, const float* S_inv, int64_t L,
                 int tri, float* q, int64_t ldq, int impl, void* stream);

/* out[i, :] (+)= sum_l W[i,l] * (G_l k_i)     (N x M fp32), G (L x M x M symmetric) as planes
 * (same convention as svgp_rowquad).  accumulate != 0 adds to `out`.  If dots != NULL also
 * dots[i,l] += k_i^T G_l k_i for l < ndot (N x ndot fp32, caller zeroes) from the same products.
 * This is dObjective/dK_nm through svgp_syrk (W = p, G = dA+dA^T; the dots are dObjective/dp) and
 * through svgp_rowquad (W = 2 dq, G = S).  replaces: tf.gradients through :328-337.           */
int svgp_scaled_gemm(const svgp_kop* kop, const float* W, int64_t ldw, const void* G_hi, const void* G_lo,
                     const float* G_inv, int64_t L, float* out, int64_t ldo, int accumulate, float* dots,
                     int64_t lddots, int64_t ndot, int impl, void* stream);

/* svgp_scaled_gemm on the integer tensor-core path: G as the 4 digit planes + per-row scales of
 * svgp_split_i8(G viewed as (L * Mc) x M, nslices = 4, ldp = ldg) -- the matrices must be symmetric or given
 * transposed (row c of G_l multiplies k_i into output column c); K_nm as kop->Kr / rscale.  Mc = rows of each G_l
 * (M for the dK_nm product; any value for a skinny product such as K_nm Wm^T with L = 1, W = NULL).  Exact integer accumulation
 * of the 10 digit-plane pairs of order <= 3, one fp32 rounding when an accumulator tile leaves TMEM, fp32 running sums over
 * the L matrices.  nfull: the first nfull matrices use all 10 pairs, the rest the 8 pairs of the three leading digits of both
 * operands (the S_l - Kinv family of pass D tolerates that, the dA_l + dA_l^T family does not; pass L for full precision).
 * K_bias (2 x N) / G_bias (2 x L * Mc): svgp_i8_pair_bias of kop->Kr and of G_planes, or both NULL.  With them the expectation
 * of the digit-plane pairs that are not multiplied enters every entry before it is rounded: the digits of the format have mean
 * -1/2, which leaves a deviation of ~1e-9 of an entry but of ONE sign over the whole N x M product -- visible only in sums over
 * all of it that cancel 1e5-fold (the kernel hyper-parameter gradients at M = 4096).                                          */
int svgp_scaled_gemm_i8(const svgp_kop* kop, const float* W, int64_t ldw, const void* G_planes, int64_t ldg,
                        const float* G_scale, int64_t L, int64_t Mc, float* out, int64_t ldo, int accumulate,
                        float* dots, int64_t lddots, int64_t ndot, int64_t nfull, const float* K_bias, const float* G_bias,
                        void* stream);

/* Expected value of the dropped digit-plane pairs, one operand's share, from the digit sums of its four int8 planes
 * (planes[s][r][c], pitch ld bytes, planes nrows * ld bytes apart; pad columns zero): bias[0][r] = -(S_1 + S_2 + S_3)[r] / 512
 * for products with ten pairs, bias[1][r] = bias[0][r] - S_0[r] / 2 for products with eight (three leading digits).           */
int svgp_i8_pair_bias(const void* planes, int64_t nrows, int64_t ld, float* bias, void* stream);

/* out (N x M) (+)= W (N x L) @ V (L x M), all fp32 -- rank-L part of dK_nm (p_m, mean terms)  */
int svgp_gemm_f32(int64_t Mr, int64_t Nc, int64_t Kd, const float* A, int64_t lda, const float* B,
                  int64_t ldb, float* C, int64_t ldc, int accumulate, void* stream);

/* ---------------------------------------------------------------------------------------
 * K3  batched float64 factorisations over the latent channels
 * replaces: tf.linalg.cholesky :270-274 / :129-130, tf.linalg.inv :239,319,331 / :83,154,161
 * ------------------------------------------------------------------------------------- */
/* in-place lower Cholesky of `batch` SPD matrices (M x M, ld, stride); the strict upper
 * triangle is zeroed.  status[b] = 0 ok, 1 + column of the first non-positive pivot.
 * ws: double[batch * 32 * 32] scratch.                                                        */
int svgp_chol_f64(double* A, int64_t M, int64_t ld, int64_t stride, int64_t batch, int* status,
                  double* ws, void* stream);
/* Linv = inverse of the lower-triangular factor (strict upper triangle of Linv zeroed)        */
int svgp_trinv_f64(const double* Lf, double* Linv, int64_t M, int64_t ld, int64_t stride,
                   int64_t batch, double* ws, void* stream);
/* S = T^T T for lower-triangular T (both triangles of S written): X^-1 = Linv^T Linv after the two calls above.
 * Skips the structurally zero part of the reduction (about a quarter of a full product).      */
int svgp_ltl_f64(const double* T, double* S, int64_t M, int64_t ld, int64_t stride, int64_t batch, void* stream);
/* C[b] = alpha op(A[b]) op(B[b]) + beta C[b]; row-major, trans flags 0/1, stride 0 broadcasts */
int svgp_gemm_f64(int transA, int transB, int64_t Mr, int64_t Nc, int64_t Kd, double alpha,
                  const double* A, int64_t lda, int64_t strideA, const double* B, int64_t ldb,
                  int64_t strideB, double beta, double* C, int64_t ldc, int64_t strideC, int64_t batch,
                  void* stream);

/* ---------------------------------------------------------------------------------------
 * K4  fused row terms
 * ------------------------------------------------------------------------------------- */
/* p = reciprocal_no_nan(noise), py = p*y and the per-channel sums
 * sums[0,l] = sum_i p kappa_i, sums[1,l] = sum_i p y^2, sums[2,l] = sum_i log noise
 * (double[3*L], accumulated).   replaces :282, :297-299 (row sums), utils.py:498-502          */
int svgp_rowstats_fwd(const float* y, const float* noise, const float* kappa, int64_t N, int64_t L,
                      float* p, float* py, double* sums, void* stream);
/* p_v = kappa - h + q1 (optionally clipped to [lo,hi], SVGPVAE_model.py:891-892) written
 * over q1; clipsum[l] += sum_i p_il (p_v_clipped - p_v_raw).                                  */
int svgp_predictive_fwd(const float* kappa, const float* h, float* q1_pv, const float* p, int64_t N,
                        int64_t L, int clip, float clip_lo, float clip_hi, double* clipsum,
                        unsigned char* clipmask, void* stream);

/* Backward of the row terms, fused (one pass over the N x L tensors each).
 * pre  (before the adjoint SYRK): G_q1 = dObjective/dq1 (g_pv; on clipped entries 0.5 gce p, SVGPVAE_model.py:891-892),
 *      the stacked row weights of the adjoint products Wst = [p | 2 G_q1] and PYst = [p y | g_pm] (N x 2L each),
 *      G_p_clip = -0.5 gce (pv - pv_raw) when clipping, G_kappa[i] = sum_l G_q1.  clipmask == NULL: no clip branch
 *      (pv, kappa, h, q1raw, gce, G_p_clip unused); g_pv may be NULL (zero upstream).
 * post (after the adjoint products): G_y, G_noise (through p = reciprocal_no_nan(noise) and log noise) and
 *      G_kappa[i] += sum_l p gs0 from kGk = k^T (dA + dA^T) k, G_py = K_nm dV and gsums (3 x L, double) = the adjoints
 *      of the three row sums of svgp_rowstats_fwd.
 * replaces: tf.gradients through SVGPVAE_model.py:282-299, :332-337 and utils.py:498-502 (row-local part).            */
int svgp_rowterms_bwd_pre(const float* g_pv, const float* g_pm, const float* p, const float* y, const unsigned char* clipmask,
                          const float* pv, const float* kappa, const float* h, const float* q1raw, const float* gce, int64_t N,
                          int64_t L, float* G_q1, float* Wst, float* PYst, float* G_p_clip, float* G_kappa, void* stream);
int svgp_rowterms_bwd_post(const float* y, const float* noise, const float* p, const float* kappa, const float* kGk,
                           const float* G_py, const double* gsums, const float* G_p_clip, int64_t N, int64_t L, float* G_y,
                           float* G_noise, float* G_kappa, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SVGP_B200_H_ */
