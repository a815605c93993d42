/* mfm_b200 — C ABI of the B200-native Markovian-Flow-Matching hot path.
 *
 * Drop-in boundary for the data-parallel hot path of albcab/mfm.  The reference has no FFI of its
 * own (it is pure Python/JAX); each entry point below replaces the jitted JAX computation cited
 * next to it (paths relative to the reference repository).  A maintainer binds these from JAX
 * with jax.ffi / from Python with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - all array pointers are DEVICE pointers (float32 / uint32 / uint8), row-major [N, d];
 *   - keys are raw jax.random legacy keys: uint32[2] (or uint32[N,2]) in device memory;
 *   - every call enqueues work on `stream` and returns 0 on success or a negative MFM_ERR_* code;
 *     mfm_last_error() returns a description.  Nothing is allocated inside a call: scratch comes
 *     from the caller-provided workspace whose size the matching *_workspace_bytes() reports;
 *   - mfm_ode_* / mfm_flow_*_step run a data-dependent loop (adaptive Runge-Kutta).  For small ensembles (n * d <= 4 Mi
 *     elements; MFM_ODE_GRAPH=0|1 forces either way) the loop is a CUDA-graph WHILE node and the call is asynchronous like all
 *     others; for large ones the host polls a device counter once per iteration, i.e. the call synchronises `stream`.
 *   - arithmetic type: float32 everywhere; dense contractions emulate fp32 products on the tensor cores (operands split
 *     into two 16-bit parts, three fp16 passes - the weight gradients too; 3xTF32 for narrow / unaligned layers - with fp32 accumulation):
 *     fp32-accurate results.
 */
#ifndef MFM_B200_H
#define MFM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* mfm_stream_t; /* == cudaStream_t */

enum { MFM_TARGET_GMM = 0, MFM_TARGET_PHI4 = 1, MFM_TARGET_PINES = 2, MFM_TARGET_GAUSS = 3, MFM_TARGET_PINES_WHITE = 4 };
enum { MFM_ACT_RELU = 0, MFM_ACT_TANH = 1, MFM_ACT_ELU = 2, MFM_ACT_GELU = 3, MFM_ACT_SWISH = 4 };

/* Target descriptor: replaces the Python closure `logdensity_fn` that the reference passes to
 * bblackjax.mcmc.mala.init/kernel (mala.py:51-54,86-93) and `dist.loglik/logprior/logprob`
 * (distributions.py).  logprob_beta(x) = beta * loglik(x) + logprior(x)
 * (exe_flow_matching.py:301). */
typedef struct mfm_target {
    int kind;            /* MFM_TARGET_* */
    int dim;             /* d */
    float beta;          /* tempering inverse temperature (1 = untempered) */
    /* GMM (distributions.py:42-61): dim must be 2 */
    int n_modes;
    const float* modes;   /* [K,2] */
    const float* stds;    /* [K,2] = sqrt(covs) */
    const float* weights; /* [K] */
    /* phi-four (distributions.py:114-160), Dirichlet(0) boundary */
    float phi_a, phi_beta;
    /* pines LGCP (distributions.py:231-307, cox_process_utils.py:98-165) */
    const float* counts;  /* [d] flat bin counts */
    const float* kinv;    /* [d,d] inverse Gram matrix (symmetric), fp32 */
    const float* kinv_mu; /* [d] mu * rowsum(kinv) */
    const float* kinv_diag; /* [d] diagonal of kinv */
    const float* kinv_split; /* optional: mfm_gemm_presplit mirror of kinv (d*d + 16 floats; constant for the whole run), or NULL */
    float mu, log_norm, poisson_a;
    /* whitened pines (use_whitened=True, distributions.py:276-297; cox_process_utils.py:118-140): the state is the white noise e,
     * latents f = L e + mu, loglik = Poisson(f), logprior = -|e|^2/2 + log_norm.  chol = L [d,d] row-major, chol_t = L^T,
     * chol_sq_t = (L o L)^T (diagonal of the Hessian), mu_vec = mu * 1 [d]; counts / mu / poisson_a / log_norm as above. */
    const float* chol; const float* chol_t; const float* chol_sq_t; const float* mu_vec;
    /* independent Gaussian (distributions.py:80-97) */
    float gauss_mean, gauss_std;
} mfm_target_t;

/* VectorFieldNet parameters (exe_flow_matching.py:56-90).  One flat fp32 parameter buffer; layer i
 * (flax name Dense_i) has kernel [in_i, out_i] row-major at params + w_off[i] and bias [out_i] at
 * params + b_off[i].  Each branch has two hidden layers, hidden_t = [Ht0, Ht1], hidden_x = [Hx0, Hx1],
 * hidden_xt = [Hxt0, Hxt1] (the fields at the end of the struct):
 *   Dense_0 (2F, Ht0)   Dense_1 (Ht0, Ht1)          time branch -> s_t
 *   Dense_2 (d, Hx0)    Dense_3 (Hx0, Hx1)          x branch    -> s_x
 *   Dense_4 (Ht1, d)                                nn_t head
 *   Dense_5 (Hx1 + Ht1, Hxt0), input [s_x | s_t]    Dense_6 (Hxt0, Hxt1)   joint branch
 *   Dense_7 (Hxt1, d)                               nn_xt head
 * With all six widths equal to `hidden` = H: 2F->H->H, d->H->H, H->d, 2H->H->H, H->d. */
typedef struct mfm_field {
    int dim, hidden, fourier_dim;
    const float* params;     /* flat buffer */
    long long w_off[8], b_off[8];
    long long n_params;      /* total floats */
    const float* omega;      /* [F] fourier_random (module attribute, :350-351) */
    float grad_clip;         /* <=0: no clip; else clip grad logprob to +-grad_clip (:87-90) */
    /* reference (base) distribution of the flow, ref_dists[args.ref_dist] (exe_flow_matching.py:48-54,149,244).  Used by the
     * conditional FM batch (x0 = ref.sample_model, :156), by the independent / importance-sampling flow steps (:249-256,283-289)
     * and by mfm_ref_sample / mfm_ref_logprob.  Kind ref_kind below; MFM_REF_INDEP_GAUSS: IndepGaussian(dim, mean,
     * var = ref_std^2), stdgauss = (0, 1), widegauss = (0, sqrt(5)). */
    float ref_mean, ref_std;
    /* activation of the six hidden layers, args.non_linearity (exe_flow_matching.py:40-46, multi_modal.py:181):
     * MFM_ACT_RELU (0, the default of every configuration), TANH, ELU, GELU (jax.nn.gelu's default tanh approximation), SWISH */
    int act;
    /* MFM_REF_INDEP_GAUSS (0): the IndepGaussian above (ref_log_norm, ref_band unused; a zero-filled tail is exactly that).
     * MFM_REF_PHI4_BASE (1): PhiFourBase(dim, alpha, beta), prior_type 'coupled' (distributions.py:168-226), the Gaussian
     * N(0, P^-1) with the tridiagonal precision P = beta (diag(2c + 1/c) - c (sub + super diagonal)), c = alpha dim.  P = L L^T with
     * L lower bidiagonal (diagonal l, sub-diagonal s_i = L[i][i-1]); ref_band (device, 2 d + 2 floats) = a[d] (a_i = -s_{i+1} / l_i,
     * a_{d-1} = 0), rl[d] (rl_i = 1 / l_i), beta c, beta / c.  sample_model = L^-T z, z = normal(key, (d,)), by the back-substitution
     * x_{d-1} = rl_{d-1} z_{d-1}, x_i = a_i x_{i+1} + rl_i z_i; logprob(x) = -q/2 + ref_log_norm
     * with q = beta (c sum_{i=0..d} (x_i - x_{i-1})^2 + sum x_i^2 / c), x_{-1} = x_d = 0, ref_log_norm = -d/2 log 2 pi + sum log l_i.
     * d <= MFM_REF_BAND_MAX_DIM for this kind (the row is staged in shared memory). */
    int ref_kind;
    float ref_log_norm;
    const float* ref_band;
    /* hidden widths of the three branches (layer table above).  All six zero: every width is `hidden` (a zero-filled tail is
     * the equal-width network).  Otherwise all six must be > 0 and `hidden` must equal the largest of them, else the field and
     * FM entry points return MFM_ERR_ARG.  Only two layers per branch are supported. */
    int hidden_t[2], hidden_x[2], hidden_xt[2];
} mfm_field_t;
enum { MFM_REF_INDEP_GAUSS = 0, MFM_REF_PHI4_BASE = 1 };
#define MFM_REF_BAND_MAX_DIM 12192

typedef struct mfm_ode_opts {
    float rtol, atol;        /* multi_modal.py:205-206 */
    int mxstep;              /* :207 */
    int hutch;               /* 1: Hutchinson (Gaussian probe); 0: exact trace */
    int n_times;             /* output grid size (2, or 5 for 4-mode, exe_flow_matching.py:347) */
} mfm_ode_opts_t;

const char* mfm_last_error(void);
int mfm_version(void);
/* number of CUDA kernels this library has launched in the calling process (diagnostics / bench) */
unsigned long long mfm_launch_count(void);
/* dense-layer backend: 0 = auto (tcgen05/TMEM/TMA kernels: persistent CTA-pair cta_group::2 kernel when M >= 256,
 * single-CTA tiles when the shape is otherwise eligible), 1 = warp-level mma.sync kernel only, 2 = single-CTA tcgen05
 * only, 3 = one-tile CTA-pair kernel (separate cross-term accumulators: 3x smaller accumulator-truncation bias, no
 * epilogue overlap).  Same 3xTF32 arithmetic every way; environment variable MFM_GEMM=mma|tc1|tc2. */
void mfm_set_gemm_backend(int backend);
/* CTA-pair kernel operand split: 1 (default) = leave the raw fp32 tile as the hi operand (the tensor core ignores the
 * 13 low mantissa bits of a tf32 operand; measured on B200) and store only lo = rn_tf32(x - trunc(x)), which saves
 * a third of the splitter's shared-memory traffic; 0 = hi = rn_tf32(x), lo = rn_tf32(x - hi).
 * Environment variable MFM_TC_RAWHI=0|1. */
void mfm_set_gemm_raw_hi(int raw_hi);
/* Cross terms of the persistent kernel when both operands are K-major (A[m][k], B[n][k]): 0 = two kind::tf32 MMAs per
 * k-step (a_lo*b_hi, a_hi*b_lo: "3xTF32"); 1 = one kind::f16 MMA with K=16 over bf16 copies [a_lo | a] x [b | b_lo]
 * built by the splitter warps (error ~2^-19 relative on terms that are 2^-11 of the product).
 * Environment variable MFM_GEMM_CROSS=tf32|bf16. */
void mfm_set_gemm_cross_bf16(int enable);
/* Stream-K for the remainder round of the persistent kernel: when the tile count is not a multiple of the number of
 * CTA pairs (74), the k-blocks of the last, partially filled round are cut into equal contiguous ranges over the pairs;
 * partial accumulators go through an L2-resident per-stream scratch area the library allocates on first use (19.4 MB)
 * and the pair that owns a tile's last k-range adds them, in a fixed order, before the epilogue functor runs.
 * 1 (default) = on, 0 = whole tiles only.  Environment variable MFM_STREAMK=0|1. */
void mfm_set_gemm_streamk(int enable);
/* Scaled-fp16 three-pass kernel (csrc/gemm_tcgen05_h16.cuh), the DEFAULT for dense layers whose operands are both K-major with
 * K a multiple of 16: each operand is scaled by a per-tensor power of two (max |x| -> [2^14, 2^15)) and split into two fp16 parts,
 * the product is hi.hi' + hi.lo' + lo.hi' in three kind::f16 MMAs per 16 k-values; operand rounding 2^-22.  The maxima are exact:
 * every producer of a GEMM operand folds max |value| into a device slot, operands nobody tracked get one reduction pass.
 * Layers hand their results over pre-split (the epilogue writes the consumer's operand format next to the fp32 tensor) and the
 * weight gradients read the same copies as MN-major tiles (csrc/gemm_tcgen05_wgrad16.cuh).  Used by the MLP entry points when the
 * network is at least 512 wide and the batch has at least 256 rows; narrower / shorter problems keep the kernels below.
 * 0 = fall back to tf32 hi*hi + bf16 cross terms everywhere.  Environment variable MFM_GEMM_H16=0|1. */
void mfm_set_gemm_h16(int enable);
int mfm_gemm_h16_enabled(void);
/* one-line description of the arithmetic the dense layers currently use (bench.py quotes it) */
const char* mfm_gemm_describe(void);
/* Pre-split B operand (test / benchmark hooks; the ABI entry points below do this themselves for the MLP weights, inside their
 * workspace).  mfm_gemm_presplit writes the mirror of n_floats K-major fp32 values - split16 layout of scaled fp16 parts
 * (n_floats % 16 == 0, pointers 64-byte aligned) or, with the h16 kernel switched off, the bf16 cross mirror (% 8, 32-byte aligned);
 * `mirror` must hold n_floats + 16 floats: max |src| is kept behind the parts.  mfm_gemm_register_mirror announces it for the calling
 * thread's next GEMMs (base == NULL clears the registry). */
int mfm_gemm_presplit(const float* src, float* mirror, long long n_floats, mfm_stream_t stream);
void mfm_gemm_register_mirror(const float* base, long long n_floats, const float* mirror);
/* out[0] = max |x[r, c]| over rows x cols (cols, ld multiples of 4): the reduction the h16 kernel falls back to */
int mfm_absmax(const float* x, long long ld, int rows, int cols, float* out, mfm_stream_t stream);
/* Dense layer as the MLP calls it (test / benchmark hook): C = relu?(A[M,K] * Bt[N,K]^T + bias); a_amax (optional, device) = max |A|
 * as A's producer tracked it, c_amax (optional, device, zeroed by the caller) receives max |C|.  a_split (optional): A once more in
 * the split16 layout of scaled fp16 parts, as the producing layer's epilogue leaves it (for a contiguous A: mfm_gemm_presplit),
 * scaled by the power of two derived from *a_scale_src; the kernel then loads that copy and splits nothing in shared memory. */
int mfm_gemm_dense(int M, int N, int K, const float* A, long long lda, const float* Bt, long long ldb, const float* bias, int relu,
                   float* C, long long ldc, const float* a_amax, float* c_amax, const float* a_split, const float* a_scale_src,
                   mfm_stream_t stream);
/* Host-only test hook: the work list the persistent kernel derives for an M x N x K problem on n_pairs CTA pairs, as
 * rows of 7 ints (pair, tile, first k-block, end k-block, kind 0 whole / 1 contribution / 2 finishing part, first
 * contributing pair, number of contributing pairs).  Returns the number of rows; writes at most `cap` of them. */
int mfm_debug_gemm_plan(int M, int N, int K, int n_pairs, int streamk, int* rows, int cap);

/* ---- RNG: jax.random semantics (threefry2x32, legacy keys) ----------------------------------
 * Draw layout.  0 (default): float32 draws (32 random bits each) - the parity mode `north_star` names.  1: the layout of the
 * reference AS SHIPPED, which sets jax_enable_x64 (multi_modal.py:14): every uniform / normal draw consumes 64 bits
 * (random_bits(key, 64, shape): word i of the 2n-word stream is the high half, word n + i the low half), is transformed in
 * float64 (mantissa fill of 52 bits; sqrt(2) erfinv(uniform(nextafter(-1, 0), 1))) and rounded to float32 once, because this
 * library computes in float32.  The switch applies to EVERY draw the library makes (mfm_threefry_uniform / _normal, MALA noise
 * and accept uniforms, the FM batch, Hutchinson probes, flow-MH proposals, resampling); keys and splits are unaffected.
 * Environment variable MFM_RNG_X64=0|1. */
void mfm_set_rng_x64(int enable);
int mfm_rng_x64_enabled(void);
/* jax.random.split(key, num) -> out uint32[num,2] */
int mfm_threefry_split(const uint32_t* key, int num, uint32_t* out, mfm_stream_t stream);
/* vmap(lambda k: split(k, num))(keys[n]) -> out uint32[n,num,2] */
int mfm_threefry_split_batched(const uint32_t* keys, int n, int num, uint32_t* out, mfm_stream_t stream);
/* jax.random.bits(key, (n,), uint32) */
int mfm_threefry_bits(const uint32_t* key, long long n, uint32_t* out, mfm_stream_t stream);
/* jax.random.uniform(key, (n,), minval, maxval): the bounds are rounded to float32 for float32 draws (as jax does) and used as
 * float64 values for float64 draws */
int mfm_threefry_uniform(const uint32_t* key, long long n, double minval, double maxval, float* out, mfm_stream_t stream);
/* jax.random.normal(key, (n,), float32) */
int mfm_threefry_normal(const uint32_t* key, long long n, float* out, mfm_stream_t stream);
/* vmap(lambda k: uniform(k, (d,), float32, minval, maxval))(keys[n]) -> out [n,d] */
int mfm_threefry_uniform_batched(const uint32_t* keys, int n, int d, double minval, double maxval, float* out, mfm_stream_t stream);
/* vmap(lambda k: normal(k, (d,)))(keys[n]) -> out [n,d] */
int mfm_threefry_normal_batched(const uint32_t* keys, int n, int d, float* out, mfm_stream_t stream);
/* host-side threefry split (key management outside the device), same semantics */
void mfm_host_threefry_split(const uint32_t key[2], int num, uint32_t* out);

/* ---- dense contraction used by every layer (test hook) --------------------------------------
 * C[M,N] = relu?(opA(A)[M,K] * opB(B)[K,N] + bias[N]); fp32 in/out, 3xTF32 on tensor cores.
 * a_kmajor: A[m*lda+k] (else A[k*lda+m]);  b_nmajor: B[k*ldb+n] (else B[n*ldb+k]). */
int mfm_gemm_tf32x3(int M, int N, int K, const float* A, long long lda, int a_kmajor, const float* B, long long ldb,
                    int b_nmajor, const float* bias, int relu, float* C, long long ldc, mfm_stream_t stream);

/* Backward-data form of a dense layer (test / benchmark hook of the fused epilogue):
 * C[M,N] = (A[M,K] * Bt[N,K]^T + add[M,N]) where mask[M,N] > 0, else 0; add and mask optional; add may alias C. */
int mfm_gemm_tf32x3_gated(int M, int N, int K, const float* A, long long lda, const float* Bt, long long ldb, const float* mask,
                          long long ldm, const float* add, long long ldadd, float* C, long long ldc, mfm_stream_t stream);

/* Dense layer over the first *n_rows_dev rows only (test hook of the ODE driver's active-chain compaction: the row count
 * lives in device memory and every kernel reads it; rows beyond it are left untouched).  C = A[M,K] * Bt[N,K]^T + bias. */
int mfm_gemm_tf32x3_rows(int M, int N, int K, const float* A, long long lda, const float* Bt, long long ldb, const float* bias,
                         float* C, long long ldc, const int* n_rows_dev, mfm_stream_t stream);

/* ---- targets -------------------------------------------------------------------------------- */
size_t mfm_target_workspace_bytes(const mfm_target_t* t, int n);
/* vmap(init)(positions, logprob_beta): mala.py:51-54, exe_flow_matching.py:316.
 * loglik_out (optional) receives the untempered log-likelihood (exe_flow_matching.py:418). */
int mfm_logdensity_and_grad(const mfm_target_t* t, int n, const float* x, float* logp, float* grad,
                            float* loglik_out, void* ws, size_t ws_bytes, mfm_stream_t stream);

/* ---- MALA (bblackjax/mcmc/mala.py:86-118 + diffusions.py:22-33 + proposal.py) --------------- */
size_t mfm_mala_workspace_bytes(const mfm_target_t* t, int n);
/* keys = split(rng_key, n); vmap(kernel)(keys, states, logprob_beta, step_size)
 * (exe_flow_matching.py:303,313).  State arrays are updated IN PLACE.
 * chain_offset/n_total: this rank holds chains [chain_offset, chain_offset+n) of an n_total-chain
 * ensemble; per-chain keys are rows of split(rng_key, n_total) so sharded runs draw the same
 * numbers as the single-GPU run.  per_chain_keys=1: rng_key is uint32[n,2], the already-split
 * per-chain keys (what jax.vmap hands to bblackjax's kernel); chain_offset/n_total are ignored. */
int mfm_mala_step(const mfm_target_t* t, const uint32_t* rng_key, int per_chain_keys, int n, int chain_offset, int n_total,
                  float step_size, float* position, float* logdensity, float* logdensity_grad,
                  float* acceptance_rate, uint8_t* is_accepted, float* proposed_position,
                  float* proposed_weight, void* ws, size_t ws_bytes, mfm_stream_t stream);

/* ---- CNF push / pull (exe_flow_matching.py:206-242, jax.experimental.ode.odeint) ------------ */
size_t mfm_ode_workspace_bytes(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n);
/* direction +1: transform_and_logdet (u -> x, ldj);  -1: inverse_and_logdet (x -> u, ldj).
 * hutch_keys uint32[n,2]: per-chain probe keys (ignored when !hutch).  stats (optional, device
 * int32[8], 8-byte aligned): total accepted steps, total attempted steps, max attempted steps per chain, field
 * evaluations, then an int64 in [4..5]: chain-evaluations = rows actually evaluated summed over the field evaluations
 * (finished chains are compacted away), [6..7] reserved. */
int mfm_ode_flow(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int direction, int n,
                 const uint32_t* hutch_keys, const float* y0, float* y1, float* ldj, int* stats,
                 void* ws, size_t ws_bytes, mfm_stream_t stream);
/* single evaluation of (v, div v) at (x[n,d], t[n]) — test hook for VectorFieldNet parity */
int mfm_field_eval(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n,
                   const float* x, const float* time, const float* z, float* v, float* div,
                   void* ws, size_t ws_bytes, mfm_stream_t stream);

/* ---- flow-MH step (exe_flow_matching.py:246-278) -------------------------------------------- */
enum { MFM_FLOW_RW_MH = 0, MFM_FLOW_INDEP_MH = 1 };
size_t mfm_flow_mh_workspace_bytes(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n);
int mfm_flow_mh_step(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int variant,
                     const uint32_t* rng_key, int per_chain_keys, int n, int chain_offset, int n_total,
                     float* position, float* logdensity, float* logdensity_grad,
                     float* acceptance_rate, uint8_t* is_accepted, float* proposed_position,
                     float* proposed_weight, int* stats, void* ws, size_t ws_bytes, mfm_stream_t stream);

/* conditional_importance_sampling (exe_flow_matching.py:280-296; --num_importance_samples K > 0): per chain the current state is
 * pulled back (weight exp(l - logq(u) - V)), K fresh reference samples are pushed through the flow with their own probe keys,
 * and one of the K + 1 candidates is drawn with jax.random.choice(key_choice, K + 1, p = normalised weights).  As coded the
 * gradient of the state is NOT recomputed (logdensity_grad is left untouched); acceptance_rate = proposed_weight = the chosen
 * candidate's normalised weight, proposed_position = the chosen sample (the old position when candidate 0 wins). */
size_t mfm_flow_cis_workspace_bytes(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n, int n_is);
int mfm_flow_cis_step(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n_is, const uint32_t* rng_key,
                      int per_chain_keys, int n, int chain_offset, int n_total, float* position, float* logdensity,
                      float* acceptance_rate, uint8_t* is_accepted, float* proposed_position, float* proposed_weight, int* stats,
                      void* ws, size_t ws_bytes, mfm_stream_t stream);

/* ---- reference distribution of the flow (f->ref_kind; only the ref_* fields and dim of `f` are read) ------------------
 * mfm_ref_sample: vmap(ref_dist.sample_model)(keys[n]) -> out [n,d] (exe_flow_matching.py:156,249,284,453).
 * mfm_ref_logprob: vmap(ref_dist.logprob)(x[n,d]) -> out [n] (:251-252,283,289,457). */
int mfm_ref_sample(const mfm_field_t* f, const uint32_t* keys, int n, float* out, mfm_stream_t stream);
int mfm_ref_logprob(const mfm_field_t* f, int n, const float* x, float* out, mfm_stream_t stream);

/* ---- flow-matching update (exe_flow_matching.py:151-179, 362-368, 129-137, 184) ------------- */
size_t mfm_fm_workspace_bytes(const mfm_field_t* f, const mfm_target_t* t, int n);
/* loss = sum |v(x_t, t) - (x - x0)|^2 and d loss / d params (flat, same layout as params).
 * loss_out: device float[1].  grads are OVERWRITTEN (not accumulated). */
int mfm_fm_loss_grad(const mfm_field_t* f, const mfm_target_t* t, const uint32_t* rng_key, int n,
                     int chain_offset, int n_total, float sigma, const float* positions,
                     float* loss_out, float* grads, void* ws, size_t ws_bytes, mfm_stream_t stream);
/* The same computation in two calls so that the multi-GPU host can overlap the gradient all-reduce with the
 * backward pass: part 1 = batch, forward, loss and the gradients of Dense_7..Dense_4, i.e. grads[w_off[4] .. n_params);
 * part 2 = the gradients of Dense_3..Dense_0, grads[0 .. w_off[4]), from the activations part 1 left in `ws` (same
 * arguments, same workspace, nothing else may use `ws` in between); part 0 = both (== mfm_fm_loss_grad).
 * Part 1 also writes the BIAS gradients of Dense_3 and Dense_1 (they are column sums of signals it produces); both lie in
 * grads[0 .. w_off[4]), which nothing reads before part 2 has returned.  The weight gradients run on a second, internal stream
 * and are joined to `stream` before each call returns (not while `stream` is being captured into a CUDA graph). */
int mfm_fm_loss_grad_part(const mfm_field_t* f, const mfm_target_t* t, const uint32_t* rng_key, int n, int chain_offset,
                          int n_total, float sigma, const float* positions, float* loss_out, float* grads, void* ws,
                          size_t ws_bytes, int part, mfm_stream_t stream);
/* same with the NON-conditional batch, flow_fn (exe_flow_matching.py:139-147; the reference's --cond_flow switched off):
 * key_time, key_ref = split(key); x_t = t x + (1 - (1-sigma) t) ref, target = x - (1-sigma) ref, ref = normal(key_ref, (N,d)). */
int mfm_fm_loss_grad_uncond(const mfm_field_t* f, const mfm_target_t* t, const uint32_t* rng_key, int n, int chain_offset,
                            int n_total, float sigma, const float* positions, float* loss_out, float* grads, void* ws,
                            size_t ws_bytes, mfm_stream_t stream);
/* same, from explicit (x_t, t, target) — test hook */
int mfm_fm_loss_grad_from_batch(const mfm_field_t* f, const mfm_target_t* t, int n, const float* xt,
                                const float* times, const float* target_v, float* loss_out, float* grads,
                                void* ws, size_t ws_bytes, mfm_stream_t stream);

/* optax.apply_if_finite(chain(adamw(lr_fn, b1, b2, eps, wd, mask=no-bias), clip(c)), max_err)
 * opt_state: device int32[8] = {adam count, notfinite_count, total_notfinite, last_finite, scratch x4}.
 * decay_mask: uint8[n_params] (1 = kernel, decayed; 0 = bias).  Learning rate (create_learning_rate_fn, :189-198): linear warm-up
 * 0 -> lr_base over lr_warmup_steps, then linear decay to 0 at lr_total_steps (warm-up 0 = lr_base*(1-count/lr_total_steps)). */
int mfm_adamw_step(float* params, const float* grads, float* mu, float* nu, const uint8_t* decay_mask,
                   long long n_params, int* opt_state, float lr_base, int lr_total_steps, int lr_warmup_steps, float b1, float b2,
                   float eps, float weight_decay, float clip, int max_consecutive_errors, mfm_stream_t stream);

/* ---- adaptive tempering (exe_flow_matching.py:391-402) ---------------------------------------
 * beta_out[0] = jaxopt.Bisection(ess_zero, lower=prev_beta, upper=1, maxiter=30, tol=1e-5).run().params with
 * ess_zero(beta) = 1/sum(softmax(loglik*(beta-prev_beta))^2) - alpha*n.  logliks: ALL n chains of the ensemble
 * (all-gather first when sharded); prev_beta, beta_out: device float[1]. */
int mfm_tempering_beta(const float* logliks, int n, const float* prev_beta, float alpha, float* beta_out,
                       mfm_stream_t stream);

/* ---- final sampling: importance weights + multinomial resampling (exe_flow_matching.py:453-459) ------------
 * log_weights[i] = logdensity[i] - ref_logdensity[i] - vols[i]   (:457);   weights[i] = exp(log_weights[i] - max)   (:458) */
int mfm_importance_weights(const float* logdensity, const float* ref_logdensity, const float* vols, int n, float* log_weights,
                           float* weights, mfm_stream_t stream);
/* jax.random.choice(key, n_pop, (n_draw,), replace=True, p=p) -> idx_out int32[n_draw] (:459; p need not be normalised):
 * p_cuml = cumsum(p) (sequential float32), r = p_cuml[-1] * (1 - uniform(key, (n_draw,))), idx = searchsorted(p_cuml, r). */
size_t mfm_random_choice_workspace_bytes(int n_pop);
int mfm_random_choice(const uint32_t* key, int n_pop, const float* p, int n_draw, int* idx_out, void* ws, size_t ws_bytes,
                      mfm_stream_t stream);
/* jnp.take(src[n_pop,d], idx[n_draw], axis=0) -> out[n_draw,d] */
int mfm_gather_rows(const float* src, const int* idx, int n_pop, int n_draw, int d, float* out, mfm_stream_t stream);

/* ---- evaluation metrics (mcmc_utils.py:28-85, :88-111; exe_flow_matching.py:463-488) ----------------------
 * stein_disc(X, logprob_fn, beta): kernelised Stein discrepancy with the IMQ kernel (1 + |x-x'|^2)^beta, beta = -1/2 in
 * every call.  X [T,d] samples, grad_logp [T,d] = grad log pi at the samples (mfm_logdensity_and_grad).
 * out_uv = (U-statistic, V-statistic).  Pair values in float32, sums in float64 in a fixed order. */
size_t mfm_pairwise_workspace_bytes(int t);
int mfm_stein_disc(const float* X, const float* grad_logp, int T, int d, float beta, float* out_uv, void* ws, size_t ws_bytes,
                   mfm_stream_t stream);
/* max_mean_disc(X, Y): squared MMD with the Gaussian kernel exp(-|x-y|^2 / 2), X and Y [m,d]; out[0] =
 * (sum k(X,X) - m)/(m^2 - m) - 2 sum k(X,Y)/m^2 + (sum k(Y,Y) - m)/(m^2 - m). */
int mfm_max_mean_disc(const float* X, const float* Y, int m, int d, float* out, void* ws, size_t ws_bytes, mfm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MFM_B200_H */
