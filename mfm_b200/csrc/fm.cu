// Flow-matching update: conditional-flow batch, loss, gradient w.r.t. the MLP parameters, and the
// fused AdamW -> clip -> apply_if_finite step.
//
// Replaces:
//   cond_flow_fn / flow_matching_loss        exe_flow_matching.py:151-179
//   jax.value_and_grad(loss_fn, argnums=2)   :364-365  (hand-written backward of VectorFieldNet)
//   optax chain in create_train_state        :129-137, :184   [restated in oracle/optim.py]
#include "internal.h"
#include "gemm_tf32x3.cuh"
#include "gemm_tcgen05_wgrad16.cuh"
#include "ref_dist.cuh"

namespace mfm {

// ---------------------------------------------------------------------------------------------
// batch generation:  t ~ U[0,1)^(N,1); x0_i = normal(split(key_ref,N)_i,(d,)); eps ~ N(0,I)^(N,d)
// x_t = sigma*eps + t*x + (1-t)*x0 ; target = x - x0      (one warp per chain)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
fm_batch_kernel(const uint32_t* __restrict__ rng_key, int n, int chain_offset, int n_total, int d, float sigma,
                float ref_mean, float ref_std, const float* __restrict__ x, float* __restrict__ times, float* __restrict__ xt,
                float* __restrict__ target, float* __restrict__ xt_amax, int x64) {
    __shared__ double2 ltab[16];
    log_tab_load(ltab);                                                    // (before any warp leaves: contains a barrier)
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;                                                    // whole warps leave together
    float vm = 0.0f, tm = 0.0f;
    const uint32_t gc = (uint32_t)(chain_offset + c);
    // key_time, key_ref, key_gauss, key_ot = split(rng_key, 4)
    const u32x2 k_time = threefry_split_key(rng_key[0], rng_key[1], 0u, 4u);
    const u32x2 k_ref = threefry_split_key(rng_key[0], rng_key[1], 1u, 4u);
    const u32x2 k_gauss = threefry_split_key(rng_key[0], rng_key[1], 2u, 4u);
    const float t = rng_uniform_at(k_time.a, k_time.b, gc, (uint32_t)n_total, x64);
    const u32x2 k_row = threefry_split_key(k_ref.a, k_ref.b, gc, (uint32_t)n_total);
    const uint32_t total = (uint32_t)n_total * (uint32_t)d;
    const uint32_t half = ((uint32_t)d + 1u) >> 1;
    const float omt = 1.0f - t;
    for (uint32_t b = lane; b < half; b += 32) {
        const uint32_t hi = b + half;
        const bool has_hi = hi < (uint32_t)d;
        u32x2 o; o.a = o.b = 0u;
        if (!x64) o = threefry2x32(k_row.a, k_row.b, b, has_hi ? hi : 0u);
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            if (s == 1 && !has_hi) break;
            const uint32_t j = s == 0 ? b : hi;
            // ref_dist.sample_model: mean + std * normal (distributions.py:96-97); exact identity for stdgauss (0, 1)
            const float nrm = x64 ? rng_normal_at(k_row.a, k_row.b, j, (uint32_t)d, 1) : bits_to_normal_t(s == 0 ? o.a : o.b, ltab);
            const float x0 = __fadd_rn(ref_mean, __fmul_rn(ref_std, nrm));
            const float eps = x64 ? rng_normal_at(k_gauss.a, k_gauss.b, gc * (uint32_t)d + j, total, 1) : rng_normal_at_t(k_gauss.a, k_gauss.b, gc * (uint32_t)d + j, total, ltab);
            const long long idx = (long long)c * d + j;
            const float xv = x[idx];
            // sigma*eps + t*x + (1-t)*x0, left to right (:167)
            const float xtv = __fadd_rn(__fadd_rn(__fmul_rn(sigma, eps), __fmul_rn(t, xv)), __fmul_rn(omt, x0));
            xt[idx] = xtv; vm = fmaxf(vm, fabsf(xtv));
            const float tg = xv - x0;                                      // :168
            target[idx] = tg; tm = fmaxf(tm, fabsf(tg));
        }
    }
    if (lane == 0) times[c] = t;
    if (xt_amax) {
        amax_publish_warp(xt_amax, vm);                                    // x_t is the A operand of Dense_2 / the K^-1 GEMM
        amax_publish_warp(xt_amax + (AM_TGT - AM_X), tm);                  // (xt_amax is slot AM_X of the pool) bounds the loss gradient
    }
}

// The same batch with the PhiFourBase reference distribution (ref_kind MFM_REF_PHI4_BASE): x0 = L^-T z where z is the normal row
// fm_batch_kernel draws (same keys, same paired float32 layout, same x64 layout).  The row z is staged in shared memory
// (band_solve_warp, ref_dist.cuh), solved there, and then x_t / target are formed exactly as above.  Dynamic shared memory:
// band_row_floats(d) floats per warp.
__global__ void __launch_bounds__(256)
fm_batch_phi4_kernel(const uint32_t* __restrict__ rng_key, int n, int chain_offset, int n_total, int d, float sigma,
                     const float* __restrict__ band, const float* __restrict__ x, float* __restrict__ times, float* __restrict__ xt,
                     float* __restrict__ target, float* __restrict__ xt_amax, int x64) {
    __shared__ double2 ltab[16];
    extern __shared__ float band_rows[];
    log_tab_load(ltab);                                                    // (before any warp leaves: contains a barrier)
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;                                                    // whole warps leave together
    const int m = (d + 31) >> 5, mp = m | 1;
    const float inv_m = 1.0f / (float)m;
    float* r = band_rows + (threadIdx.x >> 5) * 32 * mp;
    float vm = 0.0f, tm = 0.0f;
    const uint32_t gc = (uint32_t)(chain_offset + c);
    const u32x2 k_time = threefry_split_key(rng_key[0], rng_key[1], 0u, 4u);
    const u32x2 k_ref = threefry_split_key(rng_key[0], rng_key[1], 1u, 4u);
    const u32x2 k_gauss = threefry_split_key(rng_key[0], rng_key[1], 2u, 4u);
    const float t = rng_uniform_at(k_time.a, k_time.b, gc, (uint32_t)n_total, x64);
    const u32x2 k_row = threefry_split_key(k_ref.a, k_ref.b, gc, (uint32_t)n_total);
    const uint32_t total = (uint32_t)n_total * (uint32_t)d;
    const uint32_t half = ((uint32_t)d + 1u) >> 1;
    // z = normal(k_row, (d,)) into shared memory
    for (uint32_t b = lane; b < half; b += 32) {
        const uint32_t hi = b + half;
        const bool has_hi = hi < (uint32_t)d;
        if (x64) {
            r[band_slot((int)b, m, mp, inv_m)] = rng_normal_at(k_row.a, k_row.b, b, (uint32_t)d, 1);
            if (has_hi) r[band_slot((int)hi, m, mp, inv_m)] = rng_normal_at(k_row.a, k_row.b, hi, (uint32_t)d, 1);
        } else {
            const u32x2 o = threefry2x32(k_row.a, k_row.b, b, has_hi ? hi : 0u);
            r[band_slot((int)b, m, mp, inv_m)] = bits_to_normal_t(o.a, ltab);
            if (has_hi) r[band_slot((int)hi, m, mp, inv_m)] = bits_to_normal_t(o.b, ltab);
        }
    }
    band_solve_warp(r, d, band, lane);                                     // ref_dist.sample_model: x0 = L^-T z
    const float omt = 1.0f - t;
    for (int j = lane; j < d; j += 32) {
        const float x0 = r[band_slot(j, m, mp, inv_m)];
        const float eps = x64 ? rng_normal_at(k_gauss.a, k_gauss.b, gc * (uint32_t)d + j, total, 1) : rng_normal_at_t(k_gauss.a, k_gauss.b, gc * (uint32_t)d + j, total, ltab);
        const long long idx = (long long)c * d + j;
        const float xv = x[idx];
        const float xtv = __fadd_rn(__fadd_rn(__fmul_rn(sigma, eps), __fmul_rn(t, xv)), __fmul_rn(omt, x0));   // (:167)
        xt[idx] = xtv; vm = fmaxf(vm, fabsf(xtv));
        const float tg = xv - x0;                                          // :168
        target[idx] = tg; tm = fmaxf(tm, fabsf(tg));
    }
    if (lane == 0) times[c] = t;
    if (xt_amax) {                                                         // the same maxima fm_batch_kernel publishes
        amax_publish_warp(xt_amax, vm);
        amax_publish_warp(xt_amax + (AM_TGT - AM_X), tm);
    }
}

// Non-conditional variant, flow_fn (exe_flow_matching.py:139-147, --cond_flow off):
//   key_time, key_ref = split(key);  t ~ U[0,1)^(N,1);  ref ~ N(0,I)^(N,d) (ONE draw for the whole batch)
//   x_t = t*x + (1 - (1-sigma) t) * ref ;  target = x - (1-sigma) * ref      (one warp per chain)
__global__ void __launch_bounds__(256)
fm_batch_uncond_kernel(const uint32_t* __restrict__ rng_key, int n, int chain_offset, int n_total, int d, float sigma,
                       const float* __restrict__ x, float* __restrict__ times, float* __restrict__ xt, float* __restrict__ target,
                       float* __restrict__ xt_amax, int x64) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    float vm = 0.0f;
    const uint32_t gc = (uint32_t)(chain_offset + c);
    const u32x2 k_time = threefry_split_key(rng_key[0], rng_key[1], 0u, 2u);
    const u32x2 k_ref = threefry_split_key(rng_key[0], rng_key[1], 1u, 2u);
    const float t = rng_uniform_at(k_time.a, k_time.b, gc, (uint32_t)n_total, x64);
    const uint32_t total = (uint32_t)n_total * (uint32_t)d;
    const float oms = 1.0f - sigma;
    const float sds = 1.0f - oms * t;                                     // :144
    for (int j = lane; j < d; j += 32) {
        const float ref = rng_normal_at(k_ref.a, k_ref.b, gc * (uint32_t)d + (uint32_t)j, total, x64);
        const long long idx = (long long)c * d + j;
        const float xv = x[idx];
        const float xtv = __fadd_rn(__fmul_rn(t, xv), __fmul_rn(sds, ref));      // :145
        xt[idx] = xtv; vm = fmaxf(vm, fabsf(xtv));
        target[idx] = xv - __fmul_rn(oms, ref);                          // :146
    }
    if (lane == 0) times[c] = t;
    if (xt_amax) amax_publish_warp(xt_amax, vm);
}

// diff = v - target; delta = 2*diff; dgt = delta*gc; per-block partial sums of diff^2
__global__ void __launch_bounds__(256)
fm_loss_delta_kernel(long long total, const float* __restrict__ v, const float* __restrict__ target,
                     const float* __restrict__ gc, float* __restrict__ delta, float* __restrict__ dgt,
                     float* __restrict__ block_partial, float* __restrict__ delta_amax, float* __restrict__ dgt_amax) {
    __shared__ float red[32];
    float s = 0.0f, m0 = 0.0f, m1 = 0.0f;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const float df = v[i] - target[i];
        s += df * df;
        const float dl = 2.0f * df;
        const float dg = dl * gc[i];
        delta[i] = dl; dgt[i] = dg;
        m0 = fmaxf(m0, fabsf(dl)); m1 = fmaxf(m1, fabsf(dg));
    }
    if (delta_amax) { amax_publish_warp(delta_amax, m0); amax_publish_warp(dgt_amax, m1); }   // both are GEMM operands of the backward pass
    s = block_sum(s, red);
    if (threadIdx.x == 0) block_partial[blockIdx.x] = s;
}

// The same, four elements per thread, ALSO writing delta and dgt in the split16 layout of the scaled-fp16 GEMMs (they are the
// A operands of two backward-data layers and the G operands of two weight gradients).  Their scales must be known before the
// first element is written: |delta| <= 2 (max |v| + max |target|) with both maxima exact (tracked by EpiFieldV and the batch
// kernel), |dgt| <= |delta| * clip (gc is clipped to [-clip, clip]).  The bounds go to bound_out[0 / 1] for the consumers.
__global__ void __launch_bounds__(256)
fm_loss_delta_split_kernel(long long total4, const float4* __restrict__ v, const float4* __restrict__ target, const float4* __restrict__ gc,
                           float4* __restrict__ delta, float4* __restrict__ dgt, float* __restrict__ block_partial,
                           float* __restrict__ delta_amax, float* __restrict__ dgt_amax, const float* __restrict__ v_amax,
                           const float* __restrict__ tgt_amax, float clip, float* __restrict__ delta_s, float* __restrict__ dgt_s,
                           float* __restrict__ bound_delta, float* __restrict__ bound_dgt) {
    __shared__ float red[32];
    const float bd = 2.0f * (*v_amax + *tgt_amax), bg = bd * clip;
    const float sd = __uint_as_float(h16_scale_exp_(bd) << 23), sg = __uint_as_float(h16_scale_exp_(bg) << 23);
    if (blockIdx.x == 0 && threadIdx.x == 0) { *bound_delta = bd; *bound_dgt = bg; }
    float s = 0.0f, m0 = 0.0f, m1 = 0.0f;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
        const float4 a = v[i], b = target[i], g = __ldg(gc + i);
        const float4 df = make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w);
        s += df.x * df.x; s += df.y * df.y; s += df.z * df.z; s += df.w * df.w;        // (same order as the scalar kernel's grid-stride sum is NOT required: the partials differ anyway)
        const float4 dl = make_float4(2.0f * df.x, 2.0f * df.y, 2.0f * df.z, 2.0f * df.w);
        const float4 dg = make_float4(dl.x * g.x, dl.y * g.y, dl.z * g.z, dl.w * g.w);
        delta[i] = dl; dgt[i] = dg;
        m0 = amax4(m0, dl); m1 = amax4(m1, dg);
        const long long e = 4 * i;                                                      // first of the four elements
        uint2 hp, lp;
        split_pair(dl.x * sd, dl.y * sd, hp.x, lp.x); split_pair(dl.z * sd, dl.w * sd, hp.y, lp.y);
        char* p = reinterpret_cast<char*>(delta_s + (e & ~15ll)) + 2 * (e & 15);
        *reinterpret_cast<uint2*>(p) = hp; *reinterpret_cast<uint2*>(p + 32) = lp;
        split_pair(dg.x * sg, dg.y * sg, hp.x, lp.x); split_pair(dg.z * sg, dg.w * sg, hp.y, lp.y);
        p = reinterpret_cast<char*>(dgt_s + (e & ~15ll)) + 2 * (e & 15);
        *reinterpret_cast<uint2*>(p) = hp; *reinterpret_cast<uint2*>(p + 32) = lp;
    }
    if (delta_amax) { amax_publish_warp(delta_amax, m0); amax_publish_warp(dgt_amax, m1); }
    s = block_sum(s, red);
    if (threadIdx.x == 0) block_partial[blockIdx.x] = s;
}

__global__ void final_sum_kernel(int n, const float* __restrict__ partial, float* __restrict__ out) {
    __shared__ float red[32];
    float s = 0.0f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s += partial[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[0] = s;
}

// column sums of a [n, cols] matrix (bias gradients).  Block (x, y): 32 columns x one slab of rows;
// slab partials are then added in fixed order (deterministic, no atomics).
constexpr int COLSUM_SLABS = 64;
__global__ void __launch_bounds__(256)
colsum_partial_kernel(int n, int cols, const float* __restrict__ a, long long lda, float* __restrict__ partial) {
    __shared__ float sm[8][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + cx;
    const int per = (n + gridDim.y - 1) / gridDim.y;
    const int r0 = blockIdx.y * per, r1 = min(n, r0 + per);
    float s = 0.0f;
    if (col < cols) for (int r = r0 + ry; r < r1; r += 8) s += a[(long long)r * lda + col];
    sm[ry][cx] = s;
    __syncthreads();
    if (ry == 0 && col < cols) {
        float t = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += sm[k][cx];
        partial[(long long)blockIdx.y * cols + col] = t;
    }
}
__global__ void colsum_final_kernel(int cols, int slabs, const float* __restrict__ partial, float* __restrict__ out) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= cols) return;
    float t = 0.0f;
    for (int z = 0; z < slabs; ++z) t += partial[(long long)z * cols + col];
    out[col] = t;
}

// column sums of the [nb, cols] per-32-row partials the backward-data epilogues leave (nb <= a few thousand): 32 columns per
// block, 8 row groups, fixed order - one launch instead of the partial + final pair
__global__ void __launch_bounds__(256) colsum_blocks_kernel(int nb, int cols, const float* __restrict__ part, long long ldp, float* __restrict__ out) {
    __shared__ float sm[8][33];
    const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + cx;
    float s = 0.0f;
    if (col < cols) for (int r = ry; r < nb; r += 8) s += part[(long long)r * ldp + col];
    sm[ry][cx] = s;
    __syncthreads();
    if (ry == 0 && col < cols) {
        float t = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += sm[k][cx];
        out[col] = t;
    }
}

// out[i] = sum_z partial[z*stride + i]
__global__ void splitk_reduce_kernel(long long count, int splits, long long stride, const float* __restrict__ partial,
                                     float* __restrict__ out) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= count) return;
    float s = 0.0f;
    for (int z = 0; z < splits; ++z) s += partial[(long long)z * stride + i];
    out[i] = s;
}

// split16 copies of a weight gradient's two operands and the device floats their scales came from (all four or none)
struct WgradSplit { const float* a_s = nullptr; const float* a_src = nullptr; const float* g_s = nullptr; const float* g_src = nullptr; };

// dW[in,out] = A^T[in,n] * D[n,out]  (A stored [n,in], lda), split over the batch dimension.  With the operands' split16
// copies at hand (ws) the product runs on three fp16 tensor-core passes (gemm_tcgen05_wgrad16.cuh), else on 3xTF32.
static int wgrad(int n, int in, int out, const float* A, long long lda, const float* D, long long ldd, float* dW,
                 float* splitbuf, size_t splitbuf_floats, cudaStream_t st, WgradSplit ws = WgradSplit()) {
    GemmShape probe{in, out, n, A, lda, D, ldd, nullptr};
    GemmShape p16{in, out, n, ws.a_s, lda, ws.g_s, ldd, nullptr};
    const bool h16w = ws.a_s && ws.a_src && ws.g_s && ws.g_src && tc2w::eligible(p16);
    // wave-aware split of the batch (reduction) dimension: fill the 148 SMs with whole waves
    const int path = h16w ? 2 : gemm_path<false, true>(probe);     // 2 = CTA pair, 1 = single CTA, 0 = mma.sync
    const long long tiles = path == 2 ? (long long)ceil_div(in, 2 * tc2::BM) * ceil_div(out, tc2::BN)
                          : path == 1 ? (long long)ceil_div(in, tc::BM) * ceil_div(out, tc::BN)
                                      : (long long)ceil_div(in, GBM) * ceil_div(out, GBN);
    const int slots = path == 2 ? 74 : (path == 1 ? 148 : 296);    // resident tiles per wave
    int max_splits = n / 512;
    if (max_splits > 64) max_splits = 64;
    while (max_splits > 1 && (size_t)max_splits * in * out > splitbuf_floats) --max_splits;
    int splits = 1;
    static const int forced = getenv("MFM_WGRAD_SPLITS") ? atoi(getenv("MFM_WGRAD_SPLITS")) : 0;     // tuning aid
    if (path == 2) {
        // CTA-pair kernels (one 256 x 256 tile per pair and launch wave): pick the split that minimises a small cost model -
        // waves x (fixed prologue + epilogue of a tile + its share of the k-loop) + the pass that adds the partial tiles.  Filling
        // the waves alone (the rule below) over-splits short batches: at 8 192 chains 9 slices of a 1024 x 1024 layer are two waves
        // of 15-stage tiles whose un-overlapped epilogues and 37 MB of partials cost more than the k-loop itself.
        const double t_fixed = 10.0, t_stage = h16w ? 1.3 : 2.4;                 // us: per tile; per 64 chains of one tile's k-loop
        const double red_us_per_mb = 0.4;                                        // the partials are written once and read once
        double best_t = 1e30;
        for (int sp = 1; sp <= max_splits; ++sp) {
            const long long waves = (tiles * sp + slots - 1) / slots;
            const double stages = (double)((n + sp - 1) / sp + 63) / 64.0;
            const double t = (double)waves * (t_fixed + stages * t_stage) + (sp > 1 ? (double)(sp + 1) * (double)in * out * 4e-6 * red_us_per_mb : 0.0);
            if (t < best_t - 1e-9) { best_t = t; splits = sp; }
        }
    } else {
        double best = 0.0;
        for (int sp = 1; sp <= max_splits; ++sp) {
            const long long ctas = tiles * sp;
            const double eff = (double)ctas / (double)(((ctas + slots - 1) / slots) * slots);
            if (eff > best + 1e-9) { best = eff; splits = sp; }
            if (eff >= 0.92) { splits = sp; break; }
        }
    }
    if (forced > 0) splits = forced < max_splits ? forced : (max_splits > 0 ? max_splits : 1);
    if (splits <= 1) {
        EpiStd e{dW, (long long)out, nullptr, nullptr, 0, nullptr, 0, 1.0f, 0};
        if (h16w) MFM_CUDA_CHECK((tc2w::launch(p16, e, ws.a_src, ws.g_src, st)));
        else MFM_CUDA_CHECK((launch_gemm<false, true>(probe, e, st)));
        return MFM_OK;
    }
    int kper = (n + splits - 1) / splits;
    kper = (kper + 63) / 64 * 64;                 // multiple of every kernel's k-tile (16 / 32 / 64)
    EpiStd e{splitbuf, (long long)out, nullptr, nullptr, 0, nullptr, 0, 1.0f, 0, 1, (long long)in * out};
    if (h16w) { p16.k_split = kper; MFM_CUDA_CHECK((tc2w::launch(p16, e, ws.a_src, ws.g_src, st))); }
    else { probe.k_split = kper; MFM_CUDA_CHECK((launch_gemm<false, true>(probe, e, st))); }
    const int nz = (n + kper - 1) / kper;
    splitk_reduce_kernel<<<ceil_div((long long)in * out, 256), 256, 0, st>>>((long long)in * out, nz, (long long)in * out, splitbuf, dW);
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}

// dX[n,in] = (D[n,out] * W^T) gated by mask, optionally + add       (W stored [in,out])
// cs_part (optional): [ceil(n / 32)][in] scratch; when the product runs on the scaled-fp16 kernel its epilogue also leaves the
// per-32-row column sums of dX there (*cs_done = true) - dX is the back-propagated signal whose column sum is a bias gradient
static int dgrad(int n, int in, int out, const float* D, long long ldd, const float* W, float* dX, long long ldx,
                 const float* mask, long long ldm, const float* add, long long ldadd, cudaStream_t st, DenseAmax am = DenseAmax(),
                 float* cs_part = nullptr, bool* cs_done = nullptr) {
    GemmShape p{n, in, out, D, ldd, W, (long long)out, nullptr};
    p.a_amax = am.a; p.a_split = am.a_split; p.a_scale_src = am.a_scale_src;
    const bool general = am.mask_mul != 0;      // gates are activation derivatives: the ACT = true functors
    if (cs_done) *cs_done = false;
    if (am.out_split && am.w_norm && am.a) {
        // dX also leaves pre-split for the backward-data layer that consumes it (EpiStdS; the bound uses the kernel's ROW norm)
        auto run = [&](auto e) -> cudaError_t {
            e.amax_out = am.out; e.mask_mul = am.mask_mul;
            if constexpr (decltype(e)::kColSum) { e.colsum_part = cs_part; e.ldcs = in; }
            return launch_gemm<true, false>(p, e, st);
        };
        if (general) MFM_CUDA_CHECK(run(EpiStdSA{dX, ldx, nullptr, mask, ldm, add, ldadd, 0, 1, am.out_split, am.a, nullptr, 0.0f, am.w_norm, nullptr, am.add_bound, am.out_bound}));
        else {
            EpiStdST<false, true> ec{dX, ldx, nullptr, mask, ldm, add, ldadd, 0, 1, am.out_split, am.a, nullptr, 0.0f, am.w_norm, nullptr, am.add_bound, am.out_bound};
            if (cs_part && cs_done && tc2h::gemm_h16() && gemm_backend() == 0 && gemm_path<true, false>(p) == 2 && tc2h::eligible(p, ec)) {
                MFM_CUDA_CHECK(run(ec));
                *cs_done = true;
            } else
                MFM_CUDA_CHECK(run(EpiStdS{dX, ldx, nullptr, mask, ldm, add, ldadd, 0, 1, am.out_split, am.a, nullptr, 0.0f, am.w_norm, nullptr, am.add_bound, am.out_bound}));
        }
        return MFM_OK;
    }
    auto run = [&](auto e) -> cudaError_t { e.amax_out = am.out; e.mask_mul = am.mask_mul; return launch_gemm<true, false>(p, e, st); };
    if (general) MFM_CUDA_CHECK(run(EpiStdA{dX, ldx, nullptr, mask, ldm, add, ldadd, 1.0f, 0}));
    else MFM_CUDA_CHECK(run(EpiStd{dX, ldx, nullptr, mask, ldm, add, ldadd, 1.0f, 0}));
    return MFM_OK;
}

struct FmBufs {
    FieldBufs B;
    float *times, *xt, *target, *v, *delta, *dgt, *d6, *d5, *dcat, *d2, *d0, *blockpart, *splitbuf, *colpart;
    float *d6_s, *d5_s, *dcat_s;      // pre-split copies of the back-propagated signals (A operands of the next backward-data layer)
    float* cspart;                    // [ceil(n / 32)][H] column-sum partials written by the backward-data epilogues
    float *d2_s, *d0_s, *xt_s, *delta_s, *dgt_s;   // ... and of the tensors only the weight gradients read in that form
    size_t splitbuf_floats;
};

static const int FM_LOSS_BLOCKS = 1024;

static size_t fm_splitbuf_floats(const mfm_field_t& F) {
    const size_t H = F.hidden, d = F.dim, Fd = F.fourier_dim;
    size_t m = 2 * H * H;
    if (d * H > m) m = d * H;
    if (2 * Fd * H > m) m = 2 * Fd * H;
    return m * 16;     // room for 16 batch slices of the largest layer (more for smaller ones)
}

static size_t fm_bytes(const mfm_field_t& F, const mfm_target_t& T, int n) {
    const size_t H = F.hidden, d = F.dim, N = n;
    return field_bufs_bytes(F, T, n, true) + ws_slice(N, 4) + ws_slice(N * d, 4) * 5 + ws_slice(N * H, 4) * 4 +
           ws_slice(N * 2 * H, 4) + ws_slice(FM_LOSS_BLOCKS, 4) + ws_slice(fm_splitbuf_floats(F), 4) +
           ws_slice((size_t)COLSUM_SLABS * (H > d ? H : d), 4) + ws_slice(N * H, 4) * 4 + ws_slice(N * 2 * H, 4) + ws_slice(N * d, 4) * 3 + ws_slice(((N + 31) / 32) * H, 4) + 1024;
}

static bool fm_take(FmBufs& M, Workspace& w, const mfm_field_t& F, int n, const mfm_target_t* T) {
    const size_t H = F.hidden, d = F.dim, N = n;
    field_bufs_take(M.B, w, F, n, true, T);
    M.times = w.take<float>(N);
    M.xt = w.take<float>(N * d); M.target = w.take<float>(N * d); M.v = w.take<float>(N * d);
    M.delta = w.take<float>(N * d); M.dgt = w.take<float>(N * d);
    M.d6 = w.take<float>(N * H); M.d5 = w.take<float>(N * H); M.d2 = w.take<float>(N * H); M.d0 = w.take<float>(N * H);
    M.dcat = w.take<float>(N * 2 * H);
    M.blockpart = w.take<float>(FM_LOSS_BLOCKS);
    M.colpart = w.take<float>((size_t)COLSUM_SLABS * (H > d ? H : d));
    M.splitbuf_floats = fm_splitbuf_floats(F);
    M.splitbuf = w.take<float>(M.splitbuf_floats);
    M.d6_s = w.take<float>(N * H); M.d5_s = w.take<float>(N * H); M.dcat_s = w.take<float>(N * 2 * H);
    M.d2_s = w.take<float>(N * H); M.d0_s = w.take<float>(N * H);
    M.xt_s = w.take<float>(N * d); M.delta_s = w.take<float>(N * d); M.dgt_s = w.take<float>(N * d);
    M.cspart = w.take<float>(((N + 31) / 32) * H);
    return w.ok;
}

#define W_(i) (F.params + F.w_off[i])
#define GW_(i) (grads + F.w_off[i])
#define GB_(i) (grads + F.b_off[i])

// Second stream for the weight gradients.  dW_l needs only the layer's input and the back-propagated signal G_l, nothing downstream
// needs dW_l: issued on their own stream they fill the SM pairs a backward-data GEMM's last, partial wave of tiles leaves idle
// (at 8 192 chains a 1024-wide layer is 128 tiles on 74 pairs) and vice versa.  Same kernels, same arithmetic, same results;
// each weight gradient waits for everything issued on the main stream before it, the call joins the streams before it returns.
// Off while the main stream is being captured into a graph and for short batches (MFM_FM_STREAMS=0|1 overrides).
struct FmAux { cudaStream_t s = nullptr; cudaEvent_t fork[12] = {}; cudaEvent_t join = nullptr; bool ok = false; };
static FmAux* fm_aux() {
    static FmAux aux[16];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
    FmAux& a = aux[dev];
    if (!a.ok) {
        if (cudaStreamCreateWithFlags(&a.s, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        for (int i = 0; i < 12; ++i) if (cudaEventCreateWithFlags(&a.fork[i], cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        if (cudaEventCreateWithFlags(&a.join, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        a.ok = true;
    }
    return &a;
}

// part 0: everything; part 1: forward, loss and the gradients of layers 7..4 (the tail [w_off[4], n_params) of
// the flat buffer); part 2: the gradients of layers 3..0 (the head) from the activations part 1 left in
// the workspace.  The split lets the host all-reduce the tail while part 2 runs.
// xt_amax: slot holding max |x_t| when the batch kernel tracked it (null: field_eval reduces it).
static int fm_forward_backward(const mfm_field_t& F, const mfm_target_t& T, int n, FmBufs& M, float* loss_out,
                               float* grads, cudaStream_t st, int part, const float* xt_amax = nullptr, bool tgt_tracked = false) {
    const int d = F.dim, H = F.hidden, Fd = F.fourier_dim;
    FieldBufs& B = M.B;
    int rc;
    if (part == 2) field_register_mirrors(F, B);      // built by part 1 in this workspace
    // tensor maxima of the backward pass (AmaxSlot; null when the scaled-fp16 GEMM is off)
    float* am = tc2h::gemm_h16() ? B.amax : nullptr;
    auto slot = [&](int i) -> float* { return am ? am + i : nullptr; };
    // weight gradients from the split16 copies (gemm_tcgen05_wgrad16.cuh): same conditions as the copies' producers
    static const bool no_wsplit = getenv("MFM_H16_NOWGRAD") != nullptr;
    static const bool no_split = getenv("MFM_H16_NOSPLIT") != nullptr;
    const bool wsp = !no_wsplit && !no_split && am != nullptr && M.d6_s != nullptr && B.h0_s != nullptr && H % 16 == 0 && (2 * Fd) % 16 == 0 && n >= 256 &&
                     ((reinterpret_cast<uintptr_t>(B.h0_s) | reinterpret_cast<uintptr_t>(B.cat_s)) & 63) == 0;
    const bool wspd = wsp && d % 16 == 0;      // the [n, d] operands have copies too
    // the loss kernel writes delta / dgt pre-split itself when it can bound them beforehand (tracked maxima of v and of the
    // targets, a clipped score): no separate passes, and the two backward-data layers that read them load the copies
    static const bool no_fused_loss = getenv("MFM_FM_NOFUSEDLOSS") != nullptr;
    const bool fused_loss = !no_fused_loss && wspd && tgt_tracked && xt_amax != nullptr && F.grad_clip > 0.0f;
    // scale sources of the delta / dgt copies: their bounds (fused) or their exact maxima (separate passes)
    const float* delta_src = fused_loss ? am + AM_BOUND + AM_DELTA : slot(AM_DELTA);
    const float* dgt_src = fused_loss ? am + AM_BOUND + AM_DGT : slot(AM_DGT);
    // max |x_t|: the batch kernel's slot, or the one field_eval reduces into when d is a multiple of 16 (else untracked: no h2 copy)
    const float* xa_src = xt_amax ? xt_amax : (d % 16 == 0 ? slot(AM_X) : nullptr);
    if (part != 2) {
        MFM_CUDA_CHECK(cudaMemsetAsync(grads, 0, (size_t)F.n_params * sizeof(float), st));
        if ((rc = field_prepare_weights(F, B, st))) return rc;
        // x_t leaves the batch kernel with its exact maximum: its split16 copy (the weight gradient of Dense_2 needs it anyway) is
        // made first, so that the two GEMMs that read x_t - Dense_2 and the pines K^-1 product - load it pre-split too
        const bool xt_pre = wspd && xt_amax != nullptr;
        if (xt_pre && (rc = presplit_weights(M.xt, M.xt_s, (long long)n * d, xt_amax, st))) return rc;
        B.v_amax = fused_loss ? slot(AM_V) : nullptr;
        if ((rc = field_eval(F, T, n, M.xt, M.times, nullptr, 1.0f, M.v, nullptr, B, st, nullptr, nullptr, xt_amax, xt_pre ? M.xt_s : nullptr))) return rc;
        B.v_amax = nullptr;
        const long long tot = (long long)n * d;
        const int lb = (int)((tot + 255) / 256 < FM_LOSS_BLOCKS ? (tot + 255) / 256 : FM_LOSS_BLOCKS);
        if (fused_loss)
            fm_loss_delta_split_kernel<<<lb, 256, 0, st>>>(tot / 4, reinterpret_cast<const float4*>(M.v), reinterpret_cast<const float4*>(M.target),
                                                           reinterpret_cast<const float4*>(B.gc), reinterpret_cast<float4*>(M.delta), reinterpret_cast<float4*>(M.dgt),
                                                           M.blockpart, slot(AM_DELTA), slot(AM_DGT), slot(AM_V), slot(AM_TGT), F.grad_clip,
                                                           M.delta_s, M.dgt_s, am + AM_BOUND + AM_DELTA, am + AM_BOUND + AM_DGT);
        else
            fm_loss_delta_kernel<<<lb, 256, 0, st>>>(tot, M.v, M.target, B.gc, M.delta, M.dgt, M.blockpart, slot(AM_DELTA), slot(AM_DGT));
        MFM_LAUNCH_CHECK();
        final_sum_kernel<<<1, 256, 0, st>>>(lb, M.blockpart, loss_out);
        MFM_LAUNCH_CHECK();
        // split16 copies of the [n, d] operands of the weight gradients of layers 2, 7 and 4 (their maxima are exact only now:
        // one element-wise pass each, 8 B per element)
        if (wspd) {
            if (!xt_pre && (rc = presplit_weights(M.xt, M.xt_s, tot, xa_src, st))) return rc;
            if (!fused_loss) {
                if ((rc = presplit_weights(M.delta, M.delta_s, tot, slot(AM_DELTA), st))) return rc;
                if ((rc = presplit_weights(M.dgt, M.dgt_s, tot, slot(AM_DGT), st))) return rc;
            }
        }
    }
    auto bias_grad = [&](const float* a, long long lda, int cols, float* out) -> int {
        if (n < 8 * COLSUM_SLABS) {             // few rows: one launch
            colsum_blocks_kernel<<<ceil_div(cols, 32), 256, 0, st>>>(n, cols, a, lda, out);
            MFM_LAUNCH_CHECK();
            return MFM_OK;
        }
        const int slabs = COLSUM_SLABS;
        colsum_partial_kernel<<<dim3(ceil_div(cols, 32), slabs), 256, 0, st>>>(n, cols, a, lda, M.colpart);
        MFM_LAUNCH_CHECK();
        colsum_final_kernel<<<ceil_div(cols, 256), 256, 0, st>>>(cols, slabs, M.colpart, out);
        MFM_LAUNCH_CHECK();
        return MFM_OK;
    };
    // ... or from the per-32-row partials a backward-data epilogue left in M.cspart (cs == true), else from the tensor itself
    auto bias_grad_cs = [&](bool cs, const float* a, long long lda, int cols, float* out) -> int {
        if (!cs) return bias_grad(a, lda, cols, out);
        const int nb = (n + 31) / 32;
        if (nb <= 8 * COLSUM_SLABS) {           // few partial rows: one launch
            colsum_blocks_kernel<<<ceil_div(cols, 32), 256, 0, st>>>(nb, cols, M.cspart, cols, out);
            MFM_LAUNCH_CHECK();
            return MFM_OK;
        }
        colsum_partial_kernel<<<dim3(ceil_div(cols, 32), COLSUM_SLABS), 256, 0, st>>>(nb, cols, M.cspart, cols, M.colpart);
        MFM_LAUNCH_CHECK();
        colsum_final_kernel<<<ceil_div(cols, 256), 256, 0, st>>>(cols, COLSUM_SLABS, M.colpart, out);
        MFM_LAUNCH_CHECK();
        return MFM_OK;
    };
    bool cs6 = false, cs5 = false, csx = false, cst = false, cs2 = false, cs0 = false;
    float* sb = M.splitbuf; const size_t sbf = M.splitbuf_floats;
    // pre-split copies along the backward-data chain (as in field_eval): slot ids of the exact maxima / bounds, ROW norms of the kernels
    const bool sp = am != nullptr && M.d6_s != nullptr && H % 16 == 0 && n >= 256;
    auto BD = [&](int i) -> float* { return am + AM_BOUND + i; };
    auto WR = [&](int l) -> const float* { return am + AM_WNORM_ROW + l; };
    // (exact max of D, [D pre-split, slot of its scale]) -> exact max of dX [, dX pre-split, slot of its bound, layer, bound of `add`]
    auto G_ = [&](const float* a, const float* a_split, const float* src, float* out, float* c_split, int slot_id, int layer, const float* add_bound) {
        DenseAmax m; m.a = a; m.out = out;
        m.mask_mul = F.act != MFM_ACT_RELU ? 1 : 0;       // gates are activation derivatives (B.d*) instead of output signs
        if (sp && a_split) { m.a_split = a_split; m.a_scale_src = src; }
        if (sp && c_split) { m.out_split = c_split; m.out_bound = BD(slot_id); m.w_norm = WR(layer); m.add_bound = add_bound; }
        return m;
    };
    const bool dmul = F.act != MFM_ACT_RELU;
    const float* g_h0 = dmul ? B.dh0 : B.h0; const float* g_h2 = dmul ? B.dh2 : B.h2; const float* g_cat = dmul ? B.dcat : B.cat;
    const float* g_h5 = dmul ? B.dh5 : B.h5; const float* g_h6 = dmul ? B.dh6 : B.h6;
    auto WS_ = [&](bool on, const float* a_s, const float* a_src, const float* g_s, const float* g_src) {
        WgradSplit w; if (on) { w.a_s = a_s; w.a_src = a_src; w.g_s = g_s; w.g_src = g_src; } return w;
    };
    // weight gradients on the second stream (see FmAux)
    static const int streams_env = getenv("MFM_FM_STREAMS") ? atoi(getenv("MFM_FM_STREAMS")) : -1;
    FmAux* aux = nullptr;
    {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        const bool capturing = cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone;
        if (!capturing && (streams_env > 0 || (streams_env < 0 && n >= 1024))) aux = fm_aux();
    }
    cudaStream_t sw = aux ? aux->s : st;
    int n_fork = 0;
    auto fork_w = [&]() -> int {          // the next weight gradient may start once everything issued on st so far has finished
        if (!aux) return MFM_OK;
        cudaEvent_t e = aux->fork[n_fork++ % 12];
        MFM_CUDA_CHECK(cudaEventRecord(e, st));
        MFM_CUDA_CHECK(cudaStreamWaitEvent(sw, e, 0));
        return MFM_OK;
    };
    auto join_w = [&]() -> int {          // ... and the caller's stream continues only after the last one
        if (!aux) return MFM_OK;
        MFM_CUDA_CHECK(cudaEventRecord(aux->join, sw));
        MFM_CUDA_CHECK(cudaStreamWaitEvent(st, aux->join, 0));
        return MFM_OK;
    };
    if (part != 2) {
    // layer 7 (nn_xt head): y = h6 W7 + b7
    if ((rc = fork_w())) return rc;
    if ((rc = wgrad(n, H, d, B.h6, H, M.delta, d, GW_(7), sb, sbf, sw, WS_(wspd, B.h6_s, BD(AM_H6), M.delta_s, delta_src)))) return rc;
    if ((rc = bias_grad(M.delta, d, d, GB_(7)))) return rc;
    if ((rc = dgrad(n, H, d, M.delta, d, W_(7), M.d6, H, g_h6, H, nullptr, 0, st, G_(slot(AM_DELTA), fused_loss ? M.delta_s : nullptr, delta_src, slot(AM_D6), M.d6_s, AM_D6, 7, nullptr), M.cspart, &cs6))) return rc;
    if ((rc = bias_grad_cs(cs6, M.d6, H, H, GB_(6)))) return rc;        // bias gradients: column sums of the signal just written
    // layer 6
    if ((rc = fork_w())) return rc;
    if ((rc = wgrad(n, H, H, B.h5, H, M.d6, H, GW_(6), sb, sbf, sw, WS_(wsp, B.h5_s, BD(AM_H5), M.d6_s, BD(AM_D6))))) return rc;
    if ((rc = dgrad(n, H, H, M.d6, H, W_(6), M.d5, H, g_h5, H, nullptr, 0, st, G_(slot(AM_D6), M.d6_s, BD(AM_D6), slot(AM_D5), M.d5_s, AM_D5, 6, nullptr), M.cspart, &cs5))) return rc;
    if ((rc = bias_grad_cs(cs5, M.d5, H, H, GB_(5)))) return rc;
    // layer 5 (joint, input cat = [s_x | s_t])
    if ((rc = fork_w())) return rc;
    if ((rc = wgrad(n, 2 * H, H, B.cat, 2 * H, M.d5, H, GW_(5), sb, sbf, sw, WS_(wsp, B.cat_s, BD(AM_SX), M.d5_s, BD(AM_D5))))) return rc;
    // d s_x = (d5 W5[:H]^T) * relu'(s_x)
    if ((rc = dgrad(n, H, H, M.d5, H, W_(5), M.dcat, 2 * H, g_cat, 2 * H, nullptr, 0, st, G_(slot(AM_D5), M.d5_s, BD(AM_D5), slot(AM_DCX), M.dcat_s, AM_DCX, 5, nullptr), M.cspart, &csx))) return rc;
    if ((rc = bias_grad_cs(csx, M.dcat, 2 * H, H, GB_(3)))) return rc;  // (layer 3's bias; its slot lies in the head of the flat buffer, which nobody reads before part 2 ends)
    // d s_t (joint part) = d5 W5[H:]^T   (no gate yet; its bound enters the next layer's through `add`)
    if ((rc = dgrad(n, H, H, M.d5, H, W_(5) + (long long)H * H, M.dcat + H, 2 * H, nullptr, 0, nullptr, 0, st,
                    G_(slot(AM_D5), M.d5_s, BD(AM_D5), nullptr, M.dcat_s + H, AM_DCT0, 5, nullptr)))) return rc;
    // layer 4 (nn_t head): g_t = s_t W4 + b4, dL/dg_t = delta * clip(grad logprob)
    if ((rc = fork_w())) return rc;
    if ((rc = wgrad(n, H, d, B.cat + H, 2 * H, M.dgt, d, GW_(4), sb, sbf, sw, WS_(wspd, B.cat_s + H, BD(AM_ST), M.dgt_s, dgt_src)))) return rc;
    if ((rc = bias_grad(M.dgt, d, d, GB_(4)))) return rc;
    // d s_t = (dgt W4^T + joint part) * relu'(s_t)   (in place)
    if ((rc = dgrad(n, H, d, M.dgt, d, W_(4), M.dcat + H, 2 * H, g_cat + H, 2 * H, M.dcat + H, 2 * H, st,
                    G_(slot(AM_DGT), fused_loss ? M.dgt_s : nullptr, dgt_src, slot(AM_DCT), M.dcat_s + H, AM_DCT, 4, sp ? BD(AM_DCT0) : nullptr), M.cspart, &cst))) return rc;
    if ((rc = bias_grad_cs(cst, M.dcat + H, 2 * H, H, GB_(1)))) return rc;
    }
    if (part == 1) return join_w();
    // layer 3 (x branch)
    if ((rc = fork_w())) return rc;
    if ((rc = wgrad(n, H, H, B.h2, H, M.dcat, 2 * H, GW_(3), sb, sbf, sw, WS_(wsp && xa_src, B.h2_s, BD(AM_H2), M.dcat_s, BD(AM_DCX))))) return rc;
    if ((rc = dgrad(n, H, H, M.dcat, 2 * H, W_(3), M.d2, H, g_h2, H, nullptr, 0, st, G_(slot(AM_DCX), M.dcat_s, BD(AM_DCX), slot(AM_D2), wsp ? M.d2_s : nullptr, AM_D2, 3, nullptr), M.cspart, &cs2))) return rc;
    if ((rc = bias_grad_cs(cs2, M.d2, H, H, GB_(2)))) return rc;
    // layer 2
    if ((rc = fork_w())) return rc;
    if ((rc = wgrad(n, d, H, M.xt, d, M.d2, H, GW_(2), sb, sbf, sw, WS_(wspd && xa_src, M.xt_s, xa_src, M.d2_s, BD(AM_D2))))) return rc;
    // layer 1 (time branch)
    if ((rc = fork_w())) return rc;
    if ((rc = wgrad(n, H, H, B.h0, H, M.dcat + H, 2 * H, GW_(1), sb, sbf, sw, WS_(wsp, B.h0_s, BD(AM_H0), M.dcat_s + H, BD(AM_DCT))))) return rc;
    if ((rc = dgrad(n, H, H, M.dcat + H, 2 * H, W_(1), M.d0, H, g_h0, H, nullptr, 0, st, G_(slot(AM_DCT), M.dcat_s + H, BD(AM_DCT), slot(AM_D0), wsp ? M.d0_s : nullptr, AM_D0, 1, nullptr), M.cspart, &cs0))) return rc;
    if ((rc = bias_grad_cs(cs0, M.d0, H, H, GB_(0)))) return rc;
    // layer 0
    if ((rc = fork_w())) return rc;
    if ((rc = wgrad(n, 2 * Fd, H, B.ff, 2 * Fd, M.d0, H, GW_(0), sb, sbf, sw, WS_(wsp, B.ff_s, BD(AM_FF), M.d0_s, BD(AM_D0))))) return rc;
    return join_w();
}

// ---------------------------------------------------------------------------------------------
// optimizer
// ---------------------------------------------------------------------------------------------
// scratch[0] = number of non-finite gradient entries
__global__ void finite_check_kernel(long long n, const float* __restrict__ g, int* __restrict__ scratch) {
    int bad = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        bad |= !isfinite(g[i]);
    bad = __any_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && bad) atomicAdd(scratch, 1);
}

// opt_state: [adam count, notfinite_count, total_notfinite, last_finite, scratch(nonfinite), apply flag]
__global__ void opt_decide_kernel(int* __restrict__ st, int max_err) {
    if (threadIdx.x != 0) return;
    const bool finite = st[4] == 0;
    const int nf = finite ? 0 : st[1] + 1;                 // notfinite_count
    st[1] = nf;
    if (!finite) st[2] += 1;                               // total_notfinite
    st[3] = finite ? 1 : 0;                                // last_finite
    st[5] = (finite || nf > max_err) ? 1 : 0;              // apply the inner update?
}

__global__ void __launch_bounds__(256)
adamw_kernel(long long n, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ mu,
             float* __restrict__ nu, const uint8_t* __restrict__ decay, const int* __restrict__ st, float lr_base,
             int lr_total, int lr_warmup, float b1, float b2, float eps, float wd, float clip) {
    if (st[5] == 0) return;                                // rejected update: params and moments untouched
    const int count = st[0];
    const float c1 = (float)(count + 1);
    const float bc1 = 1.0f - powf(b1, c1), bc2 = 1.0f - powf(b2, c1);
    // join_schedules([linear_schedule(0 -> lr, warmup), linear_schedule(lr -> 0, total - warmup)], [warmup])  (:189-198);
    // optax.linear_schedule: (init - end) * (1 - clip(count, 0, steps) / steps) + end, the constant init for steps <= 0
    float lr;
    if (count < lr_warmup) {
        const int cc = count < 0 ? 0 : count;
        lr = (0.0f - lr_base) * (1.0f - (float)cc / (float)lr_warmup) + lr_base;
    } else {
        const int steps = lr_total - lr_warmup;
        int cc = count - lr_warmup; cc = cc < 0 ? 0 : (cc > steps ? steps : cc);
        lr = steps > 0 ? lr_base * (1.0f - (float)cc / (float)steps) : lr_base;
    }
    const float omb1 = 1.0f - b1, omb2 = 1.0f - b2;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float gi = g[i];
        const float m = omb1 * gi + b1 * mu[i];
        const float v = omb2 * gi * gi + b2 * nu[i];
        mu[i] = m; nu[i] = v;
        float u = (m / bc1) / (sqrtf(v / bc2) + eps);
        const float pi = p[i];
        if (decay[i]) u += wd * pi;
        u = -lr * u;
        u = fminf(fmaxf(u, -clip), clip);                  // optax.clip on the update
        p[i] = pi + u;
    }
}

__global__ void opt_advance_kernel(int* __restrict__ st) {
    if (threadIdx.x == 0 && st[5]) st[0] += 1;
}

}  // namespace mfm

extern "C" {
using namespace mfm;

size_t mfm_fm_workspace_bytes(const mfm_field_t* f, const mfm_target_t* t, int n) { return fm_bytes(*f, *t, n); }

// samples_ref: the call draws x0 from the reference distribution (the conditional batch)
static int fm_check(const mfm_field_t* f, const mfm_target_t* t, bool samples_ref = false) {
    if (!f || !t) { mfm_set_last_error_msg("null descriptor"); return MFM_ERR_ARG; }
    if (f->dim != t->dim) { mfm_set_last_error_msg("field.dim != target.dim"); return MFM_ERR_ARG; }
    return ref_check(f, samples_ref);
}

int mfm_fm_loss_grad(const mfm_field_t* f, const mfm_target_t* t, const uint32_t* rng_key, int n, int chain_offset,
                     int n_total, float sigma, const float* positions, float* loss_out, float* grads, void* ws,
                     size_t ws_bytes, mfm_stream_t stream) {
    mfm::CrossScope cross_scope;
    return mfm_fm_loss_grad_part(f, t, rng_key, n, chain_offset, n_total, sigma, positions, loss_out, grads, ws, ws_bytes, 0, stream);
}

int mfm_fm_loss_grad_part(const mfm_field_t* f, const mfm_target_t* t, const uint32_t* rng_key, int n, int chain_offset,
                          int n_total, float sigma, const float* positions, float* loss_out, float* grads, void* ws,
                          size_t ws_bytes, int part, mfm_stream_t stream) {
    mfm::CrossScope cross_scope;
    int rc = fm_check(f, t, true);
    if (rc) return rc;
    if (part < 0 || part > 2) { mfm_set_last_error_msg("part must be 0, 1 or 2"); return MFM_ERR_ARG; }
    if (!rng_key || !positions || !loss_out || !grads) { mfm_set_last_error_msg("null argument"); return MFM_ERR_ARG; }
    if (n <= 0) return MFM_OK;
    if (n_total < chain_offset + n || chain_offset < 0) { mfm_set_last_error_msg("bad chain_offset/n_total"); return MFM_ERR_ARG; }
    if ((long long)n_total * f->dim * (mfm::rng_x64() ? 2 : 1) > 0xFFFFFFFFll) { mfm_set_last_error_msg("n_total*d exceeds the 32-bit counter space"); return MFM_ERR_UNSUPPORTED; }
    Workspace w(ws, ws_bytes);
    FmBufs M;
    if (!fm_take(M, w, *f, n, t)) { mfm_set_last_error_msg("workspace too small (mfm_fm_loss_grad)"); return MFM_ERR_WORKSPACE; }
    float* xt_amax = (mfm::tc2h::gemm_h16() && M.B.amax) ? M.B.amax + AM_X : nullptr;
    if (part != 2) {
        if (M.B.amax) MFM_CUDA_CHECK(cudaMemsetAsync(M.B.amax + AM_EVAL_END, 0, (AM_POOL - AM_EVAL_END) * sizeof(float), stream));   // this pass's maxima
        if (f->ref_kind == MFM_REF_PHI4_BASE) {
            const int wpb = band_warps_per_block(f->dim);
            fm_batch_phi4_kernel<<<ceil_div(n, wpb), 32 * wpb, (size_t)wpb * band_row_floats(f->dim) * sizeof(float), stream>>>(
                rng_key, n, chain_offset, n_total, f->dim, sigma, f->ref_band, positions, M.times, M.xt, M.target, xt_amax, rng_x64());
        } else {
            fm_batch_kernel<<<ceil_div(n, 8), 256, 0, stream>>>(rng_key, n, chain_offset, n_total, f->dim, sigma, f->ref_mean, f->ref_std,
                                                                 positions, M.times, M.xt, M.target, xt_amax, rng_x64());
        }
        MFM_LAUNCH_CHECK();
    }
    return fm_forward_backward(*f, *t, n, M, loss_out, grads, stream, part, xt_amax, xt_amax != nullptr);   // fm_batch_kernel tracks max |target| too
}

int mfm_fm_loss_grad_uncond(const mfm_field_t* f, const mfm_target_t* t, const uint32_t* rng_key, int n, int chain_offset,
                            int n_total, float sigma, const float* positions, float* loss_out, float* grads, void* ws,
                            size_t ws_bytes, mfm_stream_t stream) {
    mfm::CrossScope cross_scope;
    int rc = fm_check(f, t);
    if (rc) return rc;
    if (!rng_key || !positions || !loss_out || !grads) { mfm_set_last_error_msg("null argument"); return MFM_ERR_ARG; }
    if (n <= 0) return MFM_OK;
    if (n_total < chain_offset + n || chain_offset < 0) { mfm_set_last_error_msg("bad chain_offset/n_total"); return MFM_ERR_ARG; }
    if ((long long)n_total * f->dim * (mfm::rng_x64() ? 2 : 1) > 0xFFFFFFFFll) { mfm_set_last_error_msg("n_total*d exceeds the 32-bit counter space"); return MFM_ERR_UNSUPPORTED; }
    Workspace w(ws, ws_bytes);
    FmBufs M;
    if (!fm_take(M, w, *f, n, t)) { mfm_set_last_error_msg("workspace too small (mfm_fm_loss_grad_uncond)"); return MFM_ERR_WORKSPACE; }
    float* xt_amax = (mfm::tc2h::gemm_h16() && M.B.amax) ? M.B.amax + AM_X : nullptr;
    if (M.B.amax) MFM_CUDA_CHECK(cudaMemsetAsync(M.B.amax + AM_EVAL_END, 0, (AM_POOL - AM_EVAL_END) * sizeof(float), stream));
    fm_batch_uncond_kernel<<<ceil_div(n, 8), 256, 0, stream>>>(rng_key, n, chain_offset, n_total, f->dim, sigma, positions,
                                                                M.times, M.xt, M.target, xt_amax, rng_x64());
    MFM_LAUNCH_CHECK();
    return fm_forward_backward(*f, *t, n, M, loss_out, grads, stream, 0, xt_amax);
}

int mfm_fm_loss_grad_from_batch(const mfm_field_t* f, const mfm_target_t* t, int n, const float* xt, const float* times,
                                const float* target_v, float* loss_out, float* grads, void* ws, size_t ws_bytes,
                                mfm_stream_t stream) {
    mfm::CrossScope cross_scope;
    int rc = fm_check(f, t);
    if (rc) return rc;
    if (!xt || !times || !target_v || !loss_out || !grads) { mfm_set_last_error_msg("null argument"); return MFM_ERR_ARG; }
    if (n <= 0) return MFM_OK;
    Workspace w(ws, ws_bytes);
    FmBufs M;
    if (!fm_take(M, w, *f, n, t)) { mfm_set_last_error_msg("workspace too small (mfm_fm_loss_grad_from_batch)"); return MFM_ERR_WORKSPACE; }
    const size_t nd = (size_t)n * f->dim * sizeof(float);
    MFM_CUDA_CHECK(cudaMemcpyAsync(M.xt, xt, nd, cudaMemcpyDeviceToDevice, stream));
    MFM_CUDA_CHECK(cudaMemcpyAsync(M.target, target_v, nd, cudaMemcpyDeviceToDevice, stream));
    MFM_CUDA_CHECK(cudaMemcpyAsync(M.times, times, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    if (M.B.amax) MFM_CUDA_CHECK(cudaMemsetAsync(M.B.amax + AM_EVAL_END, 0, (AM_POOL - AM_EVAL_END) * sizeof(float), stream));
    return fm_forward_backward(*f, *t, n, M, loss_out, grads, stream, 0);     // the caller's x_t: field_eval reduces its maximum
}

int mfm_adamw_step(float* params, const float* grads, float* mu, float* nu, const uint8_t* decay_mask, long long n_params,
                   int* opt_state, float lr_base, int lr_total_steps, int lr_warmup_steps, float b1, float b2, float eps, float weight_decay,
                   float clip, int max_consecutive_errors, mfm_stream_t stream) {
    if (!params || !grads || !mu || !nu || !decay_mask || !opt_state || n_params <= 0 || lr_total_steps <= 0 || lr_warmup_steps < 0 ||
        lr_warmup_steps > lr_total_steps) {
        mfm_set_last_error_msg("bad argument (mfm_adamw_step)"); return MFM_ERR_ARG;
    }
    MFM_CUDA_CHECK(cudaMemsetAsync(opt_state + 4, 0, 2 * sizeof(int), stream));
    const int blocks = (int)((n_params + 255) / 256 < 1184 ? (n_params + 255) / 256 : 1184);
    finite_check_kernel<<<blocks, 256, 0, stream>>>(n_params, grads, opt_state + 4);
    MFM_LAUNCH_CHECK();
    opt_decide_kernel<<<1, 32, 0, stream>>>(opt_state, max_consecutive_errors);
    MFM_LAUNCH_CHECK();
    adamw_kernel<<<blocks, 256, 0, stream>>>(n_params, params, grads, mu, nu, decay_mask, opt_state, lr_base,
                                             lr_total_steps, lr_warmup_steps, b1, b2, eps, weight_decay, clip);
    MFM_LAUNCH_CHECK();
    opt_advance_kernel<<<1, 32, 0, stream>>>(opt_state);
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}

}  // extern "C"

/* Test hook of the scaled-fp16 weight-gradient kernel (not in the ABI header): dW[in,out] = A^T G with A [n,in], G [n,out];
 * a_s / g_s: scratch for the split16 copies (same sizes), slots: device float[2] receiving max|A|, max|G|;
 * use_split = 0 runs the 3xTF32 path on the fp32 operands instead. */
extern "C" int mfm_debug_wgrad16(int n, int in, int out, const float* A, const float* G, float* dW, float* a_s, float* g_s, float* slots,
                                 float* splitbuf, long long splitbuf_floats, int use_split, mfm_stream_t stream) {
    using namespace mfm;
    WgradSplit ws;
    if (use_split) {
        if (in % 16 || out % 16) { mfm_set_last_error_msg("mfm_debug_wgrad16: in / out must be multiples of 16"); return MFM_ERR_ARG; }
        if (use_split == 1) {            // (2: the copies are already there - timing runs)
            MFM_CUDA_CHECK(tc2h::launch_absmax(A, in, n, in, nullptr, slots, stream));
            MFM_CUDA_CHECK(tc2h::launch_absmax(G, out, n, out, nullptr, slots + 1, stream));
            int rc;
            if ((rc = presplit_weights(A, a_s, (long long)n * in, slots, stream))) return rc;
            if ((rc = presplit_weights(G, g_s, (long long)n * out, slots + 1, stream))) return rc;
        }
        ws.a_s = a_s; ws.a_src = slots; ws.g_s = g_s; ws.g_src = slots + 1;
        GemmShape p16{in, out, n, a_s, (long long)in, g_s, (long long)out, nullptr};
        if (!tc2w::eligible(p16)) { mfm_set_last_error_msg("mfm_debug_wgrad16: shape not eligible for the fp16 kernel"); return MFM_ERR_UNSUPPORTED; }
    }
    return wgrad(n, in, out, A, in, G, out, dW, splitbuf, (size_t)splitbuf_floats, stream, ws);
}
