// Fused CNF push / pull for the SMALL reference shapes (4-mode and the 16-mode mixture: d = 2, H = 128, 128 chains):
// ONE kernel launch integrates the augmented ODE from start to finish.
//
// What `north_star` describes as "a persistent ODE-integration kernel [that] integrates a CTA-tile of chains entirely
// on-chip": a CTA owns 16 chains (one m16 tensor-core row tile) and runs their whole adaptive Dormand-Prince solve -
// initial step size, the six stages, error control, accept / reject, dense output - without leaving the SM.  Chains are
// independent, so no grid-wide synchronisation exists; each chain keeps its own (t, dt, segment, counters) exactly as in
// the lock-step multi-kernel driver (flow.cu::ode_solve), which stays the path for large ensembles and wide fields.
// The ODE state, the seven stage slopes and every activation of the 8-layer MLP live in shared memory; the weights
// (462 KB for d = 2: more than one SM's shared memory, SURVEY F6) are streamed from L2 as mma.sync B fragments with a
// 128-k register prefetch.  Dense layers: 3xTF32 on mma.sync.m16n8k8 with the partial sums flushed to fp32 registers
// every 32 k (the arithmetic of gemm_tf32x3.cuh); the 16 warps split a layer's output columns, one n-tile of 8 each; the A
// operand is split into tf32 hi / lo planes once per layer.
// Forward-mode tangents (one Hutchinson probe, or the d basis tangents of the exact trace) reuse the same row tile, one
// pass per tangent.  Eligibility: all six hidden widths equal, H in {64, 128}, d <= 16, 2F <= 256, relu / tanh / elu (their derivatives follow from the
// stored outputs), the warp-per-chain targets (mixture, phi-four, Gaussian).
//
// Before: ~120 launches per Runge-Kutta iteration (1.4 ms each at 128 chains even from a CUDA-graph loop); now the whole
// solve is one launch (measured numbers: DESIGN.md section 7).
#pragma once

namespace mfm {
namespace small {

constexpr int CH = 16;                  // chains per CTA = rows of one m16 MMA tile
constexpr int NWARP = 16, NTHR = NWARP * 32;     // one n-tile of 8 output columns per warp (N = 128)
constexpr int DP = 16;                  // padded state dimension (d <= 16)
constexpr int LDH = 132;                // pitch of [16][<=128] buffers: pitch % 32 == 4 -> conflict-free A-fragment reads
constexpr int LDC = 260;                // pitch of [16][<=256] buffers

struct Args {
    mfm_field_t F; mfm_target_t T;
    int n, hutch, n_seg; float target[16]; float rtol, atol; int mxstep; float sgn;
    const float* y0; const float* z; float* y1; float* ldj; int* counters;
    const float* wt;      // the dense kernels transposed (FieldBufs::wt: layer i at wt + F.w_off[i], [out][in])
};

// shared-memory carve-up (floats)
struct Smem {
    float* big;      // [16][LDC]: Fourier features, later the two tangent buffers ta | tb ([16][LDH] each)
    uint32_t *ahi, *alo;   // [16][LDC] each: the tf32 hi / lo parts of the current layer's A operand (split once, read by all warps)
    float *h0, *h2, *h5, *h6, *zw2;      // [16][LDH]
    float* cat;      // [16][LDC] = [s_x | s_t]
    float *xi, *gt, *y7, *gc, *hx, *zs, *yx, *outx;   // [16][DP]
    float* kx;       // [7][16][DP]
    float *tf, *yl, *outl, *tt, *dt, *d1, *negdiv;    // [16]
    float* kl;       // [7][16]
    float* tscr;     // [NWARP][5][DP] scratch of the warp-per-chain target functions
    int *seg, *icount, *ntry;                          // [16]
};
constexpr int BIG = (CH * LDC > 2 * CH * LDH) ? CH * LDC : 2 * CH * LDH;     // Fourier features [16][LDC], later ta | tb
constexpr int SMEM_FLOATS = BIG + 3 * CH * LDC + 5 * CH * LDH + 8 * CH * DP + 7 * CH * DP + 7 * CH + 7 * CH + NWARP * 5 * DP + 3 * CH;
constexpr int SMEM_BYTES = SMEM_FLOATS * 4 + 64;

__device__ __forceinline__ Smem carve(float* p) {
    Smem s;
    s.big = p; p += BIG;
    s.ahi = reinterpret_cast<uint32_t*>(p); p += CH * LDC; s.alo = reinterpret_cast<uint32_t*>(p); p += CH * LDC;
    s.cat = p; p += CH * LDC;
    s.h0 = p; p += CH * LDH; s.h2 = p; p += CH * LDH; s.h5 = p; p += CH * LDH; s.h6 = p; p += CH * LDH; s.zw2 = p; p += CH * LDH;
    s.xi = p; p += CH * DP; s.gt = p; p += CH * DP; s.y7 = p; p += CH * DP; s.gc = p; p += CH * DP; s.hx = p; p += CH * DP;
    s.zs = p; p += CH * DP; s.yx = p; p += CH * DP; s.outx = p; p += CH * DP;
    s.kx = p; p += 7 * CH * DP;
    s.tf = p; p += CH; s.yl = p; p += CH; s.outl = p; p += CH; s.tt = p; p += CH; s.dt = p; p += CH; s.d1 = p; p += CH; s.negdiv = p; p += CH;
    s.kl = p; p += 7 * CH;
    s.tscr = p; p += NWARP * 5 * DP;
    s.seg = reinterpret_cast<int*>(p); p += CH; s.icount = reinterpret_cast<int*>(p); p += CH; s.ntry = reinterpret_cast<int*>(p); p += CH;
    return s;
}

// derivative of the activation from its stored OUTPUT (relu: sign; tanh: 1 - h^2; elu: h > 0 ? 1 : h + 1)
__device__ __forceinline__ float dact_from_output(int act, float h) {
    if (act == MFM_ACT_RELU) return h > 0.0f ? 1.0f : 0.0f;
    if (act == MFM_ACT_TANH) return 1.0f - h * h;
    return h > 0.0f ? 1.0f : h + 1.0f;
}

// hi = the operand's own bits (the tensor core ignores the 13 low mantissa bits of a tf32 operand: hi = trunc(x), measured in
// round 1), lo = rn_tf32(x - trunc(x)): one conversion per value instead of two
__device__ __forceinline__ void split_raw(float x, uint32_t& hi, uint32_t& lo) {
    hi = __float_as_uint(x);
    lo = f2tf32(x - __uint_as_float(hi & 0xFFFFE000u));
}

// out[16][N] = f(A[16][K] W[K][N] + bias):  f = activation (mode 0, act_code as gemm_tf32x3.cuh) or a gate by the derivative
// read off `gate` (mode 1: forward-mode tangent through that layer).  A, out, gate in shared memory; WT = the kernel TRANSPOSED
// ([N][ldwt], k contiguous: the copy field_prepare_weights builds for the tensor-core GEMMs).
// Block-wide (contains barriers).  The A operand is split into its tf32 hi / lo parts ONCE, cooperatively, into the ahi / alo
// planes (every warp needs the whole A tile: splitting in each warp tripled the instruction count of the k-loop); warp w then
// computes n-tile w, w + 16, ...  3xTF32 with the cross terms in their own accumulator (two independent MMA chains), partial
// sums flushed every 32 k.
// k is PERMUTED inside every block of 16: the contraction index is summed over, so any permutation applied to both operands is
// exact, and with thread t holding k = 4t .. 4t + 3 of a block (b0, b1 of two consecutive k-steps) its B fragments are ONE
// 16-byte load from the transposed kernel per 16 k instead of four scattered 4-byte loads; the planes are written in the
// matching order (position (v >> 1) * 8 + (v & 1) * 4 + u for k = 4u + v), from which ldmatrix delivers the A fragments.
// The fragments of the first 128 k are requested BEFORE the split pass and its barrier, and every register is refilled with the
// next batch's value right after its last use, so the L2 round trips overlap the arithmetic.
// Not inlined: eleven inlined copies of the two instantiations made the kernel 38 k instructions and the loop starved on
// instruction fetch (stall_no_inst was the top stall reason in the ncu capture).
template <int KN>       // k-steps of 8 per batch: 16 (K % 128 == 0) or 8 (K == 64)
__device__ __noinline__ void mma_layer_t(const float* __restrict__ As, int lda, int K, const float* __restrict__ WT, int ldwt, int N,
                                         const float* __restrict__ bias, int mode, int act, const float* gate, int ldg,
                                         float* out, int ldo, uint32_t* ahi, uint32_t* alo) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int n_tiles = N >> 3;
    float4 bq[KN / 2];                                     // [16-k block]: k = 4t .. 4t + 3 of column nt * 8 + g
    if (warp < n_tiles) {
        const float4* w = reinterpret_cast<const float4*>(WT + (long long)(warp * 8 + g) * ldwt) + t;
#pragma unroll
        for (int j = 0; j < KN / 2; ++j) bq[j] = __ldg(w + 4 * j);
    }
    const int lgK4 = 29 - __clz(K);                        // log2(K / 4); K is a power of two (eligible())
    for (int o = threadIdx.x; o < CH * (K >> 2); o += NTHR) {
        // four consecutive k = 4u .. 4u + 3 of one row: positions base + u + {0, 4, 8, 12} of the permuted planes
        const int r = o >> lgK4, k4 = (o & ((K >> 2) - 1)) << 2;
        const float4 v = *reinterpret_cast<const float4*>(As + r * lda + k4);
        const int base = r * LDC + (k4 & ~15) + ((k4 >> 2) & 3);
        uint32_t h, l;
        split_raw(v.x, h, l); ahi[base] = h; alo[base] = l;
        split_raw(v.y, h, l); ahi[base + 4] = h; alo[base + 4] = l;
        split_raw(v.z, h, l); ahi[base + 8] = h; alo[base + 8] = l;
        split_raw(v.w, h, l); ahi[base + 12] = h; alo[base + 12] = l;
    }
    __syncthreads();
    // A fragments by ldmatrix: an m16 x k8 tf32 tile is four 8 x 8 b16 matrices (rows 0-7 | 8-15) x (k 0-3 | 4-7); lane l supplies
    // the row address of matrix l / 8, and receives exactly the m16n8k8 fragment elements a0..a3
    const uint32_t frag_off = (uint32_t)((((lane & 7) + ((lane >> 3) & 1) * 8) * LDC + (lane >> 4) * 4) * 4);
    const uint32_t hi_base = (uint32_t)__cvta_generic_to_shared(ahi) + frag_off, lo_base = (uint32_t)__cvta_generic_to_shared(alo) + frag_off;
    for (int nt = warp; nt < n_tiles; nt += NWARP) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
        for (int kb = 0; kb < K; kb += KN * 8) {
            // what the registers are refilled with: the next batch of this n-tile, else the first batch of the warp's next n-tile
            const bool more_k = kb + KN * 8 < K, more = more_k || nt + NWARP < n_tiles;
            const float4* wn = reinterpret_cast<const float4*>(WT + (long long)((more_k ? nt : nt + NWARP) * 8 + g) * ldwt + (more_k ? kb + KN * 8 : 0)) + t;
#pragma unroll
            for (int kq = 0; kq < KN / 4; ++kq) {
                float pm[4] = {0.f, 0.f, 0.f, 0.f}, px[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const int ks = kq * 4 + kk;
                    const uint32_t ko = (uint32_t)(kb + ks * 8) * 4u;
                    uint32_t ah[4], al[4], bh[2], bl[2];
                    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(ah[0]), "=r"(ah[1]), "=r"(ah[2]), "=r"(ah[3]) : "r"(hi_base + ko));
                    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(al[0]), "=r"(al[1]), "=r"(al[2]), "=r"(al[3]) : "r"(lo_base + ko));
                    const float4 q = bq[ks >> 1];
                    split_raw((ks & 1) ? q.z : q.x, bh[0], bl[0]); split_raw((ks & 1) ? q.w : q.y, bh[1], bl[1]);
                    if ((ks & 1) && more) bq[ks >> 1] = __ldg(wn + 4 * (ks >> 1));
                    mma_tf32(px, al, bh); mma_tf32(pm, ah, bh); mma_tf32(px, ah, bl);
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[e] += pm[e] + px[e];
            }
        }
        const int c0 = nt * 8 + 2 * t;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int r = g + (e >> 1) * 8, c = c0 + (e & 1);
            float v = acc[e] + (bias ? __ldg(bias + c) : 0.0f);
            if (mode == 0) { float dv; v = act_fwd(act + 1, v, dv); }
            else v *= dact_from_output(act, gate[r * ldg + c]);
            out[r * ldo + c] = v;
        }
    }
    __syncthreads();        // the planes are rewritten by the next layer; out is complete
}

#define MMA_LAYER(As, lda, K, W, ldw, N, bias, mode, act, gate, ldg, out, ldo)                                        \
    do {                                                                                                               \
        if ((K) % 128 == 0) mma_layer_t<16>(As, lda, K, W, ldw, N, bias, mode, act, gate, ldg, out, ldo, S.ahi, S.alo); \
        else mma_layer_t<8>(As, lda, K, W, ldw, N, bias, mode, act, gate, ldg, out, ldo, S.ahi, S.alo);                \
    } while (0)

// out[16][n_out] = A[16][K] W[K][n_out] + bias for tiny n_out (<= 16; the heads Dense_4 / Dense_7): 8 lanes per output, each a
// strided eighth of the K products, then a shuffle reduction (a thread per output would be a chain of K dependent loads)
__device__ __noinline__ void head_layer(const float* As, int lda, int K, const float* __restrict__ W, int n_out, const float* __restrict__ bias,
                                           float* out) {
    const int sub = threadIdx.x & 7;
    for (int o0 = 0; o0 < CH * n_out; o0 += NTHR / 8) {
        const int o = o0 + (threadIdx.x >> 3);
        const bool live = o < CH * n_out;
        const int r = live ? o / n_out : 0, j = live ? o - r * n_out : 0;
        float s = 0.0f;
        for (int k = sub; k < K; k += 8) s += As[r * lda + k] * __ldg(W + (long long)k * n_out + j);
        s += __shfl_xor_sync(0xffffffffu, s, 4); s += __shfl_xor_sync(0xffffffffu, s, 2); s += __shfl_xor_sync(0xffffffffu, s, 1);
        if (live && sub == 0) out[r * DP + j] = s + (bias ? __ldg(bias + j) : 0.0f);
    }
}

// v = sgn * field(xi, tf) and negdiv = -sgn * div for the CTA's 16 chains.  xi [16][DP], tf [16] in shared memory; results to
// vout [16][DP] and S.negdiv.  Block-wide: every thread calls it.
// (one copy of this code: inlined at its eight call sites the kernel was 43 k instructions and starved on instruction fetch)
__device__ __noinline__ void field_tile(const Args& A, const Smem& S, const float* xi, float* vout, bool want_div) {
    const mfm_field_t& F = A.F;
    const int d = F.dim, H = F.hidden, Fd = F.fourier_dim, act = F.act;
    const float* P = F.params;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // Fourier features (exe_flow_matching.py:70-71)
    for (int o = threadIdx.x; o < CH * Fd; o += NTHR) {
        const int r = o / Fd, j = o - r * Fd;
        const float deg = __fmul_rn(__fmul_rn(6.28318530717958647692f, __ldg(F.omega + j)), S.tf[r]);
        float sv, cv; sincosf(deg, &sv, &cv);
        S.big[r * LDC + j] = cv; S.big[r * LDC + Fd + j] = sv;
    }
    // Dense_2 (K = d, tiny): plain FMAs
    for (int o = threadIdx.x; o < CH * H; o += NTHR) {
        const int r = o / H, c = o - r * H;
        float s = __ldg(P + F.b_off[2] + c);
        for (int j = 0; j < d; ++j) s += xi[r * DP + j] * __ldg(P + F.w_off[2] + (long long)j * H + c);
        float dv; S.h2[r * LDH + c] = act_fwd(act + 1, s, dv);
    }
    // untempered grad logprob (clipped) and the Hessian term: warp per chain, two chains per warp
    {
        const mfm_target_t& T1 = A.T;          // (the target functions return the UNtempered log-likelihood terms; beta is not read)
        float* sc = S.tscr + warp * 5 * DP;
        float* xs = sc; float* gs = sc + DP; float* zs = sc + 2 * DP; float* hv = sc + 3 * DP; float* hd = sc + 4 * DP;
        for (int q = 0; q < CH / NWARP; ++q) {
            const int r = warp * (CH / NWARP) + q;
            for (int i = lane; i < d; i += 32) { xs[i] = xi[r * DP + i]; zs[i] = A.hutch ? S.zs[r * DP + i] : 0.0f; }
            __syncwarp();
            small_target_loglik_grad(T1, xs, gs, lane);
            if (want_div) small_target_hess(T1, xs, zs, A.hutch ? hv : nullptr, A.hutch ? nullptr : hd, lane);
            __syncwarp();
            for (int i = lane; i < d; i += 32) {
                const float gg = gs[i], clip = F.grad_clip;
                const bool in = !(clip > 0.0f) || (gg > -clip && gg < clip);
                S.gc[r * DP + i] = clip > 0.0f ? fminf(fmaxf(gg, -clip), clip) : gg;
                if (want_div) S.hx[r * DP + i] = in ? (A.hutch ? hv[i] : hd[i]) : 0.0f;
            }
            __syncwarp();
        }
    }
    __syncthreads();
    MMA_LAYER(S.big, LDC, 2 * Fd, A.wt + F.w_off[0], 2 * Fd, H, P + F.b_off[0], 0, act, nullptr, 0, S.h0, LDH);          // Dense_0
    MMA_LAYER(S.h2, LDH, H, A.wt + F.w_off[3], H, H, P + F.b_off[3], 0, act, nullptr, 0, S.cat, LDC);                // Dense_3 -> s_x
    MMA_LAYER(S.h0, LDH, H, A.wt + F.w_off[1], H, H, P + F.b_off[1], 0, act, nullptr, 0, S.cat + H, LDC);            // Dense_1 -> s_t
    head_layer(S.cat + H, LDC, H, P + F.w_off[4], d, P + F.b_off[4], S.gt);                                       // Dense_4 -> nn_t
    MMA_LAYER(S.cat, LDC, 2 * H, A.wt + F.w_off[5], 2 * H, H, P + F.b_off[5], 0, act, nullptr, 0, S.h5, LDH);            // Dense_5
    MMA_LAYER(S.h5, LDH, H, A.wt + F.w_off[6], H, H, P + F.b_off[6], 0, act, nullptr, 0, S.h6, LDH);                 // Dense_6
    head_layer(S.h6, LDH, H, P + F.w_off[7], d, P + F.b_off[7], S.y7);                                            // Dense_7 -> nn_xt
    __syncthreads();
    for (int o = threadIdx.x; o < CH * d; o += NTHR) {
        const int r = o / d, j = o - r * d;
        vout[r * DP + j] = A.sgn * (S.y7[r * DP + j] + S.gt[r * DP + j] * S.gc[r * DP + j]);                      // (:86-90)
    }
    if (!want_div) { __syncthreads(); return; }
    // divergence: forward-mode tangents through Dense_2, 3, 5 (first H rows), 6, 7 - one probe (z.(J z), :211-214) or the d basis
    // vectors (trace(jacfwd), :216-217); ta | tb live where the Fourier features were
    float* ta = S.big; float* tb = S.big + CH * LDH;
    if (threadIdx.x < CH) S.negdiv[threadIdx.x] = 0.0f;
    const int n_tan = A.hutch ? 1 : d;
    for (int jt = 0; jt < n_tan; ++jt) {
        __syncthreads();
        for (int o = threadIdx.x; o < CH * H; o += NTHR) {
            const int r = o / H, c = o - r * H;
            const float tin = A.hutch ? S.zw2[r * LDH + c] : __ldg(P + F.w_off[2] + (long long)jt * H + c);     // z W2, or row jt of W2
            ta[r * LDH + c] = tin * dact_from_output(act, S.h2[r * LDH + c]);
        }
        __syncthreads();
        MMA_LAYER(ta, LDH, H, A.wt + F.w_off[3], H, H, nullptr, 1, act, S.cat, LDC, tb, LDH);
        MMA_LAYER(tb, LDH, H, A.wt + F.w_off[5], 2 * H, H, nullptr, 1, act, S.h5, LDH, ta, LDH);
        MMA_LAYER(ta, LDH, H, A.wt + F.w_off[6], H, H, nullptr, 1, act, S.h6, LDH, tb, LDH);
        head_layer(tb, LDH, H, P + F.w_off[7], d, nullptr, S.y7);
        __syncthreads();
        if (threadIdx.x < CH) {
            const int r = threadIdx.x;
            float s = 0.0f;
            if (A.hutch) for (int j = 0; j < d; ++j) s += S.zs[r * DP + j] * (S.y7[r * DP + j] + S.gt[r * DP + j] * S.hx[r * DP + j]);
            else s = S.y7[r * DP + jt] + S.gt[r * DP + jt] * S.hx[r * DP + jt];
            S.negdiv[r] += s;
        }
    }
    __syncthreads();
    if (threadIdx.x < CH) S.negdiv[threadIdx.x] *= -A.sgn;
    __syncthreads();
}

__global__ void __launch_bounds__(NTHR, 1) ode_small_kernel(const Args A) {
    extern __shared__ float sm_raw[];
    const Smem S = carve(sm_raw);
    const int d = A.F.dim, H = A.F.hidden;
    const int c0 = blockIdx.x * CH;
    const int tid = threadIdx.x;
    const float t_final = A.target[A.n_seg - 1];
    // ---- init (ode_init_kernel) ----
    for (int o = tid; o < CH * DP; o += NTHR) {
        const int r = o / DP, j = o - r * DP;
        const bool live = c0 + r < A.n && j < d;
        const float v = live ? A.y0[(long long)(c0 + r) * d + j] : 0.0f;
        S.yx[o] = v; S.outx[o] = v; S.xi[o] = v;
        S.zs[o] = (live && A.z) ? A.z[(long long)(c0 + r) * d + j] : 0.0f;
    }
    if (tid < CH) {
        const bool live = c0 + tid < A.n;
        S.yl[tid] = 0.0f; S.outl[tid] = 0.0f; S.tt[tid] = 0.0f; S.dt[tid] = 0.0f;
        S.seg[tid] = live ? 0 : A.n_seg; S.icount[tid] = 0; S.ntry[tid] = 0;
        S.tf[tid] = A.sgn > 0 ? 0.0f : 1.0f;
    }
    __syncthreads();
    if (A.hutch) {   // per-solve constant of the Hutchinson tangent: z W2
        for (int o = tid; o < CH * H; o += NTHR) {
            const int r = o / H, c = o - r * H;
            float s = 0.0f;
            for (int j = 0; j < d; ++j) s += S.zs[r * DP + j] * __ldg(A.F.params + A.F.w_off[2] + (long long)j * H + c);
            S.zw2[r * LDH + c] = s;
        }
        __syncthreads();
    }
    float* k0 = S.kx;                       // stage slopes k_j at S.kx + j * CH * DP
    // ---- initial_step_size (ode_h0_kernel / ode_h1_kernel) ----
    field_tile(A, S, S.xi, k0, true);
    if (tid < CH) S.kl[tid] = S.negdiv[tid];
    __syncthreads();
    if (tid < CH) {
        const int r = tid;
        float s0 = 0.0f, s1 = 0.0f;
        for (int i = 0; i < d; ++i) {
            const float y = S.yx[r * DP + i], f = k0[r * DP + i];
            const float sc = A.atol + fabsf(y) * A.rtol;
            const float a = y / sc, b = f / sc; s0 += a * a; s1 += b * b;
        }
        { const float sc = A.atol + fabsf(S.yl[r]) * A.rtol; const float a = S.yl[r] / sc, b = S.kl[r] / sc; s0 += a * a; s1 += b * b; }
        const float dd0 = sqrtf(s0), dd1 = sqrtf(s1);
        const float h0 = (dd0 < 1e-5f || dd1 < 1e-5f) ? 1e-6f : 0.01f * dd0 / dd1;
        for (int i = 0; i < d; ++i) S.xi[r * DP + i] = S.yx[r * DP + i] + h0 * k0[r * DP + i];
        S.dt[r] = h0; S.d1[r] = dd1;
        const float tt = S.tt[r] + h0;
        S.tf[r] = A.sgn > 0 ? tt : 1.0f - tt;
    }
    __syncthreads();
    field_tile(A, S, S.xi, S.kx + CH * DP, true);
    if (tid < CH) S.kl[CH + tid] = S.negdiv[tid];
    __syncthreads();
    if (tid < CH) {
        const int r = tid;
        const float* f0 = k0; const float* f1 = S.kx + CH * DP;
        float s2 = 0.0f;
        for (int i = 0; i < d; ++i) {
            const float sc = A.atol + fabsf(S.yx[r * DP + i]) * A.rtol;
            const float a = (f1[r * DP + i] - f0[r * DP + i]) / sc; s2 += a * a;
        }
        { const float sc = A.atol + fabsf(S.yl[r]) * A.rtol; const float a = (S.kl[CH + r] - S.kl[r]) / sc; s2 += a * a; }
        const float h0 = S.dt[r], dd1 = S.d1[r];
        const float dd2 = sqrtf(s2) / h0;
        float h1;
        if (dd1 <= 1e-15f && dd2 <= 1e-15f) h1 = fmaxf(1e-6f, h0 * 1e-3f);
        else { const float m = (isnan(dd1) || isnan(dd2)) ? NAN : fmaxf(dd1, dd2); h1 = powf(0.01f / m, 0.2f); }
        float dt = isnan(h1) ? NAN : fminf(100.0f * h0, h1);
        if (dt < 0.0f) dt = 0.0f;
        S.dt[r] = dt;
    }
    __syncthreads();
    // ---- adaptive loop: every chain carries its own (t, dt, segment); finished chains are masked ----
    const long long max_iter = (long long)A.n_seg * (long long)A.mxstep + 2;
    int n_acc = 0, n_try = 0;              // this thread's chain (tid < CH)
    for (long long it = 0; it < max_iter; ++it) {
        const int active = (tid < CH && S.seg[tid] < A.n_seg) ? 1 : 0;
        if (!__syncthreads_or(active)) break;
#pragma unroll 1
        for (int sg = 1; sg <= 6; ++sg) {
            // stage input xi = y + dt * sum_j beta[sg-1][j] k_j ; field time t + alpha dt   (ode_stage_kernel)
            for (int o = tid; o < CH * d; o += NTHR) {
                const int r = o / d, j = o - r * d;
                if (S.seg[r] < A.n_seg) {
                    float acc = 0.0f;
#pragma unroll
                    for (int q = 0; q < 6; ++q) if (q < sg) acc += c_beta[sg - 1][q] * S.kx[q * CH * DP + r * DP + j];
                    S.xi[r * DP + j] = S.yx[r * DP + j] + S.dt[r] * acc;
                }
            }
            if (tid < CH && S.seg[tid] < A.n_seg) {
                const float ti = S.tt[tid] + S.dt[tid] * c_alpha[sg - 1];
                S.tf[tid] = A.sgn > 0 ? ti : 1.0f - ti;
            }
            __syncthreads();
            field_tile(A, S, S.xi, S.kx + sg * CH * DP, true);
            if (tid < CH) S.kl[sg * CH + tid] = S.negdiv[tid];
            __syncthreads();
        }
        // error ratio, accept / reject, controller, FSAL, dense output at the final time  (ode_finish_kernel)
        if (tid < CH && S.seg[tid] < A.n_seg) {
            const int r = tid;
            int seg = S.seg[r];
            const float tt = S.tt[r], h = S.dt[r];
            float sum = 0.0f;
            for (int i = 0; i < d; ++i) {
                float ss = 0.0f, se = 0.0f;
#pragma unroll
                for (int j = 0; j < 7; ++j) { const float k = S.kx[j * CH * DP + r * DP + i]; ss += c_sol[j] * k; se += c_err[j] * k; }
                const float y = S.yx[r * DP + i];
                const float y1 = h * ss + y;
                const float rr = (h * se) / (A.atol + A.rtol * fmaxf(fabsf(y), fabsf(y1)));
                sum += rr * rr;
            }
            float ssl = 0.0f, sel = 0.0f;
#pragma unroll
            for (int j = 0; j < 7; ++j) { const float k = S.kl[j * CH + r]; ssl += c_sol[j] * k; sel += c_err[j] * k; }
            const float yl = S.yl[r];
            const float yl1 = h * ssl + yl;
            { const float rr = (h * sel) / (A.atol + A.rtol * fmaxf(fabsf(yl), fabsf(yl1))); sum += rr * rr; }
            const float ratio = sqrtf(sum / (float)(d + 1));
            const bool accept = ratio <= 1.0f;
            float new_dt;
            if (isnan(ratio)) new_dt = NAN;
            else if (ratio == 0.0f) new_dt = h * 10.0f;
            else {
                const float dfac = ratio < 1.0f ? 1.0f : 0.2f;
                new_dt = h * fminf(10.0f, fmaxf(powf(ratio, -0.2f) * 0.9f, dfac));
            }
            if (new_dt < 0.0f) new_dt = 0.0f;
            float t_new = tt;
            if (accept) {
                t_new = tt + h;
                const float rel = (t_final - tt) / (t_new - tt);
                for (int i = 0; i < d; ++i) {
                    float ss = 0.0f, smid = 0.0f, kk0 = 0.f, kk6 = 0.f;
#pragma unroll
                    for (int j = 0; j < 7; ++j) {
                        const float k = S.kx[j * CH * DP + r * DP + i]; ss += c_sol[j] * k; smid += c_mid[j] * k;
                        if (j == 0) kk0 = k; if (j == 6) kk6 = k;
                    }
                    const float y = S.yx[r * DP + i];
                    const float y1 = h * ss + y, ymid = y + h * smid;
                    S.outx[r * DP + i] = fit_eval(y, y1, ymid, kk0, kk6, h, rel);
                    S.yx[r * DP + i] = y1;
                    S.kx[r * DP + i] = kk6;                          // FSAL
                }
                float smid = 0.0f;
#pragma unroll
                for (int j = 0; j < 7; ++j) smid += c_mid[j] * S.kl[j * CH + r];
                S.outl[r] = fit_eval(yl, yl1, yl + h * smid, S.kl[r], S.kl[6 * CH + r], h, rel);
                S.yl[r] = yl1; S.kl[r] = S.kl[6 * CH + r]; S.tt[r] = t_new;
                ++n_acc;
            }
            int ic = S.icount[r] + 1;
            ++n_try;
            S.ntry[r] = n_try; S.dt[r] = new_dt;
            while (seg < A.n_seg && !(t_new < A.target[seg] && ic < A.mxstep && new_dt > 0.0f)) { ++seg; ic = 0; }
            S.seg[r] = seg; S.icount[r] = ic;
        }
        __syncthreads();
    }
    // ---- results and statistics ----
    for (int o = tid; o < CH * d; o += NTHR) {
        const int r = o / d, j = o - r * d;
        if (c0 + r < A.n) A.y1[(long long)(c0 + r) * d + j] = S.outx[r * DP + j];
    }
    if (tid < CH && c0 + tid < A.n) {
        if (A.ldj) A.ldj[c0 + tid] = S.outl[tid];
        atomicAdd(&A.counters[1], n_acc);
        atomicAdd(&A.counters[2], n_try);
        atomicMax(&A.counters[3], n_try);
        atomicAdd(reinterpret_cast<unsigned long long*>(A.counters + 10), (unsigned long long)(2 + 6 * n_try));
    }
}

inline bool eligible(const mfm_field_t& F, const mfm_target_t& T, int n) {
    const bool target_ok = T.kind == MFM_TARGET_GMM || T.kind == MFM_TARGET_PHI4 || T.kind == MFM_TARGET_GAUSS;
    const bool act_ok = F.act == MFM_ACT_RELU || F.act == MFM_ACT_TANH || F.act == MFM_ACT_ELU;
    // (one width for every layer: networks with unequal branch widths take the graph-driven loop of ode_solve)
    return target_ok && act_ok && field_widths(F).equal && n > 0 && F.dim <= DP && (F.hidden == 64 || F.hidden == 128) && (F.fourier_dim == 32 || F.fourier_dim == 64 || F.fourier_dim == 128) && !(T.kind == MFM_TARGET_GMM && F.dim != 2);
}

}  // namespace small
}  // namespace mfm
