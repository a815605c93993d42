// CNF push/pull with adaptive Dormand-Prince 5(4) and the flow-MH transition.
//
// Replaces, for a whole batch of chains at once:
//   VectorFieldNet.__call__                      exe_flow_matching.py:56-90
//   divergence by jvp (Hutchinson) / trace(jacfwd)  :211-217, :231-237
//   transform_and_logdet / inverse_and_logdet    :206-242
//   jax.experimental.ode.odeint (jax 0.4.26)     :345-349   [restated in oracle/ode.py]
//   random_walk / indep metropolis_hastings      :246-278
//
// Layout: every per-chain quantity is SoA [n, d] / [n]; the augmented ODE state ravel((x, ldj)) is
// kept as x[n,d] + ldj[n].  All chains advance in lock-step *iterations*; each chain carries its
// own (t, dt, segment, step count) and is masked once finished — exactly the semantics of the
// batched while_loop that jax.vmap produces.  Dense layers run on tensor cores (3xTF32).
#include "internal.h"
#include <limits.h>
#include <string.h>
#include <stdlib.h>
#include "gemm_tf32x3.cuh"
#include "ref_dist.cuh"

namespace mfm {

// ---------------------------------------------------------------------------------------------
// Dormand-Prince coefficients (float32 roundings of the float64 literals, as jnp.array(..., f32))
// ---------------------------------------------------------------------------------------------
__constant__ float c_alpha[6] = {(float)(1.0 / 5), (float)(3.0 / 10), (float)(4.0 / 5), (float)(8.0 / 9), 1.0f, 1.0f};
__constant__ float c_beta[6][6] = {
    {(float)(1.0 / 5), 0, 0, 0, 0, 0},
    {(float)(3.0 / 40), (float)(9.0 / 40), 0, 0, 0, 0},
    {(float)(44.0 / 45), (float)(-56.0 / 15), (float)(32.0 / 9), 0, 0, 0},
    {(float)(19372.0 / 6561), (float)(-25360.0 / 2187), (float)(64448.0 / 6561), (float)(-212.0 / 729), 0, 0},
    {(float)(9017.0 / 3168), (float)(-355.0 / 33), (float)(46732.0 / 5247), (float)(49.0 / 176), (float)(-5103.0 / 18656), 0},
    {(float)(35.0 / 384), 0, (float)(500.0 / 1113), (float)(125.0 / 192), (float)(-2187.0 / 6784), (float)(11.0 / 84)}};
__constant__ float c_sol[7] = {(float)(35.0 / 384), 0, (float)(500.0 / 1113), (float)(125.0 / 192),
                               (float)(-2187.0 / 6784), (float)(11.0 / 84), 0};
__constant__ float c_err[7] = {(float)(35.0 / 384 - 1951.0 / 21600), 0, (float)(500.0 / 1113 - 22642.0 / 50085),
                               (float)(125.0 / 192 - 451.0 / 720), (float)(-2187.0 / 6784 - -12231.0 / 42400),
                               (float)(11.0 / 84 - 649.0 / 6300), (float)(-1.0 / 60.0)};
__constant__ float c_mid[7] = {(float)(6025192743.0 / 30085553152.0 / 2), 0, (float)(51252292925.0 / 65400821598.0 / 2),
                               (float)(-2691868925.0 / 45128329728.0 / 2), (float)(187940372067.0 / 1594534317056.0 / 2),
                               (float)(-1776094331.0 / 19743644256.0 / 2), (float)(11237099.0 / 235043384.0 / 2)};

// ---------------------------------------------------------------------------------------------
// GEMM epilogues specific to the field
// ---------------------------------------------------------------------------------------------
// v = sgn * (acc + bias + gt * gc)          (exe_flow_matching.py:86-90)
struct EpiFieldV {
    static constexpr bool kRowSum = false;
    float* V; long long ldv; const float* bias; const float* gt; const float* gc; long long ld; float sgn;
    const int* row_map;      // optional: compact row -> chain index of the output
    float* amax_out = nullptr; mutable float vmax = 0.0f;      // optional: max |v| (the FM pass bounds its loss gradient with it)
    struct Aux { float bias, gt, gc; int orow; };
    __device__ __forceinline__ Aux load(int row, int col) const {
        const long long o = (long long)row * ld + col;
        Aux a; a.bias = __ldg(bias + col); a.gt = __ldg(gt + o); a.gc = __ldg(gc + o);
        a.orow = row_map ? __ldg(row_map + row) : row;
        return a;
    }
    __device__ __forceinline__ float apply(int, int col, float acc, const Aux& a) const {
        const float v = sgn * (acc + a.bias + a.gt * a.gc);
        V[(long long)a.orow * ldv + col] = v; vmax = fmaxf(vmax, fabsf(v));
        return 0.0f;
    }
    __device__ __forceinline__ float operator()(int row, int col, float acc) const { return apply(row, col, acc, load(row, col)); }
    __device__ __forceinline__ void row_partial(int, int, float) const {}
    __device__ __forceinline__ void at_z(int) {}
    struct Col4 { float4 bias; };
    struct Row4 { float4 gt, gc; int orow; };
    bool vec_ok() const { return aligned16(V) && ldv % 4 == 0 && aligned16(bias) && aligned16(gt) && aligned16(gc) && ld % 4 == 0; }
    __device__ __forceinline__ Col4 load_col4(int col) const { Col4 c; c.bias = ldg4(bias + col); return c; }
    __device__ __forceinline__ Row4 load_row4(int row, int col) const {
        const long long o = (long long)row * ld + col;
        Row4 r; r.gt = ldg4(gt + o); r.gc = ldg4(gc + o); r.orow = row_map ? __ldg(row_map + row) : row;
        return r;
    }
    __device__ __forceinline__ float apply4(int, int col, const float4& acc, const Col4& c, const Row4& r) const {
        float4 v;
        v.x = sgn * (acc.x + c.bias.x + r.gt.x * r.gc.x); v.y = sgn * (acc.y + c.bias.y + r.gt.y * r.gc.y);
        v.z = sgn * (acc.z + c.bias.z + r.gt.z * r.gc.z); v.w = sgn * (acc.w + c.bias.w + r.gt.w * r.gc.w);
        st4(V + (long long)r.orow * ldv + col, v);
        vmax = amax4(vmax, v);
        return 0.0f;
    }
};
// Hutchinson: sum_col z * (acc + gt * hvc)    (:212-214)
struct EpiFieldDiv {
    static constexpr bool kRowSum = true;
    const float* z; const float* gt; const float* hvc; long long ld; float* partial; int n_tiles;
    struct Aux { float z, gt, hvc; };
    __device__ __forceinline__ Aux load(int row, int col) const {
        const long long o = (long long)row * ld + col;
        Aux a; a.z = __ldg(z + o); a.gt = __ldg(gt + o); a.hvc = __ldg(hvc + o);
        return a;
    }
    __device__ __forceinline__ float apply(int, int, float acc, const Aux& a) const { return a.z * (acc + a.gt * a.hvc); }
    __device__ __forceinline__ float operator()(int row, int col, float acc) const { return apply(row, col, acc, load(row, col)); }
    struct Col4 {};
    struct Row4 { float4 z, gt, hvc; };
    bool vec_ok() const { return aligned16(z) && aligned16(gt) && aligned16(hvc) && ld % 4 == 0; }
    __device__ __forceinline__ Col4 load_col4(int) const { return Col4{}; }
    __device__ __forceinline__ Row4 load_row4(int row, int col) const {
        const long long o = (long long)row * ld + col;
        Row4 r; r.z = ldg4(z + o); r.gt = ldg4(gt + o); r.hvc = ldg4(hvc + o);
        return r;
    }
    __device__ __forceinline__ float apply4(int, int, const float4& acc, const Col4&, const Row4& r) const {
        return ((r.z.x * (acc.x + r.gt.x * r.hvc.x) + r.z.y * (acc.y + r.gt.y * r.hvc.y)) +
                (r.z.z * (acc.z + r.gt.z * r.hvc.z) + r.z.w * (acc.w + r.gt.w * r.hvc.w)));
    }
    __device__ __forceinline__ void row_partial(int row, int tile, float s) const { partial[(long long)row * n_tiles + tile] = s; }
    __device__ __forceinline__ void at_z(int) {}
};

int dense(int n, int in, int out, const float* A, long long lda, const float* WT, long long ldwt, const float* bias, int relu,
                 float* C, long long ldc, const float* mask, long long ldm, int mask_div, cudaStream_t st,
                 const int* n_rows_dev, DenseAmax am) {
    GemmShape p{n, out, in, A, lda, WT, ldwt, n_rows_dev};
    p.a_amax = am.a; p.a_amax2 = am.a2; p.a_bound = am.a_bound; p.a_split = am.a_split; p.a_scale_src = am.a_scale_src;
    const bool general = relu > ACT_RELU || am.dact != nullptr || am.mask_mul != 0;     // activations other than relu: the ACT = true functors
    if (am.out_split && am.w_norm && (am.a || am.a_bound > 0.0f)) {
        // C also leaves pre-split for the layer that consumes it (EpiStdS)
        auto run = [&](auto e) -> cudaError_t {
            e.alt_amax = am.alt_amax; e.alt_w_norm = am.alt_w_norm; e.alt_bias = am.alt_bias;
            e.amax_out = am.out; e.dact = am.dact; e.lddact = am.lddact; e.mask_mul = am.mask_mul;
            return launch_gemm<true, false>(p, e, st);
        };
        if (general) MFM_CUDA_CHECK(run(EpiStdSA{C, ldc, bias, mask, ldm, nullptr, 0, relu, mask_div, am.out_split, am.a, am.a2, am.a_bound, am.w_norm, am.bias_amax, am.add_bound, am.out_bound}));
        else MFM_CUDA_CHECK(run(EpiStdS{C, ldc, bias, mask, ldm, nullptr, 0, relu, mask_div, am.out_split, am.a, am.a2, am.a_bound, am.w_norm, am.bias_amax, am.add_bound, am.out_bound}));
        return MFM_OK;
    }
    auto run = [&](auto e) -> cudaError_t {
        e.amax_out = am.out; e.dact = am.dact; e.lddact = am.lddact; e.mask_mul = am.mask_mul;
        return launch_gemm<true, false>(p, e, st);
    };
    if (general) MFM_CUDA_CHECK(run(EpiStdA{C, ldc, bias, mask, ldm, nullptr, 0, 1.0f, relu, mask_div}));
    else MFM_CUDA_CHECK(run(EpiStd{C, ldc, bias, mask, ldm, nullptr, 0, 1.0f, relu, mask_div}));
    return MFM_OK;
}

// out[c*rows + r] = in[r*cols + c]   (32x32 tiles through shared memory)
__global__ void transpose_kernel(int rows, int cols, const float* __restrict__ in, float* __restrict__ out) {
    __shared__ float tile[32][33];
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int r = r0 + j, c = c0 + threadIdx.x;
        tile[j][threadIdx.x] = (r < rows && c < cols) ? in[(long long)r * cols + c] : 0.0f;
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j, r = r0 + threadIdx.x;
        if (r < rows && c < cols) out[(long long)c * rows + r] = tile[threadIdx.x][j];
    }
}

// the same for all eight dense kernels in ONE launch (they are transposed once per ABI call; eight launches of a few
// microseconds each were a fixed cost that weighed 2 % of an FM update at 8 192 chains and 10 % at the small reference shapes)
struct TransposeAll { int in[8], out[8], tile0[9], tx[8]; long long w_off[8]; };
__global__ void transpose_all_kernel(TransposeAll D, const float* __restrict__ params, float* __restrict__ wt) {
    __shared__ float tile[32][33];
    int l = 0;
#pragma unroll
    for (int i = 1; i < 8; ++i) if ((int)blockIdx.x >= D.tile0[i]) l = i;
    const int tidx = blockIdx.x - D.tile0[l];
    const int rows = D.in[l], cols = D.out[l];
    const int c0 = (tidx % D.tx[l]) * 32, r0 = (tidx / D.tx[l]) * 32;
    const float* in = params + D.w_off[l]; float* out = wt + D.w_off[l];
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int r = r0 + j, c = c0 + threadIdx.x;
        tile[j][threadIdx.x] = (r < rows && c < cols) ? in[(long long)r * cols + c] : 0.0f;
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j, r = r0 + threadIdx.x;
        if (r < rows && c < cols) out[(long long)c * rows + r] = tile[threadIdx.x][j];
    }
}

// operator norms of the dense kernels for the output bounds of the split-writing epilogue (EpiStdS): per layer the largest
// absolute column sum (forward product x W), the largest absolute row sum (backward-data product d W^T) and max |bias|.
// One warp per matrix row, coalesced: row sums of W [in][out] give the row norm, row sums of its transpose (wt, [out][in],
// already built for the GEMMs) the column norm.  grid (8 layers, 2 kinds, WN_SLICES); slots zeroed by the caller.
constexpr int WN_SLICES = 32;
struct WeightDims { int in[8], out[8]; long long w_off[8], b_off[8]; };
__global__ void __launch_bounds__(256) weight_norms_kernel(const float* __restrict__ params, const float* __restrict__ wt, WeightDims D,
                                                           float* __restrict__ pool) {
    const int layer = blockIdx.x, kind = blockIdx.y, slice = blockIdx.z;
    const int rows = kind == 0 ? D.out[layer] : D.in[layer], cols = kind == 0 ? D.in[layer] : D.out[layer];
    const float* W = (kind == 0 ? wt : params) + D.w_off[layer];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float m = 0.0f;
    for (int r = slice * 8 + warp; r < rows; r += WN_SLICES * 8) {
        float sum = 0.0f;
        for (int c = lane; c < cols; c += 32) sum += fabsf(W[(long long)r * cols + c]);
        m = fmaxf(m, warp_sum(sum));
    }
    amax_publish_warp(pool + (kind == 0 ? AM_WNORM_COL : AM_WNORM_ROW) + layer, m);
    if (kind == 0 && slice == 0) {
        float b = 0.0f;
        for (int o = threadIdx.x; o < D.out[layer]; o += blockDim.x) b = fmaxf(b, fabsf(params[D.b_off[layer] + o]));
        amax_publish_warp(pool + AM_BIAS + layer, b);
    }
}

static void layer_dims(const mfm_field_t& F, int i, int& in, int& out) {
    const int d = F.dim, H = F.hidden, Fd = F.fourier_dim;
    const int ins[8] = {2 * Fd, H, d, H, H, 2 * H, H, H}, outs[8] = {H, H, H, H, d, H, H, d};
    in = ins[i]; out = outs[i];
}

// 8 consecutive floats -> 16 bf16 in the same 32 bytes: [bf16(b0..b7) | bf16(rest0..rest7)], rest = b - trunc_tf32(b)
// (what the tensor core drops from the raw fp32 tile): the B operand's cross tile of the persistent GEMM, ready for TMA
__global__ void presplit_kernel(const float4* __restrict__ src, uint4* __restrict__ dst, long long n8) {
    const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (g >= n8) return;
    const float4 a = __ldg(src + 2 * g), c = __ldg(src + 2 * g + 1);
    auto rest = [](float x) { return x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); };
    auto pack = [](float lo16, float hi16) { uint32_t r; asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi16), "f"(lo16)); return r; };
    dst[2 * g] = make_uint4(pack(a.x, a.y), pack(a.z, a.w), pack(c.x, c.y), pack(c.z, c.w));
    dst[2 * g + 1] = make_uint4(pack(rest(a.x), rest(a.y)), pack(rest(a.z), rest(a.w)), pack(rest(c.x), rest(c.y)), pack(rest(c.z), rest(c.w)));
}
// split16 layout of the scaled-fp16 kernel (gemm_tcgen05_h16.cuh): 16 consecutive floats -> 16 hi | 16 lo fp16 parts of the
// values scaled by h16_scale(*amax) (the kernel derives the same power of two from the same slot)
__global__ void presplit_h16_kernel(const float4* __restrict__ src, uint4* __restrict__ dst, long long n16, const float* __restrict__ amax) {
    const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (g >= n16) return;
    const float sc = tc2h::h16_scale(*amax);
    float4 v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = __ldg(src + 4 * g + j);
    uint32_t hp[8], lp[8];
    tc2h::split16(v, sc, hp, lp);
    dst[4 * g] = make_uint4(hp[0], hp[1], hp[2], hp[3]); dst[4 * g + 1] = make_uint4(hp[4], hp[5], hp[6], hp[7]);
    dst[4 * g + 2] = make_uint4(lp[0], lp[1], lp[2], lp[3]); dst[4 * g + 3] = make_uint4(lp[4], lp[5], lp[6], lp[7]);
}
// both weight mirrors (W^T and W) in one launch: blockIdx.y picks the pair
__global__ void presplit_h16_pair_kernel(const float4* __restrict__ src0, uint4* __restrict__ dst0, const float4* __restrict__ src1, uint4* __restrict__ dst1,
                                         long long n16, const float* __restrict__ amax) {
    const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (g >= n16) return;
    const float4* src = blockIdx.y ? src1 : src0; uint4* dst = blockIdx.y ? dst1 : dst0;
    const float sc = tc2h::h16_scale(*amax);
    float4 v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = __ldg(src + 4 * g + j);
    uint32_t hp[8], lp[8];
    tc2h::split16(v, sc, hp, lp);
    dst[4 * g] = make_uint4(hp[0], hp[1], hp[2], hp[3]); dst[4 * g + 1] = make_uint4(hp[4], hp[5], hp[6], hp[7]);
    dst[4 * g + 2] = make_uint4(lp[0], lp[1], lp[2], lp[3]); dst[4 * g + 3] = make_uint4(lp[4], lp[5], lp[6], lp[7]);
}
int presplit_weights(const float* src, float* dst, long long n_floats, const float* amax, cudaStream_t st) {
    if (tc2h::gemm_h16() && amax != nullptr && n_floats % 16 == 0) {
        presplit_h16_kernel<<<ceil_div(n_floats / 16, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(src), reinterpret_cast<uint4*>(dst), n_floats / 16, amax);
        MFM_LAUNCH_CHECK();
        return MFM_OK;
    }
    const long long n8 = n_floats / 8;
    presplit_kernel<<<ceil_div(n8, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(src), reinterpret_cast<uint4*>(dst), n8);
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}

// Mirrors of the dense kernels: the range [w_off[0], end of Dense_7) of the flat buffer (biases in between are converted too,
// harmlessly).  h16 mirrors need 16-float groups and 64-byte aligned tiles, bf16-cross mirrors 8-float groups.
static bool mirror_range(const mfm_field_t& F, const FieldBufs& B, bool& h16, long long& lo, long long& hi) {
    if (B.wx == nullptr || B.wxo == nullptr) return false;
    h16 = tc2h::gemm_h16() != 0 && B.amax != nullptr;
    const int g = h16 ? 16 : 8;
    if (((reinterpret_cast<uintptr_t>(F.params) | reinterpret_cast<uintptr_t>(B.wt)) & (h16 ? 63 : 31)) != 0) return false;
    for (int i = 0; i < 8; ++i) { int in, out; layer_dims(F, i, in, out); if (in % g || out % g || F.w_off[i] % g) return false; }
    int in7, out7; layer_dims(F, 7, in7, out7);
    lo = F.w_off[0]; hi = (long long)F.w_off[7] + (long long)in7 * out7;
    return true;
}

int field_prepare_weights(const mfm_field_t& F, FieldBufs& B, cudaStream_t st) {
    tc2p::clear_cross(); tc2h::clear_mirrors_h16();
    {
        TransposeAll D; D.tile0[0] = 0;
        for (int i = 0; i < 8; ++i) {
            layer_dims(F, i, D.in[i], D.out[i]); D.w_off[i] = F.w_off[i];
            D.tx[i] = ceil_div(D.out[i], 32);
            D.tile0[i + 1] = D.tile0[i] + D.tx[i] * ceil_div(D.in[i], 32);
        }
        transpose_all_kernel<<<D.tile0[8], dim3(32, 8), 0, st>>>(D, F.params, B.wt);
        MFM_LAUNCH_CHECK();
    }
    if (B.amax) {
        // max |parameter|: the scale of both weight mirrors, and the bound of the exact path's basis tangents (entries of W2)
        MFM_CUDA_CHECK(tc2h::launch_absmax(F.params, F.n_params, 1, (int)(F.n_params & ~3ll), nullptr, B.amax + AM_W, st));
        MFM_CUDA_CHECK(cudaMemsetAsync(B.amax + AM_WNORM_COL, 0, 24 * sizeof(float), st));
        WeightDims D;
        for (int i = 0; i < 8; ++i) { layer_dims(F, i, D.in[i], D.out[i]); D.w_off[i] = F.w_off[i]; D.b_off[i] = F.b_off[i]; }
        weight_norms_kernel<<<dim3(8, 2, WN_SLICES), 256, 0, st>>>(F.params, B.wt, D, B.amax);
        MFM_LAUNCH_CHECK();
    }
    bool h16 = false; long long lo = 0, hi = 0;
    if (mirror_range(F, B, h16, lo, hi)) {
        int rc;
        if (h16 && (hi - lo) % 16 == 0) {
            presplit_h16_pair_kernel<<<dim3(ceil_div((hi - lo) / 16, 256), 2), 256, 0, st>>>(reinterpret_cast<const float4*>(B.wt + lo), reinterpret_cast<uint4*>(B.wx + lo),
                                                                                              reinterpret_cast<const float4*>(F.params + lo), reinterpret_cast<uint4*>(B.wxo + lo),
                                                                                              (hi - lo) / 16, B.amax + AM_W);
            MFM_LAUNCH_CHECK();
        } else {
            if ((rc = presplit_weights(B.wt + lo, B.wx + lo, hi - lo, h16 ? B.amax + AM_W : nullptr, st))) return rc;
            if ((rc = presplit_weights(F.params + lo, B.wxo + lo, hi - lo, h16 ? B.amax + AM_W : nullptr, st))) return rc;
        }
        field_register_mirrors(F, B);
    }
    return MFM_OK;
}

// (re-)announce the mirrors field_prepare_weights built in this workspace (a later ABI call on the same workspace: FM part 2)
void field_register_mirrors(const mfm_field_t& F, const FieldBufs& B) {
    tc2p::clear_cross(); tc2h::clear_mirrors_h16();
    bool h16 = false; long long lo = 0, hi = 0;
    if (!mirror_range(F, B, h16, lo, hi)) return;
    if (h16) {
        tc2h::register_mirror_h16(B.wt + lo, (size_t)(hi - lo), B.wx + lo, B.amax + AM_W);
        tc2h::register_mirror_h16(F.params + lo, (size_t)(hi - lo), B.wxo + lo, B.amax + AM_W);
    } else {
        tc2p::register_cross(B.wt + lo, (size_t)(hi - lo), B.wx + lo);
        tc2p::register_cross(F.params + lo, (size_t)(hi - lo), B.wxo + lo);
    }
}

// ---------------------------------------------------------------------------------------------
// elementwise helpers
// ---------------------------------------------------------------------------------------------
__global__ void fourier_kernel(int n, int F, const float* __restrict__ omega, const float* __restrict__ t,
                               float* __restrict__ ff, const int* __restrict__ n_rows_dev, float* __restrict__ ff_s, float* __restrict__ ff_bound) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i == 0 && ff_bound) *ff_bound = 1.0f;          // the slot the copy's scale derives from (consumer's a_scale_src)
    if (n_rows_dev) n = min(n, *n_rows_dev);
    if (i >= (long long)n * F) return;
    const int c = (int)(i / F), j = (int)(i % F);
    // degt = 2*pi*fourier_random*t  (left to right, :70)
    const float deg = __fmul_rn(__fmul_rn(6.28318530717958647692f, omega[j]), t[c]);
    float sv, cv; sincosf(deg, &sv, &cv);
    ff[(long long)c * 2 * F + j] = cv;
    ff[(long long)c * 2 * F + F + j] = sv;
    if (ff_s) {
        // pre-split copy for Dense_0 (split16 layout, scale 2^14 = h16_scale(1): |cos|, |sin| <= 1)
        const float sc = 16384.0f;
        __half* row = reinterpret_cast<__half*>(ff_s + (long long)c * 2 * F);
        const float xc = cv * sc, xs = sv * sc;
        const __half hc = __float2half_rn(xc), hs = __float2half_rn(xs);
        const int jc = j, js = F + j;
        row[2 * (jc & ~15) + (jc & 15)] = hc; row[2 * (jc & ~15) + 16 + (jc & 15)] = __float2half_rn(xc - __half2float(hc));
        row[2 * (js & ~15) + (js & 15)] = hs; row[2 * (js & ~15) + 16 + (js & 15)] = __float2half_rn(xs - __half2float(hs));
    }
}

// out[i,:] = a[i,:] * (gate[i,:] > 0);  amax (optional): max |out| is folded into the slot (out feeds a scaled-fp16 GEMM)
__global__ void gate_kernel(long long total, int H, const float* __restrict__ a, const float* __restrict__ gate,
                            long long ldg, float* __restrict__ out, const int* __restrict__ n_rows_dev, float* __restrict__ amax, int mul) {
    __shared__ float red[32];
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n_rows_dev) total = min(total, (long long)(*n_rows_dev) * H);
    float m = 0.0f;
    if (i < total) {
        const long long r = i / H; const int c = (int)(i % H);
        const float gv = gate[r * ldg + c];
        const float v = mul ? a[i] * gv : (gv > 0.0f ? a[i] : 0.0f);      // mul: `gate` holds activation derivatives
        out[i] = v; m = fabsf(v);
    }
    if (amax) amax_publish_block(amax, m, red);
}

// same, four columns per thread (H % 4 == 0, 16-byte aligned rows): HBM-bound, 12 B moved per element.
// out_s (optional): pre-split copy of `out` scaled by h16_scale(*scale_src) - gating only zeroes entries, so the exact maximum
// of `a` bounds the result.
__global__ void gate4_kernel(long long total4, int H4, const float4* __restrict__ a, const float4* __restrict__ gate,
                             long long ldg4, float4* __restrict__ out, const int* __restrict__ n_rows_dev, float* __restrict__ amax,
                             float* __restrict__ out_s, const float* __restrict__ scale_src, int mul) {
    __shared__ float red[32];
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n_rows_dev) total4 = min(total4, (long long)(*n_rows_dev) * H4);
    float m = 0.0f;
    if (i < total4) {
        const float4 g = ldg4 == H4 ? __ldg(gate + i) : __ldg(gate + (i / H4) * ldg4 + (i % H4));
        const float4 v = __ldg(a + i);
        const float4 o = mul ? make_float4(v.x * g.x, v.y * g.y, v.z * g.z, v.w * g.w)
                             : make_float4(g.x > 0.0f ? v.x : 0.0f, g.y > 0.0f ? v.y : 0.0f, g.z > 0.0f ? v.z : 0.0f, g.w > 0.0f ? v.w : 0.0f);
        out[i] = o; m = amax4(0.0f, o);
        if (out_s) {
            const float sc = tc2h::h16_scale(*scale_src);
            const long long e = 4 * i;                                  // flat element index (rows are H4 * 4 wide, H % 16 == 0)
            uint2 hp, lp;
            split_pair(o.x * sc, o.y * sc, hp.x, lp.x);
            split_pair(o.z * sc, o.w * sc, hp.y, lp.y);
            char* gp = reinterpret_cast<char*>(out_s + (e & ~15ll)) + 2 * (int)(e & 15);
            *reinterpret_cast<uint2*>(gp) = hp;
            *reinterpret_cast<uint2*>(gp + 32) = lp;
        }
    }
    if (amax) amax_publish_block(amax, m, red);
}

// exact path: tan[(i,j),:] = W2[j,:] * (h2[i,:] > 0)
__global__ void basis_tangent_kernel(int n, int d, int H, const float* __restrict__ W2, const float* __restrict__ h2,
                                     float* __restrict__ tan, const int* __restrict__ n_rows_dev, int mul) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (n_rows_dev) n = min(n, *n_rows_dev);
    if (i >= (long long)n * d * H) return;
    const int k = (int)(i % H); const long long r = i / H; const int j = (int)(r % d); const long long c = r / d;
    const float gv = h2[c * H + k];                                   // the activation (relu) or its derivative (mul)
    tan[i] = mul ? W2[(long long)j * H + k] * gv : (gv > 0.0f ? W2[(long long)j * H + k] : 0.0f);
}

// exact path: div_i = sum_j tan6[(i,j),:].W7[:,j] + sum_j gt[i,j]*hdc[i,j];  out = coef * div
__global__ void exact_trace_kernel(int n, int d, int H, const float* __restrict__ tan6, const float* __restrict__ W7,
                                   const float* __restrict__ gt, const float* __restrict__ hdc, float coef,
                                   float* __restrict__ out, const int* __restrict__ n_rows_dev,
                                   const int* __restrict__ row_map) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (n_rows_dev) n = min(n, *n_rows_dev);
    if (c >= n) return;
    float s = 0.0f;
    for (int j = 0; j < d; ++j) {
        const float* row = tan6 + ((long long)c * d + j) * H;
        for (int k = lane; k < H; k += 32) s += row[k] * W7[(long long)k * d + j];
    }
    for (int j = lane; j < d; j += 32) s += gt[(long long)c * d + j] * hdc[(long long)c * d + j];
    s = warp_sum(s);
    if (lane == 0) out[row_map ? row_map[c] : c] = coef * s;
}

__global__ void div_finish_kernel(int n, int n_tiles, const float* __restrict__ partial, float coef, float* __restrict__ out,
                                  const int* __restrict__ n_rows_dev, const int* __restrict__ row_map) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (n_rows_dev) n = min(n, *n_rows_dev);
    if (c >= n) return;
    float s = 0.0f;
    for (int t = 0; t < n_tiles; ++t) s += partial[(long long)c * n_tiles + t];
    out[row_map ? row_map[c] : c] = coef * s;
}

// ---------------------------------------------------------------------------------------------
// field evaluation
// ---------------------------------------------------------------------------------------------
size_t field_bufs_bytes(const mfm_field_t& F, const mfm_target_t& T, int n, bool hutch) {
    const size_t H = F.hidden, d = F.dim, N = n;
    size_t b = ws_slice(N * 2 * F.fourier_dim, 4) + ws_slice(N * H, 4) * 6 + ws_slice(N * 2 * H, 4) + ws_slice(N * d, 4) * 3;
    if (hutch) b += ws_slice(N * H, 4) + ws_slice(N * d, 4) + ws_slice(N * gemm_n_tiles((int)d), 4);
    else b += 2 * ws_slice(N * d * H, 4);
    b += ws_slice(N * 2 * F.fourier_dim, 4) + ws_slice(N * H, 4) * 6 + ws_slice(N * 2 * H, 4);      // pre-split copies (ff, h0, h2, h5, h6, ta, tb, cat)
    if (F.act != MFM_ACT_RELU) b += ws_slice(N * H, 4) * 4 + ws_slice(N * 2 * H, 4);                // activation derivatives
    if (T.kind == MFM_TARGET_PINES_WHITE) b += 4 * ws_slice(N * d, 4);
    return b + 3 * ws_slice((size_t)F.n_params, 4) + ws_slice(AM_POOL, 4);
}

bool field_bufs_take(FieldBufs& B, Workspace& w, const mfm_field_t& F, int n, bool hutch, const mfm_target_t* T) {
    const size_t H = F.hidden, d = F.dim, N = n;
    B.ff = w.take<float>(N * 2 * F.fourier_dim);
    B.h0 = w.take<float>(N * H); B.h2 = w.take<float>(N * H); B.h5 = w.take<float>(N * H); B.h6 = w.take<float>(N * H);
    B.ta = w.take<float>(N * H); B.tb = w.take<float>(N * H);
    B.cat = w.take<float>(N * 2 * H);
    B.gt = w.take<float>(N * d); B.gc = w.take<float>(N * d); B.hx = w.take<float>(N * d);
    B.zw2 = B.zkinv = B.divpart = B.tan_a = B.tan_b = nullptr;
    if (hutch) { B.zw2 = w.take<float>(N * H); B.zkinv = w.take<float>(N * d); B.divpart = w.take<float>(N * gemm_n_tiles((int)d)); }
    else { B.tan_a = w.take<float>(N * d * H); B.tan_b = w.take<float>(N * d * H); }
    B.wt = w.take<float>((size_t)F.n_params);
    B.wx = w.take<float>((size_t)F.n_params); B.wxo = w.take<float>((size_t)F.n_params);
    B.amax = w.take<float>(AM_POOL);
    B.ff_s = w.take<float>(N * 2 * F.fourier_dim);
    B.h0_s = w.take<float>(N * H); B.h2_s = w.take<float>(N * H); B.h5_s = w.take<float>(N * H); B.h6_s = w.take<float>(N * H);
    B.ta_s = w.take<float>(N * H); B.tb_s = w.take<float>(N * H);
    B.cat_s = w.take<float>(N * 2 * H);
    B.dh0 = B.dh2 = B.dh5 = B.dh6 = B.dcat = nullptr;
    if (F.act != MFM_ACT_RELU) {
        B.dh0 = w.take<float>(N * H); B.dh2 = w.take<float>(N * H); B.dh5 = w.take<float>(N * H); B.dh6 = w.take<float>(N * H);
        B.dcat = w.take<float>(N * 2 * H);
    }
    B.tscratch = nullptr;
    if (T && T->kind == MFM_TARGET_PINES_WHITE) { B.tscratch = w.take<float>(N * d); w.take<float>(N * d); w.take<float>(N * d); w.take<float>(N * d); }
    // fewer than 256 rows in every dense layer (tangent rows of the exact divergence included): nothing reaches the CTA-pair
    // tcgen05 kernel, so the per-call weight preparation for it (maximum, operator norms, two mirrors) and the maxima
    // bookkeeping are skipped altogether - at the small reference shapes they cost more than the layers themselves; the same for
    // narrow networks (hidden < 512: memory-bound layers, see h16_min_hidden)
    if (N * (hutch ? 1 : d) < 256 || (int)H < tc2h::h16_min_hidden()) {
        B.amax = nullptr; B.wx = B.wxo = nullptr;
        B.ff_s = B.h0_s = B.cat_s = B.h2_s = B.h5_s = B.h6_s = B.ta_s = B.tb_s = nullptr;
    }
    return w.ok;
}

#define W_(i) (F.params + F.w_off[i])
#define WT_(i) (B.wt + F.w_off[i])
#define B_(i) (F.params + F.b_off[i])

// per-solve constants of the Hutchinson estimator: z W2 and (pines) z K^-1
static int field_prepare_probe(const mfm_field_t& F, const mfm_target_t& T, int n, const float* z, FieldBufs& B, cudaStream_t st,
                               float z_bound) {
    const int d = F.dim, H = F.hidden;
    DenseAmax am; am.a_bound = z_bound;
    if (tc2h::gemm_h16() && B.amax) {       // exact max |z W2|: scales the gated tangent's pre-split copy in every field evaluation of the solve
        MFM_CUDA_CHECK(cudaMemsetAsync(B.amax + AM_ZW2, 0, sizeof(float), st));
        am.out = B.amax + AM_ZW2;
    }
    int rc = dense(n, d, H, z, d, WT_(2), d, nullptr, 0, B.zw2, H, nullptr, 0, 1, st, nullptr, am);
    if (rc) return rc;
    if (T.kind == MFM_TARGET_PINES) return pines_kinv_gemm(T, n, z, d, B.zkinv, d, nullptr, st, z_bound);
    return MFM_OK;
}

// |jax.random.normal| < 8 for float32 draws: the uniform is clipped to [nextafter(-1, 0), 1 - 2^-23] and sqrt(2) erfinv of
// that is within +-5.5 - a host-known bound for the probes this library draws itself (caller-supplied probes get a reduction)
static constexpr float NORMAL_BOUND = 8.0f;

// out_v[n,d] = sgn * v(x, tfield);  out_l[n] = -sgn * div v   (z != null: Hutchinson; else exact)
int field_eval(const mfm_field_t& F, const mfm_target_t& T, int n, const float* x, const float* tfield,
               const float* z, float sgn, float* out_v, float* out_l, FieldBufs& B, cudaStream_t st,
               const int* nr, const int* row_map, const float* x_amax, const float* x_split) {
    const float* zw2_amax = (tc2h::gemm_h16() && B.amax && z) ? B.amax + AM_ZW2 : nullptr;   // written by field_prepare_probe
    const int d = F.dim, H = F.hidden, Fd = F.fourier_dim;
    int rc;
    // tensor maxima for the scaled-fp16 GEMMs (AmaxSlot): this evaluation's slots start from zero; x gets one reduction
    // when its producer did not track it (it feeds Dense_2 and, for pines, the K^-1 GEMM)
    float* am = tc2h::gemm_h16() ? B.amax : nullptr;
    auto slot = [&](int i) -> float* { return am ? am + i : nullptr; };
    if (am) {
        MFM_CUDA_CHECK(cudaMemsetAsync(am, 0, AM_EVAL_END * sizeof(float), st));
        if (!x_amax && d % 16 == 0 && n >= 256) {
            MFM_CUDA_CHECK(tc2h::launch_absmax(x, d, n, d, nr, am + AM_X, st));
            x_amax = am + AM_X;
        }
    }
    // pre-split copies: a layer's result leaves the epilogue in tensor-core format too (EpiStdS) and the consuming layer's TMA
    // loads that copy (no splitter work, a quarter less shared-memory traffic in the consumer)
    static const bool no_split = getenv("MFM_H16_NOSPLIT") != nullptr;      // debug: every layer splits its own A operand
    const bool sp = !no_split && am != nullptr && B.h0_s != nullptr && H % 16 == 0 && (2 * Fd) % 16 == 0 && n >= 256 && ((reinterpret_cast<uintptr_t>(B.h0_s) | reinterpret_cast<uintptr_t>(B.cat_s)) & 63) == 0;
    auto BD = [&](int i) -> float* { return am + AM_BOUND + i; };
    auto WC = [&](int l) -> const float* { return am + AM_WNORM_COL + l; };
    auto BA = [&](int l) -> const float* { return am + AM_BIAS + l; };
    // (exact max of A [, second slot], host bound) -> exact max of C
    auto A_ = [&](const float* a, const float* a2, float bound, float* out) { DenseAmax m; m.a = a; m.a2 = a2; m.a_bound = bound; m.out = out; return m; };
    // ... A pre-split (copy, slot its scale came from)
    auto IN_ = [&](DenseAmax m, const float* a_split, const float* src) { if (sp) { m.a_split = a_split; m.a_scale_src = src; } return m; };
    // ... C pre-split too (copy, slot id of its bound, layer whose column norm / bias bound the product)
    auto OUT_ = [&](DenseAmax m, float* c_split, int slot_id, int layer, bool has_bias) {
        if (sp) { m.out_split = c_split; m.out_bound = BD(slot_id); m.w_norm = WC(layer); m.bias_amax = has_bias ? BA(layer) : nullptr; }
        return m;
    };
    // activation (mfm_field_t::act): relu gates by the sign of the stored output; the others store act'(pre-activation) next
    // to the output (D_) and every later gate multiplies by it (M_)
    const int act = F.act + 1;                        // functor code: 1 relu, 2 tanh, 3 elu, 4 gelu, 5 swish
    const bool dmul = F.act != MFM_ACT_RELU;
    auto D_ = [&](DenseAmax m, float* dbuf, long long ld) { if (dmul) { m.dact = dbuf; m.lddact = ld; } return m; };
    auto M_ = [&](DenseAmax m) { m.mask_mul = dmul ? 1 : 0; return m; };
    const float* g_h2 = dmul ? B.dh2 : B.h2; const float* g_cat = dmul ? B.dcat : B.cat;
    const float* g_h5 = dmul ? B.dh5 : B.h5; const float* g_h6 = dmul ? B.dh6 : B.h6;
    fourier_kernel<<<ceil_div((long long)n * Fd, 256), 256, 0, st>>>(n, Fd, F.omega, tfield, B.ff, nr, sp ? B.ff_s : nullptr, sp ? BD(AM_FF) : nullptr);
    MFM_LAUNCH_CHECK();
    // first layers of the two branches (the exact maxima of h0 and h2 feed the COMMON scale of cat = [s_x | s_t])
    if ((rc = dense(n, 2 * Fd, H, B.ff, 2 * Fd, WT_(0), 2 * Fd, B_(0), act, B.h0, H, nullptr, 0, 1, st, nr,
                    D_(OUT_(IN_(A_(nullptr, nullptr, 1.0f, slot(AM_H0)), B.ff_s, BD(AM_FF)), B.h0_s, AM_H0, 0, true), B.dh0, H)))) return rc;      // |cos|, |sin| <= 1
    if ((rc = dense(n, d, H, x, d, WT_(2), d, B_(2), act, B.h2, H, nullptr, 0, 1, st, nr,
                    D_(OUT_((x_split && x_amax) ? IN_(A_(x_amax, nullptr, 0, slot(AM_H2)), x_split, x_amax) : A_(x_amax, nullptr, 0, slot(AM_H2)),
                            B.h2_s, AM_H2, 2, true), B.dh2, H)))) return rc;
    {   // s_t and s_x: one scale for both halves of cat
        DenseAmax mt = OUT_(IN_(A_(slot(AM_H0), nullptr, 0, slot(AM_ST)), B.h0_s, BD(AM_H0)), B.cat_s + H, AM_ST, 1, true);
        // (h2's copy exists only when Dense_2 knew max |x|: dense() needs an input maximum to bound its output)
        DenseAmax mx = OUT_(A_(slot(AM_H2), nullptr, 0, slot(AM_SX)), B.cat_s, AM_SX, 3, true);
        if (x_amax) mx = IN_(mx, B.h2_s, BD(AM_H2));
        if (sp) { mt.alt_amax = slot(AM_H2); mt.alt_w_norm = WC(3); mt.alt_bias = BA(3); mx.alt_amax = slot(AM_H0); mx.alt_w_norm = WC(1); mx.alt_bias = BA(1); }
        if ((rc = dense(n, H, H, B.h0, H, WT_(1), H, B_(1), act, B.cat + H, 2 * H, nullptr, 0, 1, st, nr, D_(mt, dmul ? B.dcat + H : nullptr, 2 * H)))) return rc;       // s_t
        if ((rc = dense(n, H, H, B.h2, H, WT_(3), H, B_(3), act, B.cat, 2 * H, nullptr, 0, 1, st, nr, D_(mx, B.dcat, 2 * H)))) return rc;           // s_x
    }
    if ((rc = dense(n, H, d, B.cat + H, 2 * H, WT_(4), H, B_(4), 0, B.gt, d, nullptr, 0, 1, st, nr, IN_(A_(slot(AM_ST), nullptr, 0, nullptr), B.cat_s + H, BD(AM_ST))))) return rc;       // nn_t
    if ((rc = dense(n, 2 * H, H, B.cat, 2 * H, WT_(5), 2 * H, B_(5), act, B.h5, H, nullptr, 0, 1, st, nr,
                    D_(OUT_(IN_(A_(slot(AM_SX), slot(AM_ST), 0, slot(AM_H5)), B.cat_s, BD(AM_SX)), B.h5_s, AM_H5, 5, true), B.dh5, H)))) return rc;
    if ((rc = dense(n, H, H, B.h5, H, WT_(6), H, B_(6), act, B.h6, H, nullptr, 0, 1, st, nr,
                    D_(OUT_(IN_(A_(slot(AM_H5), nullptr, 0, slot(AM_H6)), B.h5_s, BD(AM_H5)), B.h6_s, AM_H6, 6, true), B.dh6, H)))) return rc;
    // untempered grad logprob (clipped) and the Hessian term of the divergence
    mfm_target_t T1 = T; T1.beta = 1.0f;
    const bool want_div = out_l != nullptr;
    if ((rc = target_field_terms(T1, n, x, z, B.zkinv, F.grad_clip, B.gc, (want_div && z) ? B.hx : nullptr,
                                 (want_div && !z) ? B.hx : nullptr, nr, st, x_amax, B.tscratch, sp ? x_split : nullptr))) return rc;
    {
        GemmShape p{n, d, H, B.h6, (long long)H, WT_(7), (long long)H, nr};
        p.a_amax = slot(AM_H6);
        if (sp) { p.a_split = B.h6_s; p.a_scale_src = BD(AM_H6); }
        EpiFieldV e{out_v, (long long)d, B_(7), B.gt, B.gc, (long long)d, sgn, row_map};
        e.amax_out = am ? B.v_amax : nullptr;
        MFM_CUDA_CHECK((launch_gemm<true, false>(p, e, st)));
    }
    if (!want_div) return MFM_OK;
    if (z) {
        // tangent of the probe through the x branch: z W2 (per-solve constant, its exact maximum in AM_ZW2 when the caller
        // tracked it) gated by relu'(h2); gating only zeroes entries, so that maximum also scales the pre-split copy
        const bool spt = sp && zw2_amax != nullptr;
        if (H % 4 == 0 && ((reinterpret_cast<uintptr_t>(B.zw2) | reinterpret_cast<uintptr_t>(B.h2) | reinterpret_cast<uintptr_t>(B.ta)) & 15) == 0)
            gate4_kernel<<<ceil_div((long long)n * (H / 4), 256), 256, 0, st>>>((long long)n * (H / 4), H / 4, reinterpret_cast<const float4*>(B.zw2),
                                                                                reinterpret_cast<const float4*>(g_h2), H / 4, reinterpret_cast<float4*>(B.ta), nr, slot(AM_TA0),
                                                                                spt ? B.ta_s : nullptr, zw2_amax, dmul ? 1 : 0);
        else
            gate_kernel<<<ceil_div((long long)n * H, 256), 256, 0, st>>>((long long)n * H, H, B.zw2, g_h2, H, B.ta, nr, slot(AM_TA0), dmul ? 1 : 0);
        MFM_LAUNCH_CHECK();
        const bool vec_gate = spt && H % 4 == 0 && ((reinterpret_cast<uintptr_t>(B.zw2) | reinterpret_cast<uintptr_t>(B.h2) | reinterpret_cast<uintptr_t>(B.ta)) & 15) == 0;
        DenseAmax m1 = OUT_(A_(slot(AM_TA0), nullptr, 0, slot(AM_TB0)), B.tb_s, AM_TB0, 3, false);
        if (vec_gate) { m1.a_split = B.ta_s; m1.a_scale_src = zw2_amax; }
        if ((rc = dense(n, H, H, B.ta, H, WT_(3), H, nullptr, 0, B.tb, H, g_cat, 2 * H, 1, st, nr, M_(m1)))) return rc;
        if ((rc = dense(n, H, H, B.tb, H, WT_(5), 2 * H, nullptr, 0, B.ta, H, g_h5, H, 1, st, nr,
                        M_(OUT_(IN_(A_(slot(AM_TB0), nullptr, 0, slot(AM_TA1)), B.tb_s, BD(AM_TB0)), B.ta_s, AM_TA1, 5, false))))) return rc;   // first H rows of W5
        if ((rc = dense(n, H, H, B.ta, H, WT_(6), H, nullptr, 0, B.tb, H, g_h6, H, 1, st, nr,
                        M_(OUT_(IN_(A_(slot(AM_TA1), nullptr, 0, slot(AM_TB1)), B.ta_s, BD(AM_TA1)), B.tb_s, AM_TB1, 6, false))))) return rc;
        GemmShape p{n, d, H, B.tb, (long long)H, WT_(7), (long long)H, nr};
        p.a_amax = slot(AM_TB1);
        if (sp) { p.a_split = B.tb_s; p.a_scale_src = BD(AM_TB1); }
        const int nt = gemm_n_tiles(d);
        EpiFieldDiv e{z, B.gt, B.hx, (long long)d, B.divpart, nt};
        MFM_CUDA_CHECK((launch_gemm<true, false>(p, e, st)));
        div_finish_kernel<<<ceil_div(n, 256), 256, 0, st>>>(n, nt, B.divpart, -sgn, out_l, nr, row_map);
        MFM_LAUNCH_CHECK();
    } else {
        const long long rows = (long long)n * d;
        if (rows > 0x7FFFFFFFll) { mfm_set_last_error_msg("exact divergence: n*d too large"); return MFM_ERR_UNSUPPORTED; }
        if (nr) { mfm_set_last_error_msg("internal: compaction is not used with the exact divergence"); return MFM_ERR_UNSUPPORTED; }
        basis_tangent_kernel<<<ceil_div(rows * H, 256), 256, 0, st>>>(n, d, H, W_(2), g_h2, B.tan_a, nullptr, dmul ? 1 : 0);
        MFM_LAUNCH_CHECK();
        // the basis tangents are entries of W2 or zero (relu): max |parameter| bounds them; the other activations' derivatives
        // reach 1.13 (gelu), so their tangents get an on-the-fly maximum instead
        if ((rc = dense((int)rows, H, H, B.tan_a, H, WT_(3), H, nullptr, 0, B.tan_b, H, g_cat, 2 * H, d, st, nullptr, M_(A_(dmul ? nullptr : slot(AM_W), nullptr, 0, slot(AM_TB0)))))) return rc;
        if ((rc = dense((int)rows, H, H, B.tan_b, H, WT_(5), 2 * H, nullptr, 0, B.tan_a, H, g_h5, H, d, st, nullptr, M_(A_(slot(AM_TB0), nullptr, 0, slot(AM_TA1)))))) return rc;
        if ((rc = dense((int)rows, H, H, B.tan_a, H, WT_(6), H, nullptr, 0, B.tan_b, H, g_h6, H, d, st, nullptr, M_(A_(slot(AM_TA1), nullptr, 0, nullptr))))) return rc;
        exact_trace_kernel<<<ceil_div(n, 8), 256, 0, st>>>(n, d, H, B.tan_b, W_(7), B.gt, B.hx, -sgn, out_l, nullptr, row_map);
        MFM_LAUNCH_CHECK();
    }
    return MFM_OK;
}

// ---------------------------------------------------------------------------------------------
// adaptive Dopri5 (jax.experimental.ode semantics)
// ---------------------------------------------------------------------------------------------
struct OdeState {
    float *yx, *yl;            // current state
    float* kx[7]; float* kl[7];
    float *xi, *tf;            // stage input / field time
    float *t, *dt, *d1;        // per-chain time, step, ||f0/scale||
    int *seg, *icount, *ntry;  // segment index, steps in segment, attempts
    float *outx, *outl;        // interpolated output at the final time
    int* counters;             // [0] chains still active, [1] accepted, [2] attempted, [3] max attempts
    // active-chain compaction (Hutchinson path): stage inputs and all field activations live in
    // compact rows r < n_active, row r <-> chain idx[r]; finished chains cost nothing.
    int* idx; int* n_active;   // n_active == &counters[8]
    float *z_full, *zw2_full, *zkinv_full;   // per-solve probe constants in chain order
};

struct OdeTimes { int n_seg; float target[16]; };

__global__ void ode_init_kernel(int n, int d, const float* __restrict__ y0, OdeState S, float t0, float sgn) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < (long long)n * d) { const float v = y0[i]; S.yx[i] = v; S.outx[i] = v; S.xi[i] = v; }
    if (i < n) {
        S.yl[i] = 0.0f; S.outl[i] = 0.0f; S.t[i] = t0; S.seg[i] = 0; S.icount[i] = 0; S.ntry[i] = 0;
        S.tf[i] = sgn > 0 ? t0 : 1.0f - t0;
    }
    if (i < 4) S.counters[i] = 0;
    if (i == 0) { S.counters[10] = 0; S.counters[11] = 0; S.counters[12] = 0; }   // 64-bit count of (chain, field evaluation) pairs; loop iterations
}

// initial_step_size part 1: h0 and the trial point y0 + h0 f0
__global__ void ode_h0_kernel(int n, int d, OdeState S, float rtol, float atol, float sgn) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    const float* y = S.yx + (long long)c * d; const float* f = S.kx[0] + (long long)c * d;
    float s0 = 0.0f, s1 = 0.0f;
    for (int i = lane; i < d; i += 32) {
        const float sc = atol + fabsf(y[i]) * rtol;
        const float a = y[i] / sc, b = f[i] / sc;
        s0 += a * a; s1 += b * b;
    }
    if (lane == 0) { const float sc = atol + fabsf(S.yl[c]) * rtol; const float a = S.yl[c] / sc, b = S.kl[0][c] / sc; s0 += a * a; s1 += b * b; }
    const float d0 = sqrtf(warp_sum(s0)), d1 = sqrtf(warp_sum(s1));
    const float h0 = (d0 < 1e-5f || d1 < 1e-5f) ? 1e-6f : 0.01f * d0 / d1;
    float* xi = S.xi + (long long)c * d;
    for (int i = lane; i < d; i += 32) xi[i] = y[i] + h0 * f[i];
    if (lane == 0) {
        S.dt[c] = h0; S.d1[c] = d1;
        const float tt = S.t[c] + h0;
        S.tf[c] = sgn > 0 ? tt : 1.0f - tt;
    }
}

// initial_step_size part 2: d2, h1, dt = min(100 h0, h1)
__global__ void ode_h1_kernel(int n, int d, OdeState S, float rtol, float atol) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    const float* y = S.yx + (long long)c * d;
    const float* f0 = S.kx[0] + (long long)c * d; const float* f1 = S.kx[1] + (long long)c * d;
    float s2 = 0.0f;
    for (int i = lane; i < d; i += 32) {
        const float sc = atol + fabsf(y[i]) * rtol;
        const float a = (f1[i] - f0[i]) / sc; s2 += a * a;
    }
    if (lane == 0) { const float sc = atol + fabsf(S.yl[c]) * rtol; const float a = (S.kl[1][c] - S.kl[0][c]) / sc; s2 += a * a; }
    const float h0 = S.dt[c], d1 = S.d1[c];
    const float d2 = sqrtf(warp_sum(s2)) / h0;
    float h1;
    if (d1 <= 1e-15f && d2 <= 1e-15f) h1 = fmaxf(1e-6f, h0 * 1e-3f);
    else {
        const float m = (isnan(d1) || isnan(d2)) ? NAN : fmaxf(d1, d2);
        h1 = powf(0.01f / m, 0.2f);
    }
    float dt = (isnan(h1)) ? NAN : fminf(100.0f * h0, h1);
    if (dt < 0.0f) dt = 0.0f;       // jnp.clip(., 0, hmax=inf)
    if (lane == 0) S.dt[c] = dt;
}

// stage s in 1..6: xi = y + dt * sum_j beta[s-1][j] k_j ; field time t + alpha dt.
// Writes compact row r (chain idx[r]) when idx != null.
__global__ void ode_stage_kernel(int n, int d, int s, OdeState S, int n_seg, float sgn, const int* __restrict__ idx,
                                 const int* __restrict__ n_active, float* __restrict__ amax) {
    __shared__ float red[32];
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx) n = min(n, *n_active);
    float m = 0.0f;
    if (i < (long long)n * d) {
        const int r = (int)(i / d), col = (int)(i % d);
        const int c = idx ? idx[r] : r;
        if (S.seg[c] < n_seg) {                  // finished chain: leave its stage input untouched
            const long long o = (long long)c * d + col;
            const float h = S.dt[c];
            float acc = 0.0f;
#pragma unroll
            for (int j = 0; j < 6; ++j) if (j < s) acc += c_beta[s - 1][j] * S.kx[j][o];
            const float v = S.yx[o] + h * acc;
            S.xi[i] = v; m = fabsf(v);
            if (col == 0) {
                const float ti = S.t[c] + h * c_alpha[s - 1];
                S.tf[r] = sgn > 0 ? ti : 1.0f - ti;
            }
        }
    }
    if (amax) amax_publish_block(amax, m, red);  // the stage input is the A operand of Dense_2 (and of the pines K^-1 GEMM)
}

// same, four columns per thread (d % 4 == 0): (s + 2) arrays of 4 B per element, HBM-bound
__global__ void ode_stage4_kernel(int n, int d4, int s, OdeState S, int n_seg, float sgn, const int* __restrict__ idx,
                                  const int* __restrict__ n_active, float* __restrict__ amax) {
    __shared__ float red[32];
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx) n = min(n, *n_active);
    float m = 0.0f;
    if (i < (long long)n * d4) {
        const int r = (int)(i / d4), col = (int)(i % d4);
        const int c = idx ? idx[r] : r;
        if (S.seg[c] < n_seg) {                  // finished chain: leave its stage input untouched
            const long long o = (long long)c * d4 + col;
            const float h = S.dt[c];
            float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
            for (int j = 0; j < 6; ++j)
                if (j < s) {
                    const float b = c_beta[s - 1][j];
                    const float4 k = __ldg(reinterpret_cast<const float4*>(S.kx[j]) + o);
                    acc.x += b * k.x; acc.y += b * k.y; acc.z += b * k.z; acc.w += b * k.w;     // same order as the scalar kernel
                }
            const float4 y = __ldg(reinterpret_cast<const float4*>(S.yx) + o);
            const float4 v = make_float4(y.x + h * acc.x, y.y + h * acc.y, y.z + h * acc.z, y.w + h * acc.w);
            reinterpret_cast<float4*>(S.xi)[i] = v; m = amax4(0.0f, v);
            if (col == 0) {
                const float ti = S.t[c] + h * c_alpha[s - 1];
                S.tf[r] = sgn > 0 ? ti : 1.0f - ti;
            }
        }
    }
    if (amax) amax_publish_block(amax, m, red);
}

// deterministic stream compaction of the chains that are still integrating (single block)
__global__ void __launch_bounds__(1024) ode_compact_kernel(int n, int n_seg, const int* __restrict__ seg, int* __restrict__ idx,
                                                           int* __restrict__ n_active, long long* __restrict__ chain_evals) {
    __shared__ int wsum[32];
    __shared__ int total;
    const int per = (n + 1023) / 1024;
    const int b = threadIdx.x * per, e = min(n, b + per);
    int cnt = 0;
    for (int c = b; c < e; ++c) cnt += seg[c] < n_seg;
    // block exclusive scan of cnt
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (w == 0) {
        int v = wsum[lane], iv = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, iv, o); if (lane >= o) iv += u; }
        wsum[lane] = iv - v;
        if (lane == 31) total = iv;
    }
    __syncthreads();
    int pos = wsum[w] + inc - cnt;
    for (int c = b; c < e; ++c) if (seg[c] < n_seg) idx[pos++] = c;
    if (threadIdx.x == 0) { *n_active = total; *chain_evals += 6ll * total; }    // the next RK iteration evaluates 6 stages on `total` rows
}

// gather the per-solve probe constants of the active chains into compact rows
__global__ void ode_gather_probe_kernel(int n, int d, int H, const int* __restrict__ idx, const int* __restrict__ n_active,
                                        const float* __restrict__ z_full, const float* __restrict__ zw2_full,
                                        const float* __restrict__ zkinv_full, float* __restrict__ z, float* __restrict__ zw2,
                                        float* __restrict__ zkinv) {
    const int r = blockIdx.x;
    if (r >= min(n, *n_active)) return;
    const long long c = idx[r];
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
        z[(long long)r * d + i] = z_full[c * d + i];
        if (zkinv_full) zkinv[(long long)r * d + i] = zkinv_full[c * d + i];
    }
    for (int i = threadIdx.x; i < H; i += blockDim.x) zw2[(long long)r * H + i] = zw2_full[c * H + i];
}

__device__ __forceinline__ float fit_eval(float y0, float y1, float ymid, float dy0, float dy1, float h, float rel) {
    // fit_4th_order_polynomial + polyval (jax/experimental/ode.py)
    const float a = -2.f * h * dy0 + 2.f * h * dy1 - 8.f * y0 - 8.f * y1 + 16.f * ymid;
    const float b = 5.f * h * dy0 - 3.f * h * dy1 + 18.f * y0 + 14.f * y1 - 32.f * ymid;
    const float c = -4.f * h * dy0 + h * dy1 - 11.f * y0 - 5.f * y1 + 16.f * ymid;
    const float dd = h * dy0;
    return (((a * rel + b) * rel + c) * rel + dd) * rel + y0;
}

}  // namespace mfm
#include "targets.cuh"
#include "ode_small.cuh"      // the fused one-launch solve for the small reference shapes (uses the tableau and fit_eval above)
namespace mfm {

// error ratio, accept/reject, controller, FSAL, dense output.  One warp per chain.
__global__ void ode_finish_kernel(int n, int d, OdeState S, OdeTimes TS, float rtol, float atol, int mxstep) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    int seg = S.seg[c];
    if (seg >= TS.n_seg) return;
    const float tt = S.t[c], h = S.dt[c];
    const long long o = (long long)c * d;
    float sum = 0.0f;
    for (int i = lane; i < d; i += 32) {
        float ss = 0.0f, se = 0.0f;
#pragma unroll
        for (int j = 0; j < 7; ++j) { const float k = S.kx[j][o + i]; ss += c_sol[j] * k; se += c_err[j] * k; }
        const float y = S.yx[o + i];
        const float y1 = h * ss + y;
        const float r = (h * se) / (atol + rtol * fmaxf(fabsf(y), fabsf(y1)));
        sum += r * r;
    }
    float ssl = 0.0f, sel = 0.0f;
#pragma unroll
    for (int j = 0; j < 7; ++j) { const float k = S.kl[j][c]; ssl += c_sol[j] * k; sel += c_err[j] * k; }
    const float yl = S.yl[c];
    const float yl1 = h * ssl + yl;
    if (lane == 0) { const float r = (h * sel) / (atol + rtol * fmaxf(fabsf(yl), fabsf(yl1))); sum += r * r; }
    sum = warp_sum(sum);
    const float ratio = sqrtf(sum / (float)(d + 1));
    const bool accept = ratio <= 1.0f;                       // NaN -> reject
    // optimal_step_size
    float new_dt;
    if (isnan(ratio)) new_dt = NAN;
    else if (ratio == 0.0f) new_dt = h * 10.0f;
    else {
        const float dfac = ratio < 1.0f ? 1.0f : 0.2f;
        const float fac = fminf(10.0f, fmaxf(powf(ratio, -0.2f) * 0.9f, dfac));
        new_dt = h * fac;
    }
    if (new_dt < 0.0f) new_dt = 0.0f;
    float t_new = tt;
    if (accept) {
        t_new = tt + h;
        const float t_final = TS.target[TS.n_seg - 1];
        const float rel = (t_final - tt) / (t_new - tt);
        for (int i = lane; i < d; i += 32) {
            float ss = 0.0f, sm = 0.0f;
            float k0 = 0.f, k6 = 0.f;
#pragma unroll
            for (int j = 0; j < 7; ++j) {
                const float k = S.kx[j][o + i]; ss += c_sol[j] * k; sm += c_mid[j] * k;
                if (j == 0) k0 = k; if (j == 6) k6 = k;
            }
            const float y = S.yx[o + i];
            const float y1 = h * ss + y, ymid = y + h * sm;
            S.outx[o + i] = fit_eval(y, y1, ymid, k0, k6, h, rel);
            S.yx[o + i] = y1;
            S.kx[0][o + i] = k6;                               // FSAL
        }
        if (lane == 0) {
            float sm = 0.0f;
#pragma unroll
            for (int j = 0; j < 7; ++j) sm += c_mid[j] * S.kl[j][c];
            S.outl[c] = fit_eval(yl, yl1, yl + h * sm, S.kl[0][c], S.kl[6][c], h, rel);
            S.yl[c] = yl1; S.kl[0][c] = S.kl[6][c]; S.t[c] = t_new;
        }
    }
    if (lane == 0) {
        int ic = S.icount[c] + 1;
        const int ntry = S.ntry[c] + 1;
        S.ntry[c] = ntry;
        S.dt[c] = new_dt;
        // advance over finished output segments: while !(t < target && i < mxstep && dt > 0)
        while (seg < TS.n_seg && !(t_new < TS.target[seg] && ic < mxstep && new_dt > 0.0f)) { ++seg; ic = 0; }
        S.seg[c] = seg; S.icount[c] = ic;
        if (seg < TS.n_seg) atomicAdd(&S.counters[0], 1);
        if (accept) atomicAdd(&S.counters[1], 1);
        atomicAdd(&S.counters[2], 1);
        atomicMax(&S.counters[3], ntry);
    }
}

__global__ void copy_out_kernel(int n, int d, const float* __restrict__ sx, const float* __restrict__ sl,
                                float* __restrict__ y1, float* __restrict__ ldj) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < (long long)n * d) y1[i] = sx[i];
    if (i < n && ldj) ldj[i] = sl[i];
}

// stats: int32[8] = {accepted, attempted, max attempts per chain, field evaluations, chain-evaluations (int64 in [4..5]), 0, 0};
// chain-evaluations = sum over field evaluations of the rows actually evaluated (active-chain compaction)
__global__ void write_stats_kernel(const int* __restrict__ counters, int n_eval, long long host_chain_evals, int* __restrict__ stats,
                                   int accumulate) {
    if (threadIdx.x == 0) {
        // device-resident loop: n_eval < 0 carries -(evaluations before the loop), counters[12] the iterations the loop ran;
        // host_chain_evals < 0 carries -n (every evaluation ran on all n rows: no compaction)
        if (n_eval == INT_MIN) n_eval = 2 + 6 * counters[3];          // fused small-shape solve: as many lock-step iterations as the slowest chain took
        else if (n_eval < 0) n_eval = -n_eval + 6 * counters[12];
        if (host_chain_evals < 0) host_chain_evals = -host_chain_evals * n_eval;
        const long long ce = *reinterpret_cast<const long long*>(counters + 10) + host_chain_evals;
        long long* out_ce = reinterpret_cast<long long*>(stats + 4);
        if (accumulate) { stats[0] += counters[1]; stats[1] += counters[2]; stats[2] = max(stats[2], counters[3]); stats[3] += n_eval; *out_ce += ce; }
        else { stats[0] = counters[1]; stats[1] = counters[2]; stats[2] = counters[3]; stats[3] = n_eval; *out_ce = ce; stats[6] = 0; stats[7] = 0; }
    }
}

// ---- device-resident Runge-Kutta loop: CUDA-graph WHILE node -------------------------------------------------------------
// condition of the next iteration: chains still integrating and the iteration budget (n_seg * mxstep + 2, as the host loop)
__global__ void ode_loop_cond_kernel(cudaGraphConditionalHandle handle, int* __restrict__ counters, long long max_iter) {
    if (threadIdx.x == 0) {
        const int it = ++counters[12];
        cudaGraphSetConditional(handle, (counters[0] > 0 && it < max_iter) ? 1u : 0u);
    }
}
// everything the captured iteration depends on: descriptors by value (beta zeroed: the field uses the untempered target),
// the buffers (workspace identity) and the GEMM switches.  An instantiated graph is reused while the key is unchanged - a
// HotLoop calls with the same workspace and parameter buffer every time.
struct OdeGraphKey {
    mfm_field_t F; mfm_target_t T; mfm_ode_opts_t O; int direction, n, flags; const void *z, *z_compact, *ws, *fb;
};
struct OdeGraphEntry { OdeGraphKey key; cudaGraph_t graph; cudaGraphExec_t exec; int dev; long long max_iter; unsigned long long stamp; bool used; };
static thread_local OdeGraphEntry g_ode_graphs[8];
static thread_local unsigned long long g_ode_graph_stamp = 0;
static int g_ode_small = -1;             // fused one-launch solve for the small shapes (MFM_ODE_SMALL=0 switches it off)
static bool ode_small_enabled() {
    if (g_ode_small < 0) { const char* e = getenv("MFM_ODE_SMALL"); g_ode_small = (e && e[0] == '0') ? 0 : 1; }
    return g_ode_small != 0;
}
static int g_ode_graph_mode = -1;        // -1 unread, 0 never, 1 always, 2 auto (small ensembles)
static bool ode_use_graph(long long elements) {
    if (g_ode_graph_mode < 0) {
        const char* e = getenv("MFM_ODE_GRAPH");
        g_ode_graph_mode = (e && e[0] == '0') ? 0 : ((e && e[0] == '1') ? 1 : 2);
    }
    // big ensembles keep the host-driven loop: their iterations take tens of milliseconds (one poll each is free) and the
    // persistent GEMM's stream-K remainder rounds are not capturable (a replay would meet its own stale flags)
    return g_ode_graph_mode == 1 || (g_ode_graph_mode == 2 && elements <= (4ll << 20));
}
static cudaStream_t ode_capture_stream(int dev) {
    static thread_local cudaStream_t s[16] = {};
    if (dev < 0 || dev >= 16) return nullptr;
    if (!s[dev] && cudaStreamCreateWithFlags(&s[dev], cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); s[dev] = nullptr; }
    return s[dev];
}
template <class Body>
static int ode_graph_launch(const OdeGraphKey& key, cudaStream_t st, int* counters, long long max_iter, Body&& body) {
    int dev = 0;
    MFM_CUDA_CHECK(cudaGetDevice(&dev));
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) { cudaGetLastError(); return MFM_ERR_UNSUPPORTED; }   // the caller is capturing: plain loop
    OdeGraphEntry* e = nullptr; OdeGraphEntry* victim = &g_ode_graphs[0];
    for (auto& g : g_ode_graphs) {
        if (g.used && g.dev == dev && g.max_iter == max_iter && memcmp(&g.key, &key, sizeof(key)) == 0) { e = &g; break; }
        if (!g.used || (victim->used && g.stamp < victim->stamp)) victim = &g;
    }
    if (!e) {
        cudaStream_t cap = ode_capture_stream(dev);
        if (!cap || !tc2h::amax_scratch_for(cap)) return MFM_ERR_UNSUPPORTED;
        if (victim->used) {                 // an evicted graph may still be running
            MFM_CUDA_CHECK(cudaDeviceSynchronize());
            cudaGraphExecDestroy(victim->exec); cudaGraphDestroy(victim->graph); victim->used = false;
        }
        cudaGraph_t graph;
        MFM_CUDA_CHECK(cudaGraphCreate(&graph, 0));
        cudaGraphConditionalHandle handle;
        MFM_CUDA_CHECK(cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault));
        cudaGraphNodeParams np = {};
        np.type = cudaGraphNodeTypeConditional;
        np.conditional.handle = handle; np.conditional.type = cudaGraphCondTypeWhile; np.conditional.size = 1;
        cudaGraphNode_t node;
        MFM_CUDA_CHECK(cudaGraphAddNode(&node, graph, nullptr, 0, &np));
        cudaGraph_t loop_body = np.conditional.phGraph_out[0];
        MFM_CUDA_CHECK(cudaStreamBeginCaptureToGraph(cap, loop_body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
        int rc = body(cap);
        if (rc == MFM_OK) {
            ode_loop_cond_kernel<<<1, 32, 0, cap>>>(handle, counters, max_iter);
            if (cudaGetLastError() != cudaSuccess) rc = MFM_ERR_CUDA;
            ++g_mfm_launches;
        }
        cudaGraph_t captured = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(cap, &captured);
        if (rc != MFM_OK || ce != cudaSuccess) { cudaGetLastError(); cudaGraphDestroy(graph); if (rc == MFM_OK) mfm_set_last_error(ce, __FILE__, __LINE__); return rc != MFM_OK ? rc : MFM_ERR_CUDA; }
        cudaGraphExec_t exec;
        const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
        if (ie != cudaSuccess) { cudaGetLastError(); cudaGraphDestroy(graph); mfm_set_last_error(ie, __FILE__, __LINE__); return MFM_ERR_CUDA; }
        victim->key = key; victim->graph = graph; victim->exec = exec; victim->dev = dev; victim->max_iter = max_iter; victim->used = true;
        e = victim;
    }
    e->stamp = ++g_ode_graph_stamp;
    MFM_CUDA_CHECK(cudaGraphLaunch(e->exec, st));
    return MFM_OK;
}

static size_t ode_state_bytes(int n, int d, int H) {
    const size_t N = n, D = d;
    return ws_slice(N * D, 4) * (1 + 7 + 1 + 1 + 2) + ws_slice(N * H, 4) + ws_slice(N, 4) * (1 + 7 + 1 + 3 + 1) + ws_slice(N, 4) * 4 + 512;
}

static bool ode_state_take(OdeState& S, Workspace& w, int n, int d, int H) {
    const size_t N = n, D = d;
    S.z_full = w.take<float>(N * D); S.zkinv_full = w.take<float>(N * D); S.zw2_full = w.take<float>(N * H);
    S.idx = w.take<int>(N);
    S.yx = w.take<float>(N * D); S.xi = w.take<float>(N * D); S.outx = w.take<float>(N * D);
    for (int j = 0; j < 7; ++j) S.kx[j] = w.take<float>(N * D);
    S.yl = w.take<float>(N); S.outl = w.take<float>(N); S.tf = w.take<float>(N); S.t = w.take<float>(N);
    S.dt = w.take<float>(N); S.d1 = w.take<float>(N);
    for (int j = 0; j < 7; ++j) S.kl[j] = w.take<float>(N);
    S.seg = w.take<int>(N); S.icount = w.take<int>(N); S.ntry = w.take<int>(N);
    S.counters = w.take<int>(64);
    S.n_active = S.counters ? S.counters + 8 : nullptr;
    return w.ok;
}

static int* host_flag() {
    static thread_local int* p = nullptr;
    if (!p) { if (cudaMallocHost(&p, 64) != cudaSuccess) p = nullptr; }
    return p;
}

// Solve from y0 over [0,1]; direction +1: (v, -div); -1: (-v(x, 1-s), +div).
// z: Hutchinson probes in chain order (null -> exact trace).  With probes, the chains still
// integrating are compacted to the leading rows every iteration so finished chains cost nothing.
// z_bound: host-known bound on |z| (NORMAL_BOUND for probes drawn by this library), 0 = unknown.
static int ode_solve(const mfm_field_t& F, const mfm_target_t& T, const mfm_ode_opts_t& O, int direction, int n,
                     const float* z, const float* y0, float* y1, float* ldj, int* stats, int stats_accumulate,
                     OdeState& S, FieldBufs& B, float* z_compact, cudaStream_t st, float z_bound = NORMAL_BOUND) {
    const int d = F.dim, H = F.hidden;
    const float sgn = direction >= 0 ? 1.0f : -1.0f;
    if (O.n_times < 2 || O.n_times > 17) { mfm_set_last_error_msg("n_times must be in [2,17]"); return MFM_ERR_ARG; }
    OdeTimes TS; TS.n_seg = O.n_times - 1;
    for (int k = 1; k < O.n_times; ++k) TS.target[k - 1] = (float)((double)k / (double)(O.n_times - 1));
    if (ode_small_enabled() && small::eligible(F, T, n)) {
        // the small reference shapes: the whole solve in ONE launch, 16 chains per CTA (ode_small.cuh)
        small::Args A;
        A.F = F; A.T = T; A.n = n; A.hutch = z != nullptr ? 1 : 0; A.n_seg = TS.n_seg;
        for (int k = 0; k < 16; ++k) A.target[k] = k < TS.n_seg ? TS.target[k] : 0.0f;
        A.rtol = O.rtol; A.atol = O.atol; A.mxstep = O.mxstep; A.sgn = sgn; A.y0 = y0; A.z = z; A.y1 = y1; A.ldj = ldj; A.counters = S.counters; A.wt = B.wt;
        static bool configured = false;
        if (!configured) {
            MFM_CUDA_CHECK(cudaFuncSetAttribute(small::ode_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, small::SMEM_BYTES));
            configured = true;
        }
        MFM_CUDA_CHECK(cudaMemsetAsync(S.counters, 0, 64 * sizeof(int), st));
        small::ode_small_kernel<<<ceil_div(n, small::CH), small::NTHR, small::SMEM_BYTES, st>>>(A);
        MFM_LAUNCH_CHECK();
        if (stats) { write_stats_kernel<<<1, 32, 0, st>>>(S.counters, INT_MIN, 0, stats, stats_accumulate); MFM_LAUNCH_CHECK(); }
        return MFM_OK;
    }
    int* hflag = host_flag();
    if (!hflag) { mfm_set_last_error_msg("cudaMallocHost failed"); return MFM_ERR_CUDA; }
    int rc;
    const int gE = ceil_div((long long)n * d, 256), gW = ceil_div(n, 8);
    const bool compact = z != nullptr;
    ode_init_kernel<<<max(gE, 1), 256, 0, st>>>(n, d, y0, S, 0.0f, sgn);
    MFM_LAUNCH_CHECK();
    if (z) {
        // per-solve constants z W2 and z K^-1 in chain order (B.zw2 / B.zkinv hold them until the first gather)
        if ((rc = field_prepare_probe(F, T, n, z, B, st, z_bound))) return rc;
        if (compact) {
            MFM_CUDA_CHECK(cudaMemcpyAsync(S.zw2_full, B.zw2, (size_t)n * H * 4, cudaMemcpyDeviceToDevice, st));
            if (T.kind == MFM_TARGET_PINES)
                MFM_CUDA_CHECK(cudaMemcpyAsync(S.zkinv_full, B.zkinv, (size_t)n * d * 4, cudaMemcpyDeviceToDevice, st));
        }
    }
    int n_eval = 0;
    if ((rc = field_eval(F, T, n, S.xi, S.tf, z, sgn, S.kx[0], S.kl[0], B, st))) return rc; ++n_eval;
    ode_h0_kernel<<<gW, 256, 0, st>>>(n, d, S, O.rtol, O.atol, sgn);
    MFM_LAUNCH_CHECK();
    if ((rc = field_eval(F, T, n, S.xi, S.tf, z, sgn, S.kx[1], S.kl[1], B, st))) return rc; ++n_eval;
    ode_h1_kernel<<<gW, 256, 0, st>>>(n, d, S, O.rtol, O.atol);
    MFM_LAUNCH_CHECK();
    const int* idx = nullptr; const int* nact = nullptr; const float* zc = z;
    if (compact) {
        ode_compact_kernel<<<1, 1024, 0, st>>>(n, TS.n_seg, S.seg, S.idx, S.n_active, reinterpret_cast<long long*>(S.counters + 10));
        MFM_LAUNCH_CHECK();
        idx = S.idx; nact = S.n_active; zc = z_compact;
    }
    const long long max_iter = (long long)TS.n_seg * (long long)O.mxstep + 2;
    // (the two evaluations above reduced max |xi| into AM_X themselves; the stage kernels keep folding into it)
    float* x_amax = (tc2h::gemm_h16() && B.amax && d % 16 == 0 && n >= 256) ? B.amax + AM_X : nullptr;
    bool stage_vec = d % 4 == 0 && ((reinterpret_cast<uintptr_t>(S.yx) | reinterpret_cast<uintptr_t>(S.xi)) & 15) == 0;
    for (int j = 0; j < 6; ++j) stage_vec = stage_vec && (reinterpret_cast<uintptr_t>(S.kx[j]) & 15) == 0;
    // one iteration of the lock-step Runge-Kutta loop, enqueued on `s`: 6 x (stage input, field evaluation), then the step
    // controller; counters[0] = chains still integrating afterwards
    auto rk_iteration = [&](cudaStream_t s) -> int {
        int rc2;
        if (compact) {
            ode_gather_probe_kernel<<<n, 128, 0, s>>>(n, d, H, idx, nact, z, S.zw2_full,
                                                      T.kind == MFM_TARGET_PINES ? S.zkinv_full : nullptr, z_compact, B.zw2, B.zkinv);
            MFM_LAUNCH_CHECK();
        }
        for (int sg = 1; sg <= 6; ++sg) {
            // the stage input's maximum accumulates over the solve (never reset: a stale, larger maximum is safe)
            if (stage_vec) ode_stage4_kernel<<<ceil_div((long long)n * (d / 4), 256), 256, 0, s>>>(n, d / 4, sg, S, TS.n_seg, sgn, idx, nact, x_amax);
            else ode_stage_kernel<<<gE, 256, 0, s>>>(n, d, sg, S, TS.n_seg, sgn, idx, nact, x_amax);
            MFM_LAUNCH_CHECK();
            if ((rc2 = field_eval(F, T, n, S.xi, S.tf, zc, sgn, S.kx[sg], S.kl[sg], B, s, nact, idx, x_amax))) return rc2;
        }
        MFM_CUDA_CHECK(cudaMemsetAsync(S.counters, 0, sizeof(int), s));
        ode_finish_kernel<<<gW, 256, 0, s>>>(n, d, S, TS, O.rtol, O.atol, O.mxstep);
        MFM_LAUNCH_CHECK();
        if (compact) {
            ode_compact_kernel<<<1, 1024, 0, s>>>(n, TS.n_seg, S.seg, S.idx, S.n_active, reinterpret_cast<long long*>(S.counters + 10));
            MFM_LAUNCH_CHECK();
        }
        return MFM_OK;
    };
    bool looped_on_device = false;
    if (ode_use_graph((long long)n * d)) {
        // device-resident loop: the iteration above is the body of a CUDA-graph WHILE node whose condition a one-thread kernel
        // sets from counters[0] - no host round trip per iteration and graph-internal launch latency between the ~100 kernels
        OdeGraphKey key;
        memset(&key, 0, sizeof(key));
        key.F = F; key.T = T; key.T.beta = 0.0f; key.O = O; key.direction = direction; key.n = n; key.z = z; key.z_compact = z_compact;
        key.ws = S.z_full; key.fb = B.ff; key.flags = tc2h::gemm_h16() * 16 + tc2h::split_groups() + 64 * gemm_backend();
        rc = ode_graph_launch(key, st, S.counters, max_iter, rk_iteration);
        if (rc == MFM_OK) looped_on_device = true;
        else if (rc != MFM_ERR_UNSUPPORTED) return rc;
    }
    if (!looped_on_device)
    for (long long it = 0; it < max_iter; ++it) {
        if ((rc = rk_iteration(st))) return rc;
        n_eval += 6;
        MFM_CUDA_CHECK(cudaMemcpyAsync(hflag, S.counters, sizeof(int), cudaMemcpyDeviceToHost, st));
        MFM_CUDA_CHECK(cudaStreamSynchronize(st));
        if (*hflag == 0) break;
    }
    copy_out_kernel<<<max(gE, 1), 256, 0, st>>>(n, d, S.outx, S.outl, y1, ldj);
    MFM_LAUNCH_CHECK();
    if (stats) {
        // rows evaluated outside the device count: the two evaluations of initial_step_size on all n rows, and without
        // compaction (exact divergence) every evaluation runs on all n rows
        // (device-resident loop: the number of iterations lives in counters[12]; the kernel derives both figures from it)
        const long long host_ce = compact ? 2ll * n : (looped_on_device ? -(long long)n : (long long)n * n_eval);
        write_stats_kernel<<<1, 32, 0, st>>>(S.counters, looped_on_device ? -n_eval : n_eval, host_ce, stats, stats_accumulate); MFM_LAUNCH_CHECK();
    }
    return MFM_OK;
}

// ---------------------------------------------------------------------------------------------
// flow-MH kernels
// ---------------------------------------------------------------------------------------------
// key_gen, key_acc, key_hutch1, key_hutch2 = split(keys[c], 4)   (exe_flow_matching.py:247,265)
__global__ void flow_keys_kernel(const uint32_t* __restrict__ rng_key, int n, int chain_offset, int n_total,
                                 uint32_t* __restrict__ kgen, uint32_t* __restrict__ kacc, uint32_t* __restrict__ kh1,
                                 uint32_t* __restrict__ kh2) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    u32x2 kc;
    if (n_total > 0) kc = threefry_split_key(rng_key[0], rng_key[1], (uint32_t)(chain_offset + c), (uint32_t)n_total);
    else { kc.a = rng_key[2 * c]; kc.b = rng_key[2 * c + 1]; }
    uint32_t* outs[4] = {kgen, kacc, kh1, kh2};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const u32x2 k = threefry_split_key(kc.a, kc.b, (uint32_t)j, 4u);
        outs[j][2 * c] = k.a; outs[j][2 * c + 1] = k.b;
    }
}

// out = a + scale * eps   (:268)
__global__ void axpy_kernel(long long total, const float* __restrict__ a, float scale, const float* __restrict__ eps,
                            float* __restrict__ out) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < total) out[i] = a[i] + scale * eps[i];
}
// out = mean + std * eps   (ref_dist.sample_model, distributions.py:96-97)
__global__ void ref_sample_kernel(long long total, float mean, float std_, const float* __restrict__ eps, float* __restrict__ out) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < total) out[i] = __fadd_rn(mean, __fmul_rn(std_, eps[i]));
}

// log N(x; mean, std) summed over the row (ref_dist.logprob, distributions.py:89-90)
__global__ void gauss_logprob_kernel(int n, int d, const float* __restrict__ x, float mean, float std_, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    const float var = std_ * std_;
    float s = 0.0f;
    for (int i = lane; i < d; i += 32) { const float df = x[(long long)c * d + i] - mean; s += -(logf(6.28318530717958647692f * var) + df * df / var) / 2.0f; }
    s = warp_sum(s);
    if (lane == 0) out[c] = s;
}

// PhiFourBase sample (ref_dist.sample_model with ref_kind MFM_REF_PHI4_BASE): out = L^-T z row by row, one warp per row (ref_dist.cuh);
// z and out may alias.  Dynamic shared memory: band_row_floats(d) floats per warp.
__global__ void __launch_bounds__(256)
ref_band_solve_kernel(int n, int d, const float* __restrict__ band, const float* z, float* out) {
    extern __shared__ float band_rows[];
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    const int m = (d + 31) >> 5, mp = m | 1;
    const float inv_m = 1.0f / (float)m;
    float* r = band_rows + (threadIdx.x >> 5) * 32 * mp;
    for (int j = lane; j < d; j += 32) r[band_slot(j, m, mp, inv_m)] = z[(long long)c * d + j];
    band_solve_warp(r, d, band, lane);
    for (int j = lane; j < d; j += 32) out[(long long)c * d + j] = r[band_slot(j, m, mp, inv_m)];
}

// PhiFourBase log-density (ref_dist.logprob, distributions.py:168-226) in the sum-of-squares form, which has no cancellation:
// -q/2 + log_norm, q = beta c sum_{i=0..d} (x_i - x_{i-1})^2 + (beta / c) sum x_i^2 with x_{-1} = x_d = 0; band[2d] = beta c,
// band[2d + 1] = beta / c.  One warp per row.
__global__ void __launch_bounds__(256)
ref_band_logprob_kernel(int n, int d, const float* __restrict__ band, float log_norm, const float* __restrict__ x, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    const float w_diff = __ldg(band + 2 * d), w_sq = __ldg(band + 2 * d + 1);
    const float* row = x + (long long)c * d;
    float s = 0.0f;
    for (int i = lane; i < d; i += 32) {
        const float xi = row[i];
        const float df = xi - (i > 0 ? row[i - 1] : 0.0f);
        s = fmaf(w_diff, df * df, fmaf(w_sq, xi * xi, s));
    }
    if (lane == 0) { const float xl = row[d - 1]; s = fmaf(w_diff, xl * xl, s); }     // (x_d - x_{d-1})^2
    s = warp_sum(s);
    if (lane == 0) out[c] = fmaf(-0.5f, s, log_norm);
}

// z [n, d] standard normal rows -> reference samples out (may alias z): ref_sample_kernel for IndepGaussian, the band solve for
// PhiFourBase.  One launch either way.
static int ref_transform_rows(const mfm_field_t& f, int n, const float* z, float* out, cudaStream_t stream) {
    const int d = f.dim;
    if (f.ref_kind == MFM_REF_PHI4_BASE) {
        const int wpb = band_warps_per_block(d);
        ref_band_solve_kernel<<<ceil_div(n, wpb), 32 * wpb, (size_t)wpb * band_row_floats(d) * sizeof(float), stream>>>(n, d, f.ref_band, z, out);
    } else {
        const long long tot = (long long)n * d;
        ref_sample_kernel<<<ceil_div(tot, 256), 256, 0, stream>>>(tot, f.ref_mean, f.ref_std, z, out);
    }
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}
// out[c] = ref_dist.logprob(x[c]); one launch
static int ref_logprob_rows(const mfm_field_t& f, int n, const float* x, float* out, cudaStream_t stream) {
    if (f.ref_kind == MFM_REF_PHI4_BASE)
        ref_band_logprob_kernel<<<ceil_div(n, 8), 256, 0, stream>>>(n, f.dim, f.ref_band, f.ref_log_norm, x, out);
    else
        gauss_logprob_kernel<<<ceil_div(n, 8), 256, 0, stream>>>(n, f.dim, x, f.ref_mean, f.ref_std, out);
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}

struct FlowAcceptArgs {
    int variant;
    const float *xp, *lp, *gp, *Vp, *V0, *logq_up, *logq_u0;
    const uint32_t* kacc;
    float *x, *l, *g, *acc_rate, *prop_pos, *prop_w; uint8_t* is_acc;
    int x64;
};

__global__ void flow_accept_kernel(int n, int d, FlowAcceptArgs A) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    float la;
    if (A.variant == MFM_FLOW_RW_MH) la = A.lp[c] - A.Vp[c] - A.l[c] - A.V0[c];                            // :271-274
    else la = A.lp[c] - A.logq_up[c] - A.Vp[c] + A.logq_u0[c] - A.V0[c] - A.l[c];                         // :253-256
    const float acc_prob = expf(la);
    const float u = rng_uniform_at(A.kacc[2 * c], A.kacc[2 * c + 1], 0u, 1u, A.x64);
    const bool acc = u <= acc_prob;                                                                      // :257,275
    for (int i = lane; i < d; i += 32) {
        const float v = A.xp[(long long)c * d + i];
        if (A.prop_pos) A.prop_pos[(long long)c * d + i] = v;
        if (acc) { A.x[(long long)c * d + i] = v; A.g[(long long)c * d + i] = A.gp[(long long)c * d + i]; }
    }
    if (lane == 0) {
        if (acc) A.l[c] = A.lp[c];
        if (A.acc_rate) A.acc_rate[c] = acc_prob;
        if (A.is_acc) A.is_acc[c] = acc ? 1 : 0;
        if (A.prop_w) A.prop_w[c] = 0.0f;
    }
}


// ---- conditional importance sampling (exe_flow_matching.py:280-296) -------------------------------------------------------
// key_sample, key_hutch_prev, key_hutch, key_choice = split(keys[c], 4); row (c, k) of the K fresh samples uses
// split(key_sample, K)[k] for the reference draw and split(key_hutch, K)[k] for its Hutchinson probe  (:281,284,286)
__global__ void cis_keys_kernel(const uint32_t* __restrict__ rng_key, int n, int chain_offset, int n_total, int K,
                                uint32_t* __restrict__ kprev, uint32_t* __restrict__ kchoice, uint32_t* __restrict__ ksample,
                                uint32_t* __restrict__ khutch) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= (long long)n * K) return;
    const int c = (int)(i / K), k = (int)(i % K);
    u32x2 kc;
    if (n_total > 0) kc = threefry_split_key(rng_key[0], rng_key[1], (uint32_t)(chain_offset + c), (uint32_t)n_total);
    else { kc.a = rng_key[2 * c]; kc.b = rng_key[2 * c + 1]; }
    const u32x2 k_sample = threefry_split_key(kc.a, kc.b, 0u, 4u), k_hutch = threefry_split_key(kc.a, kc.b, 2u, 4u);
    const u32x2 ks = threefry_split_key(k_sample.a, k_sample.b, (uint32_t)k, (uint32_t)K);
    const u32x2 kh = threefry_split_key(k_hutch.a, k_hutch.b, (uint32_t)k, (uint32_t)K);
    ksample[2 * i] = ks.a; ksample[2 * i + 1] = ks.b; khutch[2 * i] = kh.a; khutch[2 * i + 1] = kh.b;
    if (k == 0) {
        const u32x2 kp = threefry_split_key(kc.a, kc.b, 1u, 4u), kch = threefry_split_key(kc.a, kc.b, 3u, 4u);
        kprev[2 * c] = kp.a; kprev[2 * c + 1] = kp.b; kchoice[2 * c] = kch.a; kchoice[2 * c + 1] = kch.b;
    }
}

struct CisArgs {
    int K;
    const float *ld, *lq, *vol;            // [n*K] log-density, reference log-density and log-det of the fresh samples
    const float *lq_prev, *vol_prev;       // [n] of the pulled-back current state
    const float* samples;                  // [n*K, d]
    const uint32_t* kchoice;               // [n, 2]
    float* wbuf;                           // [n, K+1] scratch: normalised weights
    float *x, *l, *acc_rate, *prop_pos, *prop_w; uint8_t* is_acc;
    int x64;
};
// one warp per chain: weights, their normalisation, jax.random.choice(key_choice, K + 1, p = norm_weights) as cumsum ->
// r = p_cuml[-1] (1 - uniform) -> searchsorted (sequential float32 sums), then the state / info update of :293-296.
// As coded, an accepted sample keeps the PREVIOUS state's gradient.
__global__ void cis_select_kernel(int n, int d, CisArgs A) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    const int K = A.K;
    float* w = A.wbuf + (long long)c * (K + 1);
    if (lane == 0) w[0] = expf(A.l[c] - A.lq_prev[c] - A.vol_prev[c]);                       // prev_weight (:283)
    for (int k = lane; k < K; k += 32) { const long long r = (long long)c * K + k; w[1 + k] = expf(A.ld[r] - A.lq[r] - A.vol[r]); }   // (:289)
    __syncwarp();
    int choice = 0; float wsel = 0.0f;
    if (lane == 0) {
        float wsum = 0.0f;
        for (int k = 1; k <= K; ++k) wsum += w[k];                                            // weights.sum()
        const float tot = w[0] + wsum;                                                         // (:290)
        float cum = 0.0f;
        for (int k = 0; k <= K; ++k) { w[k] = w[k] / tot; }                                    // norm_weights (:291)
        float total = 0.0f;
        for (int k = 0; k <= K; ++k) total += w[k];                                            // p_cuml[-1]
        const float u = rng_uniform_at(A.kchoice[2 * c], A.kchoice[2 * c + 1], 0u, 1u, A.x64);
        const float r = total * (1.0f - u);
        choice = K + 1;
        for (int k = 0; k <= K; ++k) { cum += w[k]; if (choice > K && cum >= r) choice = k; }   // searchsorted(p_cuml, r), side = left
        if (choice > K) choice = K;                                                            // jnp indexing clamps
        wsel = w[choice];
    }
    choice = __shfl_sync(0xffffffffu, choice, 0); wsel = __shfl_sync(0xffffffffu, wsel, 0);
    const float* src = choice > 0 ? A.samples + ((long long)c * K + (choice - 1)) * d : nullptr;
    for (int i = lane; i < d; i += 32) {
        const float v = src ? src[i] : A.x[(long long)c * d + i];
        if (A.prop_pos) A.prop_pos[(long long)c * d + i] = v;                                  // proposed_position: chosen sample or prev position
        if (src) A.x[(long long)c * d + i] = v;
    }
    if (lane == 0) {
        if (choice > 0) A.l[c] = A.ld[(long long)c * K + (choice - 1)];
        if (A.acc_rate) A.acc_rate[c] = wsel;
        if (A.is_acc) A.is_acc[c] = choice > 0 ? 1 : 0;
        if (A.prop_w) A.prop_w[c] = wsel;
    }
}

}  // namespace mfm

// =============================================================================================
extern "C" {
using namespace mfm;

static int check_field(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o) {
    if (!f || !t || !o) { mfm_set_last_error_msg("null descriptor"); return MFM_ERR_ARG; }
    if (f->dim != t->dim) { mfm_set_last_error_msg("field.dim != target.dim"); return MFM_ERR_ARG; }
    if (f->hidden <= 0 || f->fourier_dim <= 0 || !f->params || !f->omega) { mfm_set_last_error_msg("bad field descriptor"); return MFM_ERR_ARG; }
    if (f->act < MFM_ACT_RELU || f->act > MFM_ACT_SWISH) { mfm_set_last_error_msg("unknown activation (mfm_field_t::act)"); return MFM_ERR_ARG; }
    return ref_check(f, false);
}

void mfm_debug_set_ode_small(int v) { g_ode_small = v ? 1 : 0; }      // test hook (not in the ABI header): fused small-shape solve on / off

size_t mfm_ode_workspace_bytes(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n) {
    return ode_state_bytes(n, f->dim, f->hidden) + field_bufs_bytes(*f, *t, n, o->hutch != 0) + 2 * ws_slice((size_t)n * f->dim, 4) + 1024;
}

int mfm_ode_flow(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int direction, int n,
                 const uint32_t* hutch_keys, const float* y0, float* y1, float* ldj, int* stats, void* ws,
                 size_t ws_bytes, mfm_stream_t stream) {
    mfm::CrossScope cross_scope;
    int rc = check_field(f, t, o);
    if (rc) return rc;
    if (n <= 0) return MFM_OK;
    Workspace w(ws, ws_bytes);
    OdeState S; FieldBufs B;
    ode_state_take(S, w, n, f->dim, f->hidden);
    field_bufs_take(B, w, *f, n, o->hutch != 0, t);
    float* z = nullptr; float* zc = nullptr;
    if (o->hutch) { z = w.take<float>((size_t)n * f->dim); zc = w.take<float>((size_t)n * f->dim); }
    if (!w.ok) { mfm_set_last_error_msg("workspace too small (mfm_ode_flow)"); return MFM_ERR_WORKSPACE; }
    if ((rc = field_prepare_weights(*f, B, stream))) return rc;
    if (o->hutch) {
        if (!hutch_keys) { mfm_set_last_error_msg("hutch_keys required"); return MFM_ERR_ARG; }
        if ((rc = mfm_threefry_normal_batched(hutch_keys, n, f->dim, z, stream))) return rc;
    }
    return ode_solve(*f, *t, *o, direction, n, z, y0, y1, ldj, stats, 0, S, B, zc, stream);
}

int mfm_field_eval(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n, const float* x,
                   const float* time, const float* z, float* v, float* div, void* ws, size_t ws_bytes,
                   mfm_stream_t stream) {
    mfm::CrossScope cross_scope;
    int rc = check_field(f, t, o);
    if (rc) return rc;
    if (n <= 0) return MFM_OK;
    Workspace w(ws, ws_bytes);
    FieldBufs B;
    const bool hutch = o->hutch != 0;
    field_bufs_take(B, w, *f, n, hutch, t);
    float* negdiv = w.take<float>(n);
    if (!w.ok) { mfm_set_last_error_msg("workspace too small (mfm_field_eval)"); return MFM_ERR_WORKSPACE; }
    if (hutch && !z) { mfm_set_last_error_msg("z required for hutch"); return MFM_ERR_ARG; }
    if ((rc = field_prepare_weights(*f, B, stream))) return rc;
    if (hutch && (rc = field_prepare_probe(*f, *t, n, z, B, stream, 0.0f))) return rc;    // caller's probes: no known bound
    // field_eval writes -sgn*div; evaluate with sgn=-1 on a negated... simpler: sgn=+1 then negate
    if ((rc = field_eval(*f, *t, n, x, time, hutch ? z : nullptr, 1.0f, v, div ? negdiv : nullptr, B, stream))) return rc;
    if (div) { axpy_kernel<<<ceil_div(n, 256), 256, 0, stream>>>(n, negdiv, -2.0f, negdiv, div); MFM_LAUNCH_CHECK(); }
    return MFM_OK;
}

size_t mfm_flow_mh_workspace_bytes(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n) {
    const size_t N = n, D = f->dim;
    return mfm_ode_workspace_bytes(f, t, o, n) + ws_slice(N * D, 4) * 6 + ws_slice(N, 4) * 6 + ws_slice(N * 2, 4) * 4 +
           target_ws_bytes(*t, n) + 1024;
}

int mfm_flow_mh_step(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int variant,
                     const uint32_t* rng_key, int per_chain_keys, int n, int chain_offset, int n_total,
                     float* position, float* logdensity, float* logdensity_grad, float* acceptance_rate,
                     uint8_t* is_accepted, float* proposed_position, float* proposed_weight, int* stats, void* ws,
                     size_t ws_bytes, mfm_stream_t stream) {
    mfm::CrossScope cross_scope;
    int rc = check_field(f, t, o);
    if (rc) return rc;
    if (!rng_key || !position || !logdensity || !logdensity_grad) { mfm_set_last_error_msg("null argument"); return MFM_ERR_ARG; }
    if (n <= 0) return MFM_OK;
    if (variant != MFM_FLOW_RW_MH && variant != MFM_FLOW_INDEP_MH) { mfm_set_last_error_msg("unknown flow-MH variant"); return MFM_ERR_ARG; }
    if (variant == MFM_FLOW_INDEP_MH && (rc = ref_check(f, true))) return rc;
    if (per_chain_keys) { chain_offset = 0; n_total = 0; }
    else if (n_total < chain_offset + n || chain_offset < 0) { mfm_set_last_error_msg("bad chain_offset/n_total"); return MFM_ERR_ARG; }
    const int d = f->dim;
    const size_t N = n, D = d;
    Workspace w(ws, ws_bytes);
    OdeState S; FieldBufs B;
    ode_state_take(S, w, n, d, f->hidden);
    field_bufs_take(B, w, *f, n, o->hutch != 0, t);
    float* z = w.take<float>(N * D); float* zc = w.take<float>(N * D);
    float* u0 = w.take<float>(N * D); float* up = w.take<float>(N * D); float* xp = w.take<float>(N * D);
    float* gp = w.take<float>(N * D); float* eps = w.take<float>(N * D);
    float* V0 = w.take<float>(N); float* Vp = w.take<float>(N); float* lp = w.take<float>(N);
    float* lq_up = w.take<float>(N); float* lq_u0 = w.take<float>(N); w.take<float>(N);
    uint32_t* kgen = w.take<uint32_t>(N * 2); uint32_t* kacc = w.take<uint32_t>(N * 2);
    uint32_t* kh1 = w.take<uint32_t>(N * 2); uint32_t* kh2 = w.take<uint32_t>(N * 2);
    Workspace wt((char*)ws + w.off, w.off <= ws_bytes ? ws_bytes - w.off : 0);
    if (!w.ok) { mfm_set_last_error_msg("workspace too small (mfm_flow_mh_step)"); return MFM_ERR_WORKSPACE; }
    const bool hutch = o->hutch != 0;

    if ((rc = field_prepare_weights(*f, B, stream))) return rc;
    flow_keys_kernel<<<ceil_div(n, 128), 128, 0, stream>>>(rng_key, n, chain_offset, n_total, kgen, kacc, kh1, kh2);
    MFM_LAUNCH_CHECK();
    if ((rc = mfm_threefry_normal_batched(kgen, n, d, eps, stream))) return rc;
    const long long tot = (long long)n * d;
    if (variant == MFM_FLOW_RW_MH) {
        // pull back the current position, random-walk in latent space, push forward
        if (hutch && (rc = mfm_threefry_normal_batched(kh2, n, d, z, stream))) return rc;
        if ((rc = ode_solve(*f, *t, *o, -1, n, hutch ? z : nullptr, position, u0, V0, stats, 0, S, B, zc, stream))) return rc;
        const float scale = 2.38f / sqrtf((float)d);                                     // :262
        axpy_kernel<<<ceil_div(tot, 256), 256, 0, stream>>>(tot, u0, scale, eps, up);
        MFM_LAUNCH_CHECK();
        if (hutch && (rc = mfm_threefry_normal_batched(kh1, n, d, z, stream))) return rc;
        if ((rc = ode_solve(*f, *t, *o, +1, n, hutch ? z : nullptr, up, xp, Vp, stats, 1, S, B, zc, stream))) return rc;
    } else {
        // independent proposal from the reference distribution (:48-54,249)
        if ((rc = ref_transform_rows(*f, n, eps, up, stream))) return rc;
        if (hutch && (rc = mfm_threefry_normal_batched(kh1, n, d, z, stream))) return rc;
        if ((rc = ode_solve(*f, *t, *o, +1, n, hutch ? z : nullptr, up, xp, Vp, stats, 0, S, B, zc, stream))) return rc;
        if (hutch && (rc = mfm_threefry_normal_batched(kh2, n, d, z, stream))) return rc;
        if ((rc = ode_solve(*f, *t, *o, -1, n, hutch ? z : nullptr, position, u0, V0, stats, 1, S, B, zc, stream))) return rc;
        if ((rc = ref_logprob_rows(*f, n, up, lq_up, stream))) return rc;                   // (:251-252)
        if ((rc = ref_logprob_rows(*f, n, u0, lq_u0, stream))) return rc;
    }
    if ((rc = target_value_and_grad(*t, n, xp, lp, gp, nullptr, wt, stream))) return rc;
    FlowAcceptArgs A{variant, xp, lp, gp, Vp, V0, lq_up, lq_u0, kacc, position, logdensity, logdensity_grad,
                     acceptance_rate, proposed_position, proposed_weight, is_accepted, rng_x64()};
    flow_accept_kernel<<<ceil_div(n, 8), 256, 0, stream>>>(n, d, A);
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}

size_t mfm_flow_cis_workspace_bytes(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n, int n_is) {
    const size_t N = n, D = f->dim, M = (size_t)n * (n_is > 0 ? n_is : 1);
    return mfm_ode_workspace_bytes(f, t, o, (int)M) + ws_slice(M * D, 4) * 5 + ws_slice(N * D, 4) * 2 + ws_slice(M, 4) * 4 + ws_slice(N, 4) * 3 +
           ws_slice(M * 2, 4) * 2 + ws_slice(N * 2, 4) * 2 + ws_slice(N * (size_t)(n_is + 1), 4) + target_ws_bytes(*t, (int)M) + 2048;
}

int mfm_flow_cis_step(const mfm_field_t* f, const mfm_target_t* t, const mfm_ode_opts_t* o, int n_is, const uint32_t* rng_key,
                      int per_chain_keys, int n, int chain_offset, int n_total, float* position, float* logdensity,
                      float* acceptance_rate, uint8_t* is_accepted, float* proposed_position, float* proposed_weight, int* stats,
                      void* ws, size_t ws_bytes, mfm_stream_t stream) {
    mfm::CrossScope cross_scope;
    int rc = check_field(f, t, o);
    if (rc) return rc;
    if (!rng_key || !position || !logdensity) { mfm_set_last_error_msg("null argument"); return MFM_ERR_ARG; }
    if (n_is <= 0) { mfm_set_last_error_msg("num_importance_samples must be > 0 for conditional importance sampling"); return MFM_ERR_ARG; }
    if ((rc = ref_check(f, true))) return rc;
    if (n <= 0) return MFM_OK;
    if ((long long)n * n_is > 0x7FFFFFFFll) { mfm_set_last_error_msg("n * num_importance_samples too large"); return MFM_ERR_UNSUPPORTED; }
    if (per_chain_keys) { chain_offset = 0; n_total = 0; }
    else if (n_total < chain_offset + n || chain_offset < 0) { mfm_set_last_error_msg("bad chain_offset/n_total"); return MFM_ERR_ARG; }
    const int d = f->dim, K = n_is, M = n * K;
    const size_t N = n, D = d, MM = M;
    const bool hutch = o->hutch != 0;
    Workspace w(ws, ws_bytes);
    OdeState S; FieldBufs B;
    ode_state_take(S, w, M, d, f->hidden);
    field_bufs_take(B, w, *f, M, hutch, t);
    float* z = w.take<float>(MM * D); float* zc = w.take<float>(MM * D);
    float* refs = w.take<float>(MM * D); float* samples = w.take<float>(MM * D); float* gscr = w.take<float>(MM * D);
    float* u_prev = w.take<float>(N * D); w.take<float>(N * D);
    float* vols = w.take<float>(MM); float* ld = w.take<float>(MM); float* lq = w.take<float>(MM); w.take<float>(MM);
    float* vol_prev = w.take<float>(N); float* lq_prev = w.take<float>(N); w.take<float>(N);
    uint32_t* ksample = w.take<uint32_t>(MM * 2); uint32_t* khutch = w.take<uint32_t>(MM * 2);
    uint32_t* kprev = w.take<uint32_t>(N * 2); uint32_t* kchoice = w.take<uint32_t>(N * 2);
    float* wbuf = w.take<float>(N * (size_t)(K + 1));
    Workspace wt((char*)ws + w.off, w.off <= ws_bytes ? ws_bytes - w.off : 0);
    if (!w.ok) { mfm_set_last_error_msg("workspace too small (mfm_flow_cis_step)"); return MFM_ERR_WORKSPACE; }
    if ((rc = field_prepare_weights(*f, B, stream))) return rc;
    cis_keys_kernel<<<ceil_div(M, 128), 128, 0, stream>>>(rng_key, n, chain_offset, n_total, K, kprev, kchoice, ksample, khutch);
    MFM_LAUNCH_CHECK();
    // pull the current state back: its weight (:282-283)
    if (hutch && (rc = mfm_threefry_normal_batched(kprev, n, d, z, stream))) return rc;
    if ((rc = ode_solve(*f, *t, *o, -1, n, hutch ? z : nullptr, position, u_prev, vol_prev, stats, 0, S, B, zc, stream))) return rc;
    if ((rc = ref_logprob_rows(*f, n, u_prev, lq_prev, stream))) return rc;
    // K fresh reference samples per chain, pushed forward with their own probe keys (:284-287)
    if ((rc = mfm_threefry_normal_batched(ksample, M, d, gscr, stream))) return rc;
    if ((rc = ref_transform_rows(*f, M, gscr, refs, stream))) return rc;
    if (hutch && (rc = mfm_threefry_normal_batched(khutch, M, d, z, stream))) return rc;
    if ((rc = ode_solve(*f, *t, *o, +1, M, hutch ? z : nullptr, refs, samples, vols, stats, 1, S, B, zc, stream))) return rc;
    if ((rc = target_value_and_grad(*t, M, samples, ld, gscr, nullptr, wt, stream))) return rc;      // logprob_beta of the samples (:288)
    if ((rc = ref_logprob_rows(*f, M, refs, lq, stream))) return rc;
    CisArgs A{K, ld, lq, vols, lq_prev, vol_prev, samples, kchoice, wbuf, position, logdensity, acceptance_rate, proposed_position, proposed_weight, is_accepted, rng_x64()};
    cis_select_kernel<<<ceil_div(n, 8), 256, 0, stream>>>(n, d, A);
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}

int mfm_ref_sample(const mfm_field_t* f, const uint32_t* keys, int n, float* out, mfm_stream_t stream) {
    if (!f) { mfm_set_last_error_msg("null descriptor"); return MFM_ERR_ARG; }
    int rc = ref_check(f, true);
    if (rc) return rc;
    if (n <= 0) return MFM_OK;
    if (!keys || !out || f->dim <= 0) { mfm_set_last_error_msg("null argument or dim <= 0 (mfm_ref_sample)"); return MFM_ERR_ARG; }
    // normal(keys[c], (d,)) into out, then mean + std * z (exactly IndepGaussian.sample_model) or the band solve in place
    if ((rc = mfm_threefry_normal_batched(keys, n, f->dim, out, stream))) return rc;
    return ref_transform_rows(*f, n, out, out, stream);
}

int mfm_ref_logprob(const mfm_field_t* f, int n, const float* x, float* out, mfm_stream_t stream) {
    if (!f) { mfm_set_last_error_msg("null descriptor"); return MFM_ERR_ARG; }
    int rc = ref_check(f, false);
    if (rc) return rc;
    if (n <= 0) return MFM_OK;
    if (!x || !out || f->dim <= 0) { mfm_set_last_error_msg("null argument or dim <= 0 (mfm_ref_logprob)"); return MFM_ERR_ARG; }
    return ref_logprob_rows(*f, n, x, out, stream);
}

}  // extern "C"
