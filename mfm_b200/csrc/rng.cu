// jax.random-compatible generators (threefry2x32, legacy uint32[2] keys, x64 off).
// Replaces the XLA threefry2x32 / erf_inv HLO behind every jax.random.* call on the hot path
// (bblackjax/util.py:81, proposal.py:179, exe_flow_matching.py:142-166,212,265-275,303).
#include "common.cuh"
#include "../../include/mfm_b200.h"
#include <stdio.h>
#include <string.h>

static thread_local char g_err[512] = "";
void mfm_set_last_error(cudaError_t e, const char* file, int line) {
    snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) at %s:%d", (int)e, cudaGetErrorString(e), file, line);
}
void mfm_set_last_error_msg(const char* msg) { snprintf(g_err, sizeof(g_err), "%s", msg); }
extern "C" const char* mfm_last_error(void) { return g_err; }
extern "C" int mfm_version(void) { return 101; }   // 101: mfm_field_t grew (ref_kind, ref_log_norm, ref_band)
unsigned long long g_mfm_launches = 0;
#include <stdlib.h>
namespace mfm {
// 1: every uniform / normal draw of the library follows jax's float64 layout (jax_enable_x64, as the reference ships:
// multi_modal.py:14) and is rounded to float32 once; 0 (default): float32 draws.  MFM_RNG_X64=1 / mfm_set_rng_x64.
static int g_rng_x64 = -1;
int rng_x64() {
    if (g_rng_x64 < 0) { const char* e = getenv("MFM_RNG_X64"); g_rng_x64 = (e && e[0] == '1') ? 1 : 0; }
    return g_rng_x64;
}
}
extern "C" void mfm_set_rng_x64(int v) { mfm::g_rng_x64 = v ? 1 : 0; }
extern "C" int mfm_rng_x64_enabled(void) { return mfm::rng_x64(); }
extern "C" unsigned long long mfm_launch_count(void) { return g_mfm_launches; }

namespace {

__global__ void split_kernel(const uint32_t* __restrict__ keys, int n, int num, uint32_t* __restrict__ out) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= (long long)n * num) return;
    const int c = (int)(i / num), j = (int)(i % num);
    const u32x2 k = threefry_split_key(keys[2 * c], keys[2 * c + 1], (uint32_t)j, (uint32_t)num);
    out[2 * i] = k.a; out[2 * i + 1] = k.b;
}

// MODE 0 bits, 1 uniform, 2 normal.  One thread per threefry block -> two stream words (float32 draws); with x64 draws every
// element is one block of its own, (e, n + e), and the thread produces its two elements from two blocks.
template <int MODE>
__global__ void stream_kernel(const uint32_t* __restrict__ keys, int nkeys, long long n, double minval_d, double maxval_d,
                              void* __restrict__ out, int x64) {
    const float minval = (float)minval_d, maxval = (float)maxval_d;      // float32 draws: the bounds are float32 values, as in jax
    const long long half = (n + 1) >> 1;
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= half * nkeys) return;
    const int c = (int)(i / half);
    const long long lo = i % half;
    long long hi = lo + half;
    const bool has_hi = hi < n;
    const long long base = (long long)c * n;
    const uint32_t k0 = keys[2 * c], k1 = keys[2 * c + 1];
    if (MODE != 0 && x64) {
        float* p = (float*)out;
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            if (s == 1 && !has_hi) break;
            const long long e = s == 0 ? lo : hi;
            const u32x2 o = threefry2x32(k0, k1, (uint32_t)e, (uint32_t)(n + e));
            if (MODE == 1) {
                const double mn = minval_d, sc = maxval_d - minval_d;
                p[base + e] = (float)fmax(mn, __dadd_rn(__dmul_rn(bits64_to_unit_double(o.a, o.b), sc), mn));
            } else p[base + e] = bits64_to_normal(o.a, o.b);
        }
        return;
    }
    const u32x2 o = threefry2x32(k0, k1, (uint32_t)lo, has_hi ? (uint32_t)hi : 0u);
    if (MODE == 0) {
        uint32_t* p = (uint32_t*)out;
        p[base + lo] = o.a; if (has_hi) p[base + hi] = o.b;
    } else if (MODE == 1) {
        float* p = (float*)out;
        const float sc = maxval - minval;
        p[base + lo] = fmaxf(minval, __fadd_rn(__fmul_rn(bits_to_unit_float(o.a), sc), minval));  // no FMA: mul then add as XLA
        if (has_hi) p[base + hi] = fmaxf(minval, __fadd_rn(__fmul_rn(bits_to_unit_float(o.b), sc), minval));
    } else {
        float* p = (float*)out;
        p[base + lo] = bits_to_normal(o.a);
        if (has_hi) p[base + hi] = bits_to_normal(o.b);
    }
}

template <int MODE>
int launch_stream(const uint32_t* keys, int nkeys, long long n, double lo, double hi, void* out, cudaStream_t st) {
    if (n <= 0 || nkeys <= 0) return MFM_OK;
    if (n > 0xFFFFFFFFll || (mfm::rng_x64() && 2 * n > 0xFFFFFFFFll)) return MFM_ERR_UNSUPPORTED;
    const long long work = ((n + 1) >> 1) * nkeys;
    stream_kernel<MODE><<<ceil_div(work, 256), 256, 0, st>>>(keys, nkeys, n, lo, hi, out, mfm::rng_x64());
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}

}  // namespace

extern "C" {

int mfm_threefry_split(const uint32_t* key, int num, uint32_t* out, mfm_stream_t stream) {
    return mfm_threefry_split_batched(key, 1, num, out, stream);
}

int mfm_threefry_split_batched(const uint32_t* keys, int n, int num, uint32_t* out, mfm_stream_t stream) {
    if (n <= 0 || num <= 0) return MFM_OK;
    split_kernel<<<ceil_div((long long)n * num, 256), 256, 0, stream>>>(keys, n, num, out);
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}

int mfm_threefry_bits(const uint32_t* key, long long n, uint32_t* out, mfm_stream_t stream) {
    return launch_stream<0>(key, 1, n, 0.0, 1.0, out, stream);
}
int mfm_threefry_uniform(const uint32_t* key, long long n, double minval, double maxval, float* out, mfm_stream_t stream) {
    return launch_stream<1>(key, 1, n, minval, maxval, out, stream);
}
int mfm_threefry_normal(const uint32_t* key, long long n, float* out, mfm_stream_t stream) {
    return launch_stream<2>(key, 1, n, 0.0, 1.0, out, stream);
}
int mfm_threefry_uniform_batched(const uint32_t* keys, int n, int d, double minval, double maxval, float* out, mfm_stream_t stream) {
    return launch_stream<1>(keys, n, d, minval, maxval, out, stream);
}
int mfm_threefry_normal_batched(const uint32_t* keys, int n, int d, float* out, mfm_stream_t stream) {
    return launch_stream<2>(keys, n, d, 0.0, 1.0, out, stream);
}

void mfm_host_threefry_split(const uint32_t key[2], int num, uint32_t* out) {
    for (int j = 0; j < num; ++j) {
        const u32x2 k = threefry_split_key(key[0], key[1], (uint32_t)j, (uint32_t)num);
        out[2 * j] = k.a; out[2 * j + 1] = k.b;
    }
}

}  // extern "C"

// Test hook (not in the ABI header): bits_to_normal_t (table-driven correctly rounded log) against bits_to_normal (generic double
// log) on the inputs start, start + stride, ...: counts bit-level mismatches and how often the Ziv test sent the fast path to the
// generic one (out[0], out[1]).
__global__ void normal_fast_check_kernel(unsigned long long n, uint32_t start, uint32_t stride, unsigned long long* out) {
    __shared__ double2 ltab[16];
    log_tab_load(ltab);
    unsigned long long bad = 0;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t bits = start + (uint32_t)i * stride;
        const float a = bits_to_normal_t(bits, ltab), b = bits_to_normal(bits);
        bad += __float_as_uint(a) != __float_as_uint(b);
    }
    if (bad) atomicAdd(out, bad);
}
extern "C" int mfm_debug_normal_fast_check(unsigned long long n, uint32_t start, uint32_t stride, unsigned long long* out, mfm_stream_t stream) {
    MFM_CUDA_CHECK(cudaMemsetAsync(out, 0, 2 * sizeof(unsigned long long), stream));
    normal_fast_check_kernel<<<148 * 8, 256, 0, stream>>>(n, start, stride, out);
    MFM_LAUNCH_CHECK();
    return MFM_OK;
}
