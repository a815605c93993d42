// Reference distribution PhiFourBase (mfm_field_t::ref_kind == MFM_REF_PHI4_BASE, distributions.py:168-226): the band solve
// x = L^-T z that turns a standard normal row into a sample, shared by the FM batch kernel (fm.cu) and the row kernels (flow.cu).
//
// L is lower bidiagonal (diagonal l, sub-diagonal s), so L^T x = z is the first-order recurrence
//   x_{d-1} = z_{d-1} / l_{d-1},   x_i = a_i x_{i+1} + b_i  with  a_i = -s_{i+1} / l_i,  b_i = z_i / l_i  (a_{d-1} = 0).
// One warp solves one row staged in shared memory: lane k owns the contiguous chunk [k m, (k+1) m) of the row (m = ceil(d/32),
// stored at pitch m | 1 so that the lanes' strided accesses hit distinct banks), composes its chunk's affine maps, a 5-step
// suffix scan of the 32 composed maps gives the value entering every chunk, and each lane reruns its chunk from that value.
// |a_i| < 1/2 for every alpha, beta, so both passes are contractions: float32 error stays at a few ulps of the row maximum.
#pragma once
#include "internal.h"

namespace mfm {

// floats of shared memory one warp stages a row of length d in
__host__ __device__ __forceinline__ int band_pitch(int d) { return ((d + 31) >> 5) | 1; }
__host__ __device__ __forceinline__ int band_row_floats(int d) { return 32 * band_pitch(d); }
// position of row element j in the staged layout (chunk k = j / m via a float reciprocal: exact for j <= 2^20, since the
// fractional part of (j + 1/2) / m stays >= 1/(2m) away from an integer)
__device__ __forceinline__ int band_slot(int j, int m, int mp, float inv_m) {
    const int k = (int)(((float)j + 0.5f) * inv_m);
    return k * mp + (j - k * m);
}

// In place on the staged row r: z -> x = L^-T z.  band = a[d], rl[d] (mfm_field_t::ref_band: a_i = -s_{i+1} / l_i, rl_i = 1 / l_i,
// formed in float64 on the host).  All 32 lanes must call.
__device__ __forceinline__ void band_solve_warp(float* r, int d, const float* __restrict__ band, int lane) {
    const int m = (d + 31) >> 5, mp = m | 1;
    const float* a = band;
    const float* rl = band + d;
    const int lo = lane * m, hi = min(lo + m, d);
    float* row = r + lane * mp - lo;                       // row[i] for i in [lo, hi)
    __syncwarp();
    // pass 1: b_i into the row, and the chunk's map y -> A y + B from the value entering it (x_hi) to x_lo
    float A = 1.0f, B = 0.0f;
    for (int i = hi - 1; i >= lo; --i) {
        const float ai = __ldg(a + i);
        const float b = row[i] * __ldg(rl + i);
        row[i] = b;
        B = fmaf(ai, B, b);
        A = ai * A;
    }
    // suffix composition over the lanes: (A, B) <- (A, B) o (A', B') of lane + off; then B = x at the start of this chunk
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const float A2 = __shfl_down_sync(0xffffffffu, A, off), B2 = __shfl_down_sync(0xffffffffu, B, off);
        if (lane + off < 32) { B = fmaf(A, B2, B); A = A * A2; }
    }
    float x = __shfl_down_sync(0xffffffffu, B, 1);
    if (lane == 31) x = 0.0f;                              // x_d = 0 (and a_{d-1} = 0)
    // pass 2: the chunk from the value entering it
    for (int i = hi - 1; i >= lo; --i) {
        x = fmaf(__ldg(a + i), x, row[i]);
        row[i] = x;
    }
    __syncwarp();
}

// Validation of the reference-distribution fields shared by every entry point that reads them.  needs_band: the call runs a
// band kernel (the shared-memory row limit applies).
inline int ref_check(const mfm_field_t* f, bool needs_band) {
    if (f->ref_kind == MFM_REF_INDEP_GAUSS) {
        if (!(f->ref_std > 0.0f)) { mfm_set_last_error_msg("field.ref_std must be > 0 (reference distribution IndepGaussian(mean, std^2))"); return MFM_ERR_ARG; }
        return MFM_OK;
    }
    if (f->ref_kind == MFM_REF_PHI4_BASE) {
        if (!f->ref_band) { mfm_set_last_error_msg("field.ref_band must point to the band factor of PhiFourBase (ref_kind 1)"); return MFM_ERR_ARG; }
        if (!isfinite(f->ref_log_norm)) { mfm_set_last_error_msg("field.ref_log_norm must be finite (ref_kind 1)"); return MFM_ERR_ARG; }
        if (needs_band && (f->dim < 1 || f->dim > MFM_REF_BAND_MAX_DIM)) {
            mfm_set_last_error_msg("PhiFourBase reference distribution: dim must be <= MFM_REF_BAND_MAX_DIM (12192)"); return MFM_ERR_UNSUPPORTED;
        }
        return MFM_OK;
    }
    mfm_set_last_error_msg("unknown reference distribution (mfm_field_t::ref_kind)");
    return MFM_ERR_ARG;
}

// warps per block of a kernel staging one row per warp: as many as fit 48 KB of shared memory, at most 8
inline int band_warps_per_block(int d) {
    const int per_warp = band_row_floats(d) * (int)sizeof(float);
    const int w = (48 * 1024 - 256) / per_warp;            // (256 bytes: fm_batch_phi4_kernel's static log table)
    return w < 1 ? 1 : (w > 8 ? 8 : w);
}

}  // namespace mfm
