// Internal (non-ABI) declarations shared between translation units.
#pragma once
#include "common.cuh"
#include "../../include/mfm_b200.h"

void mfm_set_last_error_msg(const char* msg);

namespace mfm {

// bump allocator over the caller's workspace (256-byte aligned slices)
struct Workspace {
    char* base; size_t size, off; bool ok;
    Workspace(void* p, size_t n) : base((char*)p), size(n), off(0), ok(true) {}
    template <class T> T* take(size_t count) {
        size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
        if (base == nullptr || off + bytes > size) { ok = false; off += bytes; return nullptr; }
        T* r = (T*)(base + off); off += bytes; return r;
    }
};
inline size_t ws_slice(size_t count, size_t elt) { return (count * elt + 255) & ~(size_t)255; }

int pines_n_tiles(int d);

// grad_out[n,d] = beta*(c - a e^x) - (x-mu) K^-1 ; prior_partial[n, pines_n_tiles] = per-tile
// sums of (x-mu).q  (logprior = -0.5*sum + log_norm).  n_rows_dev: optional active-row count.
int pines_grad_gemm(const mfm_target_t& T, int n, const float* X, long long ldx, float beta,
                    float* grad_out, long long ldg, float* prior_partial, const int* n_rows_dev,
                    cudaStream_t st, const float* x_amax = nullptr);
// out[n,d] = Z K^-1 (Hessian-vector product of the prior is -Z K^-1)
int pines_kinv_gemm(const mfm_target_t& T, int n, const float* Z, long long ldz, float* out, long long ldo,
                    const int* n_rows_dev, cudaStream_t st, float z_bound = 0.0f);

// value+grad of logprob_beta for any target; loglik_out optional; ws from target_ws_bytes
size_t target_ws_bytes(const mfm_target_t& T, int n);
int target_value_and_grad(const mfm_target_t& T, int n, const float* x, float* logp, float* grad,
                          float* loglik_out, Workspace& ws, cudaStream_t st);

// untempered grad logprob (+ optional Hessian-vector product with z / Hessian diagonal) for the
// vector field; for pines hv excludes the constant -zK^-1 part when zkinv is supplied.
// outputs: gc = clip(grad), hvc = 1[|grad|<clip] * (H z), hdc = 1[|grad|<clip] * diag(H)  (hvc/hdc optional)
int target_field_terms(const mfm_target_t& T, int n, const float* x, const float* z, const float* zkinv, float clip,
                       float* gc, float* hvc, float* hdc, const int* n_rows_dev, cudaStream_t st, const float* x_amax = nullptr,
                       float* scratch = nullptr, const float* x_split = nullptr);

// ---- vector field (flow.cu) -------------------------------------------------------------------
// Hidden widths of the eight dense layers (mfm_field_t::hidden_t / hidden_x / hidden_xt; an all-zero tail: every width is
// `hidden`).  Dense_0 2F->t0, Dense_1 t0->t1, Dense_2 d->x0, Dense_3 x0->x1, Dense_4 t1->d, Dense_5 (x1 + t1)->xt0 over
// cat = [s_x | s_t], Dense_6 xt0->xt1, Dense_7 xt1->d.  Negative entries of a malformed tail are read as 0 here (buffer sizes
// only): field_widths_check refuses the descriptor before anything runs.
struct FieldWidths {
    int t0, t1, x0, x1, xt0, xt1;
    bool equal;                                                   // all six == hidden (today's network)
    int cat() const { return x1 + t1; }                           // row stride of cat / dcat; s_t starts at column x1
    int tan() const { int m = x0 > x1 ? x0 : x1; m = m > xt0 ? m : xt0; return m > xt1 ? m : xt1; }   // tangents: x and joint branches
    int widest() const { const int m = tan(); return m > t0 ? (m > t1 ? m : t1) : (t0 > t1 ? t0 : t1); }
    int narrowest() const { int m = t0 < t1 ? t0 : t1; m = m < x0 ? m : x0; m = m < x1 ? m : x1; m = m < xt0 ? m : xt0; return m < xt1 ? m : xt1; }
    bool all16() const { return t0 % 16 == 0 && t1 % 16 == 0 && x0 % 16 == 0 && x1 % 16 == 0 && xt0 % 16 == 0 && xt1 % 16 == 0; }
};
inline FieldWidths field_widths(const mfm_field_t& F) {
    FieldWidths w;
    const int* v[3] = {F.hidden_t, F.hidden_x, F.hidden_xt};
    bool zero = true;
    for (int b = 0; b < 3; ++b) zero = zero && v[b][0] == 0 && v[b][1] == 0;
    auto g = [&](int b, int i) { return zero ? F.hidden : (v[b][i] > 0 ? v[b][i] : 0); };
    w.t0 = g(0, 0); w.t1 = g(0, 1); w.x0 = g(1, 0); w.x1 = g(1, 1); w.xt0 = g(2, 0); w.xt1 = g(2, 1);
    w.equal = w.t0 == F.hidden && w.t1 == F.hidden && w.x0 == F.hidden && w.x1 == F.hidden && w.xt0 == F.hidden && w.xt1 == F.hidden;
    return w;
}
// MFM_ERR_ARG (with a message) unless the width tail is all zero, or all positive with `hidden` the largest
inline int field_widths_check(const mfm_field_t* f) {
    const int* v[3] = {f->hidden_t, f->hidden_x, f->hidden_xt};
    int n_zero = 0, n_pos = 0, widest = 0;
    for (int b = 0; b < 3; ++b)
        for (int i = 0; i < 2; ++i) { n_zero += v[b][i] == 0; n_pos += v[b][i] > 0; widest = v[b][i] > widest ? v[b][i] : widest; }
    if (n_zero == 6) return 0;
    if (n_pos != 6) { mfm_set_last_error_msg("field.hidden_t / hidden_x / hidden_xt: all six widths must be > 0 (or all 0: every width is `hidden`)"); return MFM_ERR_ARG; }
    if (f->hidden != widest) { mfm_set_last_error_msg("field.hidden must equal the widest of hidden_t / hidden_x / hidden_xt"); return MFM_ERR_ARG; }
    return 0;
}
// Slots of the per-workspace pool of tensor maxima (FieldBufs::amax, 64 floats): max |value| of every tensor that is the A
// operand of a scaled-fp16 GEMM (gemm_tcgen05_h16.cuh), written by its producer with atomicMax.  Slots below AM_EVAL_END
// are zeroed at the start of every field evaluation; the others belong to the caller of field_eval (one ODE solve / one FM
// pass) and are zeroed there.  A stale (too large) maximum is safe: it only shifts the 18-octave window of full precision.
enum AmaxSlot {
    AM_H0 = 0, AM_ST, AM_H2, AM_SX, AM_H5, AM_H6, AM_TA0, AM_TB0, AM_TA1, AM_TB1, AM_FF, AM_EVAL_END = 16,
    AM_W = 16,           // max |parameter| of the flat MLP buffer (one scale for both weight mirrors)
    AM_X,                // the field's input x (FM batch x_t, ODE stage input)
    AM_DELTA, AM_DGT, AM_D6, AM_D5, AM_DCX, AM_DCT0, AM_DCT, AM_D2, AM_D0, AM_ZW2,
    AM_V,                // the field's output v (FM forward: bounds the loss gradient before it is written)
    AM_TGT,              // the FM regression targets x - x0
    AM_WNORM_COL = 32,   // [8] per dense layer: max over outputs of sum_in |W[in][out]|  (bounds the forward product)
    AM_WNORM_ROW = 40,   // [8] per dense layer: max over inputs of sum_out |W[in][out]|   (bounds the backward-data product)
    AM_BIAS = 48,        // [8] per dense layer: max |bias|
    AM_BOUND = 64,       // slot i + AM_BOUND: the BOUND the pre-split copy of tensor i was scaled with (EpiStdS::bound_out)
    AM_POOL = 128
};
struct FieldBufs {
    float *ff, *h0, *cat, *h2, *gt, *h5, *h6, *gc, *hx, *ta, *tb, *zw2, *zkinv, *divpart;
    float *tan_a, *tan_b;   // exact path [n*d, H]
    float* wt;              // transposed dense kernels: layer i at wt + F.w_off[i], stored [out][in] (K-major B operand)
    float *wx, *wxo;        // pre-split mirrors of wt / of the parameters themselves (null: layer sizes not multiples of 8)
    float* amax;            // AM_POOL floats: tensor maxima (AmaxSlot)
    // pre-split (split16, scaled fp16) copies written next to the fp32 tensors by their producers: the A operands of the
    // layers that consume them (null: the scaled-fp16 GEMM is off or the sizes are not multiples of 16)
    float *ff_s, *h0_s, *cat_s, *h2_s, *h5_s, *h6_s, *ta_s, *tb_s;
    // activation derivatives at the pre-activations of h0, h2, cat = [s_x | s_t], h5, h6 (activations other than relu, whose
    // derivative is read off the sign of the output): what the backward pass and the tangents multiply by
    float *dh0, *dh2, *dcat, *dh5, *dh6;
    float* tscratch;        // 4 x [n, d]: the whitened pines target's field terms (four GEMMs against the Cholesky factor)
    float* v_amax = nullptr;   // optional slot receiving max |v| of the next field evaluation (set by the FM pass)
};
namespace tc2p {
void register_cross(const float* base, size_t n_floats, const float* mirror);
void clear_cross();
}
namespace tc2h {
int gemm_h16();
void register_mirror_h16(const float* base, size_t n_floats, const float* mirror, const float* amax);
void clear_mirrors_h16();
cudaError_t launch_absmax(const float* x, long long ld, int rows, int cols, const int* n_rows_dev, float* out, cudaStream_t st);
float* amax_scratch_for(cudaStream_t st);
int split_groups();
int h16_min_hidden();
}
int gemm_backend();
int rng_x64();             // 1: float64-layout draws (jax_enable_x64), rounded to float32 (rng.cu)
// dst mirrors src.  h16 kernel (default): groups of 16 floats -> 16 hi | 16 lo fp16 parts of the values scaled by
// h16_scale(*amax); tf32 + bf16-cross kernel: groups of 8 floats -> 8 bf16 of the values | 8 bf16 of their tf32 truncation rests
int presplit_weights(const float* src, float* dst, long long n_floats, const float* amax, cudaStream_t st);
// clears the mirror registries when an ABI call that registered mirrors returns
struct CrossScope { ~CrossScope() { tc2p::clear_cross(); tc2h::clear_mirrors_h16(); } };
// magnitudes of a dense layer's operands / result for the scaled-fp16 GEMM (all optional)
struct DenseAmax {
    const float* a = nullptr; const float* a2 = nullptr; float a_bound = 0.0f;    // exact max |A| (device slots) or a host-known bound
    float* out = nullptr;                                                          // receives the exact max |C|
    const float* a_split = nullptr; const float* a_scale_src = nullptr;            // pre-split copy of A and the slot its scale came from
    float* out_split = nullptr; float* out_bound = nullptr;                        // write C pre-split too; slot receiving its bound
    const float* w_norm = nullptr; const float* bias_amax = nullptr; const float* add_bound = nullptr;   // ingredients of that bound
    const float* alt_amax = nullptr; const float* alt_w_norm = nullptr; const float* alt_bias = nullptr; // a sibling layer sharing C's scale
    float* dact = nullptr; long long lddact = 0;    // receives act'(pre-activation) (activations other than relu)
    int mask_mul = 0;                               // the mask operand holds derivatives: multiply instead of the > 0 gate
};
size_t field_bufs_bytes(const mfm_field_t& F, const mfm_target_t& T, int n, bool hutch);
bool field_bufs_take(FieldBufs& B, Workspace& w, const mfm_field_t& F, int n, bool hutch, const mfm_target_t* T = nullptr);
// B.wt <- transposes of the eight dense kernels (once per ABI call: the parameters may have changed)
int field_prepare_weights(const mfm_field_t& F, FieldBufs& B, cudaStream_t st);
void field_register_mirrors(const mfm_field_t& F, const FieldBufs& B);
// C[n,out] = act(A[n,in] W[in,out] + bias) gated by mask (relu' of another activation); `relu` = activation code of gemm_tf32x3.cuh
// (0 none, 1 relu, 2 tanh, 3 elu, 4 gelu, 5 swish).
// WT = the kernel transposed, WT[o*ldwt + i]: both GEMM operands are K-major, which is what the
// persistent tcgen05 kernel's bf16 cross-term path needs.
int dense(int n, int in, int out, const float* A, long long lda, const float* WT, long long ldwt, const float* bias, int relu,
          float* C, long long ldc, const float* mask, long long ldm, int mask_div, cudaStream_t st,
          const int* n_rows_dev = nullptr, DenseAmax am = DenseAmax());
// out_v = sgn * v(x, t); out_l = -sgn * div v (optional; z != null -> Hutchinson, else exact trace).
// Leaves the activations (ff, h0, cat=[s_x|s_t], h2, gt, h5, h6, gc) in B for a backward pass.
// n_rows_dev (optional): device count of leading rows that are live (compacted active chains);
// row_map (optional): compact row -> chain index used when writing out_v / out_l.
// x_amax (optional): device slot with max |x| (null: one reduction pass inside the first GEMM that reads x).
int field_eval(const mfm_field_t& F, const mfm_target_t& T, int n, const float* x, const float* tfield,
               const float* z, float sgn, float* out_v, float* out_l, FieldBufs& B, cudaStream_t st,
               const int* n_rows_dev = nullptr, const int* row_map = nullptr, const float* x_amax = nullptr,
               const float* x_split = nullptr);    // x_split: split16 copy of x scaled from *x_amax (the FM batch's), or null

}  // namespace mfm
