// msda_api.cu -- the extern "C" boundary declared in include/msda_b200.h.
//
// Host-side counterpart of the reference's ms_deform_attn_cuda_forward/backward
// (ms_deform_attn_cuda.cu:25-85, 88-158): argument validation and kernel choice.
// Tensor-level checks (contiguity, device, dtype, im2col_step divisibility) live in
// the Python shim because they need tensor metadata; this layer sees raw pointers.
//
// The plain and the fused-producer MSDA entries differ only in the Producers they hand to the
// launchers (reference points == nullptr: plain), so each backward has one body for both:
// backward() (kernel choice and "bwd_variant") and backward_deterministic().  The fp32 and the mixed-precision
// (bf16 / fp16 value) entries share the same bodies, templates over the value type.  Entries that
// come as a default and a deterministic / training twin forward to one static body each.
#include <atomic>
#include <cstdint>
#include <cstring>

#include "../../include/msda_b200.h"
#include "msda_common.cuh"

namespace msda {

// implemented in the kernel translation units.  V: element type of value / output / grad_output (float, or
// __nv_bfloat16 / __half for the mixed-precision entries); T: of the locations, weights and sums; P: of the
// 32-channel kernels' locations / weights or raw offsets / logits and their gradients (float, or V for the
// mixed-precision fused entries)
template <typename V, typename P>
cudaError_t launch_fwd_d32(const V *, const int64_t *, const int64_t *, const P *, const P *,
                           const Producers &, const Dims &, V *, cudaStream_t, bool *handled);
template <typename V, typename P>
cudaError_t launch_bwd_d32(const V *, const V *, const int64_t *, const int64_t *, const P *,
                           const P *, const Producers &, const Dims &, float *, P *, P *,
                           const DetRecords *, int gate, cudaStream_t, bool *handled);
template <typename V, typename P>
cudaError_t launch_bwd_sorted(const V *, const V *, const int64_t *, const int64_t *, const P *,
                              const P *, const Producers &, const Dims &, float *, P *, P *, int gate,
                              cudaStream_t, bool *handled);
template <typename V>
bool bwd_sorted_applies(const V *value, const float *grad_value, const Dims &);
template <typename V, typename T>
cudaError_t launch_bwd_generic_records(const V *, const V *, const int64_t *, const int64_t *, const T *, const T *,
                                       const Dims &, T *, T *, const DetRecords &, cudaStream_t);
template <typename V, typename T>
cudaError_t launch_fwd_generic(const V *, const int64_t *, const int64_t *, const T *, const T *,
                               const Dims &, V *, cudaStream_t);
template <typename V, typename T>
cudaError_t launch_bwd_generic(const V *, const V *, const int64_t *, const int64_t *, const T *,
                               const T *, const Dims &, T *, T *, T *, cudaStream_t);
template <typename V>
cudaError_t launch_narrow(const float *, V *, long long, cudaStream_t);
cudaError_t launch_linear_tf32x3(const float *, const float *, const float *, float *, int, int, int, int,
                                 float *, cudaStream_t, bool *handled, bool deterministic);
cudaError_t launch_split_weight(const float *, float *, int, int, cudaStream_t, bool *handled);
cudaError_t launch_add_layernorm(const float *, const float *, const float *, const float *, float *, long long,
                                 int, float, cudaStream_t, bool *handled);
cudaError_t launch_add_layernorm_bwd(const float *, const float *, const float *, const float *, float *, float *,
                                     float *, long long, int, float, cudaStream_t, bool *handled, float *partials);
long long add_layernorm_bwd_partials(long long rows, int cols);
template <typename R>
cudaError_t launch_add_layernorm_mixed(const float *, const R *, const float *, const float *, float *, R *, long long,
                                       int, float, cudaStream_t, bool *handled);
template <typename R>
cudaError_t launch_add_layernorm_mixed_bwd(const float *, const R *, const float *, const R *, const float *, float *,
                                           R *, float *, float *, long long, int, float, cudaStream_t, bool *handled,
                                           float *partials);
cudaError_t launch_linear_wgrad(const float *, const float *, float *, float *, long long, int, int, cudaStream_t,
                                bool *handled, float *partials);
long long linear_wgrad_partials(long long rows, int out_f, int in_f);
cudaError_t launch_transpose(const float *, float *, long long, int, cudaStream_t);
// 16-bit Linear (linear_mixed.cu): T = __nv_bfloat16 or __half
template <typename T>
cudaError_t launch_linear_mixed(const T *, const T *, const float *, T *, int, int, int, int, cudaStream_t,
                                bool *handled);
template <typename T>
cudaError_t launch_linear_mixed_wgrad(const T *, const T *, float *, float *, long long, int, int, float *,
                                      cudaStream_t, bool *handled);
long long linear_mixed_wgrad_workspace_floats(long long rows, int out_f, int in_f);
// GroupNorm: V = type of the map x (and of y16 / grad_x), float or 16-bit; G = type of grad_y (float or V)
template <typename V>
cudaError_t launch_group_norm(const V *, const float *, const float *, const float *, float *, V *y16, int, int, int,
                              int, int, float, int, const float *, int, int, double *, float *mean_rstd, cudaStream_t,
                              bool *handled);
template <typename V>
cudaError_t launch_channel_bias(V *, const float *, int, int, long long, cudaStream_t, bool *handled);
template <typename V>
cudaError_t launch_group_norm_rows(const V *, const float *, const float *, const float *, float *, int, int,
                                   long long, int, float, int, long long, long long, double *, float *mean_rstd,
                                   cudaStream_t, bool *handled);
int group_norm_workspace_doubles(int N, int groups);
template <typename G, typename V>
cudaError_t launch_group_norm_bwd(const G *, const V *, const float *, const float *, const float *, const float *,
                                  V *, float *, float *, float *, float *, int, int, int, int, int, int, int, int,
                                  double *, cudaStream_t, bool *handled);
template <typename V>
cudaError_t launch_group_norm_rows_bwd(const float *, long long, long long, const V *, const float *, const float *,
                                       const float *, const float *, V *, float *, float *, float *, int, int,
                                       long long, int, int, double *, cudaStream_t, bool *handled);
long long group_norm_bwd_workspace_doubles(int N, int C);
cudaError_t launch_debug_indices(const int64_t *, const int64_t *, const float *, const Dims &,
                                 int32_t *, int64_t *, cudaStream_t);

static std::atomic<long long> g_launches{0};
static std::atomic<int> g_options[OPT_COUNT];   // zero-initialised: 0 == auto

void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
int option_value(int which) { return g_options[which].load(std::memory_order_relaxed); }

int sm_count() {
    static std::atomic<int> cached[kMaxDevices];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 148;   // launches refuse such a device
    int v = cached[dev].load(std::memory_order_relaxed);
    if (v == 0) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0)
            v = 148;
        cached[dev].store(v, std::memory_order_relaxed);
    }
    return v;
}

// ref_bstride: the fused entries' reference-point batch stride, 0 (shared by the batch) or Lq*L*2
static int check_dims(const Dims &d, long long ref_bstride = 0) {
    if (d.N <= 0 || d.S <= 0 || d.M <= 0 || d.D <= 0 || d.L <= 0 || d.Lq <= 0 || d.P <= 0)
        return MSDA_ERR_BAD_SHAPE;
    if (d.L > MSDA_MAX_LEVELS) return MSDA_ERR_UNSUPPORTED;
    if (ref_bstride != 0 && ref_bstride != (long long)d.Lq * d.L * 2) return MSDA_ERR_BAD_SHAPE;
    return MSDA_OK;
}

// the 32-channel kernels use 128-bit accesses on value / output rows and 64-bit ones on the
// locations; a contiguous tensor view with an odd storage offset goes to the generic kernels,
// which accept any alignment like the reference's scalar kernels do
static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static bool aligned8(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }
// the 32-channel kernels read and write an (x, y) pair of locations / offsets at once: 8 bytes in fp32, 4 in 16-bit
template <typename P>
static bool pair_aligned(const P *p) { return (reinterpret_cast<uintptr_t>(p) & (2 * sizeof(P) - 1)) == 0; }

// the return code of a launcher that reports through `handled` whether it covers the problem
static int launch_rc(cudaError_t e, bool handled) {
    return e == cudaSuccess && !handled ? MSDA_ERR_UNSUPPORTED : (int)e;
}

static int option_index(const char *name) {
    if (!name) return -1;
    if (!strcmp(name, "fwd_variant")) return OPT_FWD_VARIANT;
    if (!strcmp(name, "bwd_variant")) return OPT_BWD_VARIANT;
    if (!strcmp(name, "tile_order")) return OPT_TILE_ORDER;
    if (!strcmp(name, "ctas_per_sm")) return OPT_CTAS_PER_SM;
    if (!strcmp(name, "linear_variant")) return OPT_LINEAR_VARIANT;
    if (!strcmp(name, "wgrad_chunk")) return OPT_WGRAD_CHUNK;
#ifdef MSDA_PROFILE_KNOBS      // `make profile`: knobs that skip work on purpose (WRONG results), timing experiments only
    if (!strcmp(name, "whatif_drop_reds")) return OPT_WHATIF_DROP_REDS;
    if (!strcmp(name, "whatif_linear")) return OPT_WHATIF_LINEAR;
#endif
    return -1;
}

// The forward of fp32 (V = float) and of the mixed-precision op (16-bit V, fp32 locations and weights): the
// 32-channel kernel where it applies, the generic one otherwise.  With pr.ref set, the mixed-precision fused
// producers (P = V: raw 16-bit offsets / logits, packed rows): the 32-channel kernel or MSDA_ERR_UNSUPPORTED.
template <typename V, typename P = float>
static int forward(const V *value, const int64_t *shapes, const int64_t *lstart, const P *loc,
                   const P *attw, const Producers &pr, const Dims &d, V *output, cudaStream_t st) {
    if (!value || !shapes || !lstart || !loc || !attw || !output) return MSDA_ERR_NULL_POINTER;
    if (int rc = check_dims(d, pr.ref_bstride)) return rc;
    const bool fused = pr.ref != nullptr;
    bool handled = false;
    cudaError_t e = cudaSuccess;
    const bool fast_ok = aligned16(value) && aligned16(output) && pair_aligned(loc) && aligned8(pr.ref);
    if ((fused || option_value(OPT_FWD_VARIANT) != 63) && fast_ok)   // 63 forces the generic kernel (tests)
        e = launch_fwd_d32<V, P>(value, shapes, lstart, loc, attw, pr, d, output, st, &handled);
    if (e != cudaSuccess || handled || fused) return launch_rc(e, handled);
    if constexpr (std::is_same<P, float>::value)
        e = launch_fwd_generic<V, float>(value, shapes, lstart, loc, attw, d, output, st);
    return (int)e;
}

// The backward of fp32 (V = float) and of the mixed-precision op (16-bit V: `gv` is the caller's zero-filled fp32
// accumulation buffer, rounded into the 16-bit grad_value by the entry afterwards), plain (pr.ref == nullptr: `loc`
// / `attw` are the sampling locations and attention weights) or fused, fp32 only (`loc` / `attw` are the raw
// sampling offsets and attention logits, and the gradients are taken with respect to them; P = V for the 16-bit
// ones of the mixed-precision fused entries, float otherwise).  Where no 32-channel
// kernel covers the problem (shape, or a view that is not aligned) the plain op takes the generic kernel and the
// fused one returns MSDA_ERR_UNSUPPORTED.  "bwd_variant":
//   0 (default): where the queries are the value pixels (encoder self-attention) the in-SM merging kernel (points
//       near their query) and the per-row reduction kernel (points anywhere) are both launched; every CTA of both
//       runs the same probe of the sampling locations first and the kernel the verdict goes against returns at
//       once (msda_common.cuh);
//   20..39: merging kernel forced (plain: and its tuning variants); 1..8: CTA shapes of the plain per-row kernel;
//   63: generic kernel (plain only, tests).  16-bit V takes the same meanings, each kernel in its default shape.
template <typename V, typename P = float>
static int backward(const V *grad_output, const V *value, const int64_t *shapes, const int64_t *lstart,
                    const P *loc, const P *attw, const Producers &pr, const Dims &d, float *gv,
                    P *gl, P *gw, cudaStream_t st) {
    if (!grad_output || !value || !shapes || !lstart || !loc || !attw || !gv || !gl || !gw)
        return MSDA_ERR_NULL_POINTER;
    if (int rc = check_dims(d, pr.ref_bstride)) return rc;
    const bool fused = pr.ref != nullptr;
    const int variant = option_value(OPT_BWD_VARIANT);
    const bool aligned = aligned16(value) && aligned16(grad_output) && aligned16(gv) && pair_aligned(loc) &&
                         pair_aligned(gl) && aligned8(pr.ref);
    bool handled = false;
    cudaError_t e = cudaSuccess;
    if (aligned && (fused || variant != 63)) {
        int gate = GATE_NONE;
        if ((variant == 0 || (variant >= 20 && variant < 40)) && bwd_sorted_applies<V>(value, gv, d)) {
            e = launch_bwd_sorted<V, P>(grad_output, value, shapes, lstart, loc, attw, pr, d, gv, gl, gw,
                                  variant == 0 ? GATE_RUN_IF_LOCAL : GATE_NONE, st, &handled);
            if (variant == 0) {                  // the per-row kernel follows, gated the other way
                handled = false;
                gate = GATE_RUN_IF_SPREAD;
            }
        }
        if (e == cudaSuccess && !handled)
            e = launch_bwd_d32<V, P>(grad_output, value, shapes, lstart, loc, attw, pr, d, gv, gl, gw, nullptr, gate,
                                     st, &handled);
    }
    if (e != cudaSuccess || handled || fused) return launch_rc(e, handled);
    if constexpr (std::is_same<P, float>::value)
        e = launch_bwd_generic<V, float>(grad_output, value, shapes, lstart, loc, attw, d, gv, gl, gw, st);
    return (int)e;
}

// The mixed-precision backward, plain or fused: backward() into the fp32 accumulation buffer `acc`, then the
// conversion into the 16-bit grad_value
template <typename V, typename P = float>
static int backward_mixed(const V *grad_output, const V *value, const int64_t *shapes, const int64_t *lstart,
                          const P *loc, const P *attw, const Producers &pr, const Dims &d, float *acc, V *gv, P *gl,
                          P *gw, cudaStream_t st) {
    if (!gv) return MSDA_ERR_NULL_POINTER;
    const int rc = backward<V, P>(grad_output, value, shapes, lstart, loc, attw, pr, d, acc, gl, gw, st);
    if (rc != MSDA_OK) return rc;
    return (int)launch_narrow<V>(acc, gv, (long long)d.N * d.S * d.M * d.D, st);
}

// Deterministic backward (msda_det.cu), plain or fused as in backward() (fp64: plain only): the records kernel of the
// path, then sort, bounds and gather into grad_value.  V: element type of value / grad_output / grad_value, T: of the
// records and sums (16-bit V: float; the gather writes the 16-bit grad_value directly, no accumulation buffer),
// P: of the locations and weights or raw offsets and logits and their gradients (T, or V for the 16-bit fused
// producers).
template <typename V, typename T, typename P = T>
static int backward_deterministic(const V *grad_output, const V *value, const int64_t *shapes, const int64_t *lstart,
                                  const P *loc, const P *attw, const Producers &pr, const Dims &d, V *gv, P *gl,
                                  P *gw, void *workspace, cudaStream_t st) {
    if (!grad_output || !value || !shapes || !lstart || !loc || !attw || !gv || !gl || !gw || !workspace)
        return MSDA_ERR_NULL_POINTER;
    if (int rc = check_dims(d, pr.ref_bstride)) return rc;
    DetLayout l;
    if (!det_layout(d, (int)sizeof(T), &l)) return MSDA_ERR_BAD_SHAPE;
    if (!aligned16(workspace)) return MSDA_ERR_UNSUPPORTED;
    const DetRecords rec = det_records(workspace, l);
    bool handled = false;
    cudaError_t e = cudaSuccess;
    if constexpr (std::is_same<T, float>::value) {
        const bool aligned = aligned16(value) && aligned16(grad_output) && pair_aligned(loc) && pair_aligned(gl) &&
                             aligned8(pr.ref);
        if (aligned && (pr.ref != nullptr || option_value(OPT_BWD_VARIANT) != 63))
            e = launch_bwd_d32<V, P>(grad_output, value, shapes, lstart, loc, attw, pr, d, nullptr, gl, gw, &rec,
                                     GATE_NONE, st, &handled);
    }
    if (e == cudaSuccess && !handled) {
        if (pr.ref != nullptr) return MSDA_ERR_UNSUPPORTED;
        if constexpr (std::is_same<P, T>::value)
            e = launch_bwd_generic_records<V, T>(grad_output, value, shapes, lstart, loc, attw, d, gl, gw, rec, st);
    }
    if (e == cudaSuccess) e = launch_det_reduce<V, T>(l, workspace, grad_output, gv, d, st);
    return (int)e;
}

// The fused forward with row strides and per-query tables: fp32 (V = float), or 16-bit V with 16-bit raw offsets /
// logits (P = V) and fp32 tables.  Strides in elements of P.
template <typename V>
static int fused_forward_strided(const V *value, const int64_t *shapes, const int64_t *lstart, const float *ref,
                                 long long ref_bstride, const V *offsets, int offsets_stride, const V *logits,
                                 int logits_stride, const float *offsets_table, const float *logits_table,
                                 const Dims &d, V *output, cudaStream_t st) {
    if (!value || !shapes || !lstart || !ref || !offsets || !logits || !output) return MSDA_ERR_NULL_POINTER;
    if (int rc = check_dims(d, ref_bstride)) return rc;
    const long long packed = (long long)d.M * d.L * d.P;
    if (offsets_stride < 2 * packed || logits_stride < packed || (offsets_stride & 1)) return MSDA_ERR_BAD_SHAPE;
    if ((offsets_table != nullptr) != (logits_table != nullptr)) return MSDA_ERR_NULL_POINTER;
    if (!aligned16(value) || !aligned16(output) || !pair_aligned(offsets) || !aligned8(ref) || !aligned8(offsets_table))
        return MSDA_ERR_UNSUPPORTED;
    // the kernel reads packed rows (row strides 2*M*L*P and M*L*P) as stride 0
    const bool rows_packed = offsets_stride == 2 * packed && logits_stride == packed;
    const Producers pr{ref, ref_bstride, rows_packed ? 0 : offsets_stride, rows_packed ? 0 : logits_stride,
                       offsets_table, logits_table};
    bool handled = false;
    const cudaError_t e = launch_fwd_d32<V, V>(value, shapes, lstart, offsets, logits, pr, d, output, st, &handled);
    return launch_rc(e, handled);
}

// mixed-precision residual + LayerNorm (16-bit R) and its backward; partials: the deterministic twin's workspace
template <typename R>
static int add_layernorm_mixed(const float *x, const R *residual, const float *gamma, const float *beta, float *y,
                               R *y16, long long rows, int cols, float eps, void *stream) {
    if (!x || !residual || !gamma || !beta || !y) return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || cols <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_add_layernorm_mixed<R>(x, residual, gamma, beta, y, y16, rows, cols, eps,
                                                        (cudaStream_t)stream, &handled);
    return launch_rc(e, handled);
}

template <typename R>
static int add_layernorm_mixed_backward(const float *grad_y, const R *grad_y16, const float *x, const R *residual,
                                        const float *gamma, float *grad_x, R *grad_residual, float *grad_gamma,
                                        float *grad_beta, long long rows, int cols, float eps, void *workspace,
                                        void *stream, bool deterministic) {
    if ((!grad_y && !grad_y16) || !x || !residual || !gamma || !grad_x || !grad_residual || !grad_gamma ||
        !grad_beta || (deterministic && !workspace))
        return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || cols <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_add_layernorm_mixed_bwd<R>(grad_y, grad_y16, x, residual, gamma, grad_x, grad_residual,
                                                            grad_gamma, grad_beta, rows, cols, eps,
                                                            (cudaStream_t)stream, &handled,
                                                            static_cast<float *>(workspace));
    return launch_rc(e, handled);
}

// the bodies of the entries that come in a default and a deterministic (or training) form: `deterministic` /
// `train` select the form's null-pointer rule, the workspace / mean_rstd pointer selects the launch
static int linear(const float *x, const float *weight, const float *bias, float *y, int rows, int out_f, int in_f,
                  int relu, float *workspace, void *stream, bool deterministic) {
    if (!x || !weight || !y) return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || out_f <= 0 || in_f <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_linear_tf32x3(x, weight, bias, y, rows, out_f, in_f, relu, workspace,
                                               (cudaStream_t)stream, &handled, deterministic);
    return launch_rc(e, handled);
}

static int linear_presplit(const float *x, const float *split_weight, const float *bias, float *y, int rows,
                           int out_f, int in_f, int relu, void *stream, bool deterministic) {
    if (!x || !split_weight || !y) return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || out_f <= 0 || in_f <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    // the kernel only reads the split weight
    const cudaError_t e = launch_linear_tf32x3(x, nullptr, bias, y, rows, out_f, in_f, relu,
                                               const_cast<float *>(split_weight), (cudaStream_t)stream, &handled,
                                               deterministic);
    return launch_rc(e, handled);
}

static int add_layernorm_backward(const float *grad_y, const float *x, const float *residual, const float *gamma,
                                  float *grad_v, float *grad_gamma, float *grad_beta, long long rows, int cols,
                                  float eps, void *workspace, void *stream, bool deterministic) {
    if (!grad_y || !x || !gamma || !grad_v || !grad_gamma || !grad_beta || (deterministic && !workspace))
        return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || cols <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_add_layernorm_bwd(grad_y, x, residual, gamma, grad_v, grad_gamma, grad_beta, rows,
                                                   cols, eps, (cudaStream_t)stream, &handled,
                                                   static_cast<float *>(workspace));
    return launch_rc(e, handled);
}

static int linear_wgrad(const float *grad_y, const float *x, float *grad_weight, float *grad_bias, long long rows,
                        int out_f, int in_f, void *workspace, void *stream, bool deterministic) {
    if (!grad_y || !x || !grad_weight || (deterministic && !workspace)) return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || out_f <= 0 || in_f <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_linear_wgrad(grad_y, x, grad_weight, grad_bias, rows, out_f, in_f,
                                              (cudaStream_t)stream, &handled, static_cast<float *>(workspace));
    return launch_rc(e, handled);
}

template <typename T>
static int linear_mixed(const T *x, const T *weight, const float *bias, T *y, int rows, int out_f, int in_f, int relu,
                        void *stream) {
    if (!x || !weight || !y) return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || out_f <= 0 || in_f <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_linear_mixed<T>(x, weight, bias, y, rows, out_f, in_f, relu, (cudaStream_t)stream,
                                                 &handled);
    return launch_rc(e, handled);
}

template <typename T>
static int linear_mixed_wgrad(const T *grad_y, const T *x, float *grad_weight, float *grad_bias, long long rows,
                              int out_f, int in_f, void *workspace, void *stream) {
    if (!grad_y || !x || !grad_weight || !workspace) return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || out_f <= 0 || in_f <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_linear_mixed_wgrad<T>(grad_y, x, grad_weight, grad_bias, rows, out_f, in_f,
                                                       static_cast<float *>(workspace), (cudaStream_t)stream, &handled);
    return launch_rc(e, handled);
}

// V = float: y required (the fp32 entries pass y16 = NULL); 16-bit V: y and / or y16
template <typename V>
static int group_norm_nchw(const V *x, const float *channel_bias, const float *gamma, const float *beta, float *y,
                           V *y16, float *mean_rstd, int batch, int channels, int height, int width, int groups,
                           float eps, int relu, const float *up, int up_h, int up_w, void *workspace, void *stream,
                           bool train) {
    if (!x || !gamma || !beta || (!y && !y16) || (train && !mean_rstd) || !workspace) return MSDA_ERR_NULL_POINTER;
    if (batch <= 0 || channels <= 0 || height <= 0 || width <= 0 || groups <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_group_norm<V>(x, channel_bias, gamma, beta, y, y16, batch, channels, height, width,
                                               groups, eps, relu, up, up_h, up_w, static_cast<double *>(workspace),
                                               mean_rstd, (cudaStream_t)stream, &handled);
    return launch_rc(e, handled);
}

template <typename V>
static int group_norm_nchw_to_rows(const V *x, const float *channel_bias, const float *gamma, const float *beta,
                                   float *y_rows, float *mean_rstd, long long row_stride, long long image_stride,
                                   int batch, int channels, long long plane, int groups, float eps, int relu,
                                   void *workspace, void *stream, bool train) {
    if (!x || !gamma || !beta || !y_rows || (train && !mean_rstd) || !workspace) return MSDA_ERR_NULL_POINTER;
    if (batch <= 0 || channels <= 0 || plane <= 0 || groups <= 0 || row_stride < channels || image_stride < 0)
        return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_group_norm_rows<V>(x, channel_bias, gamma, beta, y_rows, batch, channels, plane,
                                                    groups, eps, relu, row_stride, image_stride,
                                                    static_cast<double *>(workspace), mean_rstd, (cudaStream_t)stream,
                                                    &handled);
    return launch_rc(e, handled);
}

// The NCHW backward: fp32 (V = float, grad_y), or 16-bit x / grad_x with exactly one of grad_y (fp32) and grad_y16
// (V), the gradient of whichever output the forward wrote
template <typename V>
static int group_norm_backward_nchw(const float *grad_y, const V *grad_y16, const V *x, const float *channel_bias,
                                    const float *gamma, const float *beta, const float *mean_rstd, V *grad_x,
                                    float *grad_gamma, float *grad_beta, float *grad_channel_bias, float *grad_up,
                                    int batch, int channels, int height, int width, int groups, int relu, int up_h,
                                    int up_w, void *workspace, void *stream) {
    if ((!grad_y && !grad_y16) || !x || !gamma || !beta || !mean_rstd || !grad_x || !grad_gamma || !grad_beta ||
        !workspace)
        return MSDA_ERR_NULL_POINTER;
    if (grad_y && grad_y16) return MSDA_ERR_UNSUPPORTED;
    if (batch <= 0 || channels <= 0 || height <= 0 || width <= 0 || groups <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    cudaError_t e;
    if (grad_y)
        e = launch_group_norm_bwd<float, V>(grad_y, x, channel_bias, gamma, beta, mean_rstd, grad_x, grad_gamma,
                                            grad_beta, grad_channel_bias, grad_up, batch, channels, height, width,
                                            groups, relu, up_h, up_w, static_cast<double *>(workspace),
                                            (cudaStream_t)stream, &handled);
    else if constexpr (is16<V>)
        e = launch_group_norm_bwd<V, V>(grad_y16, x, channel_bias, gamma, beta, mean_rstd, grad_x, grad_gamma,
                                        grad_beta, grad_channel_bias, grad_up, batch, channels, height, width, groups,
                                        relu, up_h, up_w, static_cast<double *>(workspace), (cudaStream_t)stream,
                                        &handled);
    else
        return MSDA_ERR_NULL_POINTER;
    return launch_rc(e, handled);
}

template <typename V>
static int group_norm_rows_backward(const float *grad_y_rows, long long row_stride, long long image_stride,
                                    const V *x, const float *channel_bias, const float *gamma, const float *beta,
                                    const float *mean_rstd, V *grad_x, float *grad_gamma, float *grad_beta,
                                    float *grad_channel_bias, int batch, int channels, long long plane, int groups,
                                    int relu, void *workspace, void *stream) {
    if (!grad_y_rows || !x || !gamma || !beta || !mean_rstd || !grad_x || !grad_gamma || !grad_beta || !workspace)
        return MSDA_ERR_NULL_POINTER;
    if (batch <= 0 || channels <= 0 || plane <= 0 || groups <= 0 || row_stride < channels || image_stride < 0)
        return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_group_norm_rows_bwd<V>(grad_y_rows, row_stride, image_stride, x, channel_bias, gamma,
                                                        beta, mean_rstd, grad_x, grad_gamma, grad_beta,
                                                        grad_channel_bias, batch, channels, plane, groups, relu,
                                                        static_cast<double *>(workspace), (cudaStream_t)stream,
                                                        &handled);
    return launch_rc(e, handled);
}

template <typename V>
static int add_channel_bias_nchw(V *x, const float *bias, int batch, int channels, long long plane, void *stream) {
    if (!x || !bias) return MSDA_ERR_NULL_POINTER;
    if (batch <= 0 || channels <= 0 || plane <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_channel_bias<V>(x, bias, batch, channels, plane, (cudaStream_t)stream, &handled);
    return launch_rc(e, handled);
}

}  // namespace msda

using namespace msda;

extern "C" {

int msda_b200_abi_version(void) { return MSDA_B200_ABI_VERSION; }

const char *msda_b200_error_string(int code) {
    switch (code) {
        case MSDA_OK: return "success";
        case MSDA_ERR_NULL_POINTER: return "msda_b200: a required pointer is NULL";
        case MSDA_ERR_BAD_SHAPE: return "msda_b200: a tensor size is zero or negative";
        case MSDA_ERR_UNSUPPORTED: return "msda_b200: unsupported configuration (num_levels > 16, or a shape the fused path does not cover)";
        case MSDA_ERR_BAD_OPTION: return "msda_b200: unknown option name or value out of range";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "msda_b200: unknown error code";
}

long long msda_b200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int msda_b200_set_option(const char *name, int value) {
    const int i = option_index(name);
    if (i < 0 || value < 0 || value > 65535) return MSDA_ERR_BAD_OPTION;
    g_options[i].store(value, std::memory_order_relaxed);
    return MSDA_OK;
}

int msda_b200_get_option(const char *name, int *value) {
    const int i = option_index(name);
    if (i < 0 || !value) return MSDA_ERR_BAD_OPTION;
    *value = g_options[i].load(std::memory_order_relaxed);
    return MSDA_OK;
}

int msda_b200_forward_f32(const float *value, const int64_t *spatial_shapes,
                          const int64_t *level_start, const float *sampling_loc,
                          const float *attn_weight, int batch, int spatial_size, int num_heads,
                          int channels, int num_levels, int num_query, int num_point, float *output,
                          void *stream) {
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    return forward<float>(value, spatial_shapes, level_start, sampling_loc, attn_weight, Producers{}, d, output,
                          (cudaStream_t)stream);
}

int msda_b200_forward_f64(const double *value, const int64_t *spatial_shapes,
                          const int64_t *level_start, const double *sampling_loc,
                          const double *attn_weight, int batch, int spatial_size, int num_heads,
                          int channels, int num_levels, int num_query, int num_point,
                          double *output, void *stream) {
    if (!value || !spatial_shapes || !level_start || !sampling_loc || !attn_weight || !output)
        return MSDA_ERR_NULL_POINTER;
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    if (int rc = check_dims(d)) return rc;
    return (int)launch_fwd_generic<double, double>(value, spatial_shapes, level_start, sampling_loc,
                                           attn_weight, d, output, (cudaStream_t)stream);
}

int msda_b200_backward_f32(const float *grad_output, const float *value,
                           const int64_t *spatial_shapes, const int64_t *level_start,
                           const float *sampling_loc, const float *attn_weight, int batch,
                           int spatial_size, int num_heads, int channels, int num_levels,
                           int num_query, int num_point, float *grad_value,
                           float *grad_sampling_loc, float *grad_attn_weight, void *stream) {
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    return backward<float>(grad_output, value, spatial_shapes, level_start, sampling_loc, attn_weight, Producers{}, d,
                           grad_value, grad_sampling_loc, grad_attn_weight, (cudaStream_t)stream);
}

int msda_b200_backward_f64(const double *grad_output, const double *value,
                           const int64_t *spatial_shapes, const int64_t *level_start,
                           const double *sampling_loc, const double *attn_weight, int batch,
                           int spatial_size, int num_heads, int channels, int num_levels,
                           int num_query, int num_point, double *grad_value,
                           double *grad_sampling_loc, double *grad_attn_weight, void *stream) {
    if (!grad_output || !value || !spatial_shapes || !level_start || !sampling_loc || !attn_weight ||
        !grad_value || !grad_sampling_loc || !grad_attn_weight)
        return MSDA_ERR_NULL_POINTER;
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    if (int rc = check_dims(d)) return rc;
    return (int)launch_bwd_generic<double, double>(grad_output, value, spatial_shapes, level_start,
                                           sampling_loc, attn_weight, d, grad_value,
                                           grad_sampling_loc, grad_attn_weight, (cudaStream_t)stream);
}

int msda_b200_fused_forward_strided_f32(const float *value, const int64_t *spatial_shapes,
                                        const int64_t *level_start, const float *reference_points,
                                        long long ref_batch_stride, const float *sampling_offsets,
                                        int offsets_row_stride, const float *attn_logits,
                                        int logits_row_stride, const float *offsets_table,
                                        const float *logits_table, int batch, int spatial_size, int num_heads,
                                        int channels, int num_levels, int num_query, int num_point,
                                        float *output, void *stream) {
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    return fused_forward_strided<float>(value, spatial_shapes, level_start, reference_points, ref_batch_stride,
                                        sampling_offsets, offsets_row_stride, attn_logits, logits_row_stride,
                                        offsets_table, logits_table, d, output, (cudaStream_t)stream);
}

int msda_b200_fused_forward_f32(const float *value, const int64_t *spatial_shapes,
                                const int64_t *level_start, const float *reference_points,
                                long long ref_batch_stride, const float *sampling_offsets,
                                const float *attn_logits, int batch, int spatial_size, int num_heads,
                                int channels, int num_levels, int num_query, int num_point,
                                float *output, void *stream) {
    return msda_b200_fused_forward_strided_f32(value, spatial_shapes, level_start, reference_points,
                                               ref_batch_stride, sampling_offsets,
                                               2 * num_heads * num_levels * num_point, attn_logits,
                                               num_heads * num_levels * num_point, nullptr, nullptr, batch, spatial_size,
                                               num_heads, channels, num_levels, num_query, num_point, output,
                                               stream);
}

int msda_b200_fused_backward_f32(const float *grad_output, const float *value,
                                 const int64_t *spatial_shapes, const int64_t *level_start,
                                 const float *reference_points, long long ref_batch_stride,
                                 const float *sampling_offsets, const float *attn_logits, int batch,
                                 int spatial_size, int num_heads, int channels, int num_levels,
                                 int num_query, int num_point, float *grad_value,
                                 float *grad_sampling_offsets, float *grad_attn_logits, void *stream) {
    if (!reference_points) return MSDA_ERR_NULL_POINTER;      // (it selects the fused form)
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    return backward<float>(grad_output, value, spatial_shapes, level_start, sampling_offsets, attn_logits,
                           Producers{reference_points, ref_batch_stride}, d, grad_value, grad_sampling_offsets,
                           grad_attn_logits, (cudaStream_t)stream);
}

long long msda_b200_backward_deterministic_workspace_bytes(int batch, int spatial_size, int num_heads, int channels,
                                                          int num_levels, int num_query, int num_point,
                                                          int value_bytes) {
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    DetLayout l;
    // 16-bit value (2 bytes): the records carry fp32 weights
    if (check_dims(d) != MSDA_OK || (value_bytes != 2 && value_bytes != 4 && value_bytes != 8) ||
        !det_layout(d, value_bytes == 2 ? 4 : value_bytes, &l))
        return 0;
    return (long long)l.total;
}

int msda_b200_backward_deterministic_f32(const float *grad_output, const float *value,
                                         const int64_t *spatial_shapes, const int64_t *level_start,
                                         const float *sampling_loc, const float *attn_weight, int batch,
                                         int spatial_size, int num_heads, int channels, int num_levels,
                                         int num_query, int num_point, float *grad_value,
                                         float *grad_sampling_loc, float *grad_attn_weight, void *workspace,
                                         void *stream) {
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    return backward_deterministic<float, float>(grad_output, value, spatial_shapes, level_start, sampling_loc, attn_weight,
                                         Producers{}, d, grad_value, grad_sampling_loc, grad_attn_weight, workspace,
                                         (cudaStream_t)stream);
}

int msda_b200_backward_deterministic_f64(const double *grad_output, const double *value,
                                         const int64_t *spatial_shapes, const int64_t *level_start,
                                         const double *sampling_loc, const double *attn_weight, int batch,
                                         int spatial_size, int num_heads, int channels, int num_levels,
                                         int num_query, int num_point, double *grad_value,
                                         double *grad_sampling_loc, double *grad_attn_weight, void *workspace,
                                         void *stream) {
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    return backward_deterministic<double, double>(grad_output, value, spatial_shapes, level_start, sampling_loc, attn_weight,
                                          Producers{}, d, grad_value, grad_sampling_loc, grad_attn_weight, workspace,
                                          (cudaStream_t)stream);
}

int msda_b200_fused_backward_deterministic_f32(const float *grad_output, const float *value,
                                               const int64_t *spatial_shapes, const int64_t *level_start,
                                               const float *reference_points, long long ref_batch_stride,
                                               const float *sampling_offsets, const float *attn_logits, int batch,
                                               int spatial_size, int num_heads, int channels, int num_levels,
                                               int num_query, int num_point, float *grad_value,
                                               float *grad_sampling_offsets, float *grad_attn_logits,
                                               void *workspace, void *stream) {
    if (!reference_points) return MSDA_ERR_NULL_POINTER;      // (it selects the fused form)
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    return backward_deterministic<float, float>(grad_output, value, spatial_shapes, level_start, sampling_offsets,
                                         attn_logits, Producers{reference_points, ref_batch_stride}, d, grad_value,
                                         grad_sampling_offsets, grad_attn_logits, workspace, (cudaStream_t)stream);
}

// ---- mixed precision: bf16 / fp16 value, output, grad_output and grad_value; fp32 locations, weights and their
// gradients; fp32 sums.  The fused entries: 16-bit raw offsets, logits and their gradients, fp32 reference points ----
#define MSDA_MIXED_ENTRIES(SUFFIX, V)                                                                                \
    int msda_b200_forward_##SUFFIX(const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start,  \
                                   const float *sampling_loc, const float *attn_weight, int batch, int spatial_size,  \
                                   int num_heads, int channels, int num_levels, int num_query, int num_point,        \
                                   uint16_t *output, void *stream) {                                                \
        const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};                    \
        return forward<V>(reinterpret_cast<const V *>(value), spatial_shapes, level_start, sampling_loc, attn_weight, \
                          Producers{}, d, reinterpret_cast<V *>(output), (cudaStream_t)stream);                      \
    }                                                                                                                \
    int msda_b200_backward_##SUFFIX(const uint16_t *grad_output, const uint16_t *value, const int64_t *spatial_shapes, \
                                    const int64_t *level_start, const float *sampling_loc, const float *attn_weight, \
                                    int batch, int spatial_size, int num_heads, int channels, int num_levels,        \
                                    int num_query, int num_point, float *grad_value_accum, uint16_t *grad_value,     \
                                    float *grad_sampling_loc, float *grad_attn_weight, void *stream) {               \
        const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};                    \
        return backward_mixed<V>(reinterpret_cast<const V *>(grad_output), reinterpret_cast<const V *>(value),       \
                                 spatial_shapes, level_start, sampling_loc, attn_weight, Producers{}, d,             \
                                 grad_value_accum,                                                                   \
                                 reinterpret_cast<V *>(grad_value), grad_sampling_loc, grad_attn_weight,             \
                                 (cudaStream_t)stream);                                                              \
    }                                                                                                                \
    int msda_b200_backward_deterministic_##SUFFIX(                                                                   \
        const uint16_t *grad_output, const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start, \
        const float *sampling_loc, const float *attn_weight, int batch, int spatial_size, int num_heads, int channels, \
        int num_levels, int num_query, int num_point, uint16_t *grad_value, float *grad_sampling_loc,                \
        float *grad_attn_weight, void *workspace, void *stream) {                                                   \
        const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};                    \
        return backward_deterministic<V, float>(reinterpret_cast<const V *>(grad_output),                           \
                                                reinterpret_cast<const V *>(value), spatial_shapes, level_start,     \
                                                sampling_loc, attn_weight, Producers{}, d,                           \
                                                reinterpret_cast<V *>(grad_value), grad_sampling_loc,                \
                                                grad_attn_weight, workspace, (cudaStream_t)stream);                  \
    }                                                                                                                \
    int msda_b200_fused_forward_##SUFFIX(const uint16_t *value, const int64_t *spatial_shapes,                       \
                                         const int64_t *level_start, const float *reference_points,                  \
                                         long long ref_batch_stride, const uint16_t *sampling_offsets,               \
                                         const uint16_t *attn_logits, int batch, int spatial_size, int num_heads,    \
                                         int channels, int num_levels, int num_query, int num_point,                 \
                                         uint16_t *output, void *stream) {                                          \
        if (!reference_points) return MSDA_ERR_NULL_POINTER;      /* (it selects the fused form) */                  \
        const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};                    \
        return forward<V, V>(reinterpret_cast<const V *>(value), spatial_shapes, level_start,                        \
                             reinterpret_cast<const V *>(sampling_offsets), reinterpret_cast<const V *>(attn_logits), \
                             Producers{reference_points, ref_batch_stride}, d, reinterpret_cast<V *>(output),        \
                             (cudaStream_t)stream);                                                                  \
    }                                                                                                                \
    int msda_b200_fused_backward_##SUFFIX(                                                                           \
        const uint16_t *grad_output, const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start, \
        const float *reference_points, long long ref_batch_stride, const uint16_t *sampling_offsets,                 \
        const uint16_t *attn_logits, int batch, int spatial_size, int num_heads, int channels, int num_levels,        \
        int num_query, int num_point, float *grad_value_accum, uint16_t *grad_value, uint16_t *grad_sampling_offsets, \
        uint16_t *grad_attn_logits, void *stream) {                                                                  \
        if (!reference_points) return MSDA_ERR_NULL_POINTER;                                                         \
        const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};                    \
        return backward_mixed<V, V>(reinterpret_cast<const V *>(grad_output), reinterpret_cast<const V *>(value),    \
                                    spatial_shapes, level_start, reinterpret_cast<const V *>(sampling_offsets),      \
                                    reinterpret_cast<const V *>(attn_logits),                                        \
                                    Producers{reference_points, ref_batch_stride}, d, grad_value_accum,              \
                                    reinterpret_cast<V *>(grad_value), reinterpret_cast<V *>(grad_sampling_offsets), \
                                    reinterpret_cast<V *>(grad_attn_logits), (cudaStream_t)stream);                  \
    }                                                                                                                \
    int msda_b200_fused_backward_deterministic_##SUFFIX(                                                             \
        const uint16_t *grad_output, const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start, \
        const float *reference_points, long long ref_batch_stride, const uint16_t *sampling_offsets,                 \
        const uint16_t *attn_logits, int batch, int spatial_size, int num_heads, int channels, int num_levels,        \
        int num_query, int num_point, uint16_t *grad_value, uint16_t *grad_sampling_offsets,                         \
        uint16_t *grad_attn_logits, void *workspace, void *stream) {                                                 \
        if (!reference_points) return MSDA_ERR_NULL_POINTER;                                                         \
        const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};                    \
        return backward_deterministic<V, float, V>(                                                                  \
            reinterpret_cast<const V *>(grad_output), reinterpret_cast<const V *>(value), spatial_shapes, level_start, \
            reinterpret_cast<const V *>(sampling_offsets), reinterpret_cast<const V *>(attn_logits),                 \
            Producers{reference_points, ref_batch_stride}, d, reinterpret_cast<V *>(grad_value),                     \
            reinterpret_cast<V *>(grad_sampling_offsets), reinterpret_cast<V *>(grad_attn_logits), workspace,        \
            (cudaStream_t)stream);                                                                                   \
    }                                                                                                                \
    int msda_b200_fused_forward_strided_##SUFFIX(                                                                   \
        const uint16_t *value, const int64_t *spatial_shapes, const int64_t *level_start, const float *reference_points, \
        long long ref_batch_stride, const uint16_t *sampling_offsets, int offsets_row_stride,                         \
        const uint16_t *attn_logits, int logits_row_stride, const float *offsets_table, const float *logits_table,    \
        int batch, int spatial_size, int num_heads, int channels, int num_levels, int num_query, int num_point,       \
        uint16_t *output, void *stream) {                                                                            \
        const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};                    \
        return fused_forward_strided<V>(reinterpret_cast<const V *>(value), spatial_shapes, level_start,             \
                                        reference_points, ref_batch_stride,                                          \
                                        reinterpret_cast<const V *>(sampling_offsets), offsets_row_stride,           \
                                        reinterpret_cast<const V *>(attn_logits), logits_row_stride, offsets_table,  \
                                        logits_table, d, reinterpret_cast<V *>(output), (cudaStream_t)stream);       \
    }                                                                                                                \
    int msda_b200_add_layernorm_mixed_##SUFFIX(const float *x, const uint16_t *residual, const float *gamma,         \
                                               const float *beta, float *y, uint16_t *y16, long long rows, int cols, \
                                               float eps, void *stream) {                                            \
        return add_layernorm_mixed<V>(x, reinterpret_cast<const V *>(residual), gamma, beta, y,                      \
                                      reinterpret_cast<V *>(y16), rows, cols, eps, stream);                         \
    }                                                                                                                \
    int msda_b200_add_layernorm_mixed_backward_##SUFFIX(                                                             \
        const float *grad_y, const uint16_t *grad_y16, const float *x, const uint16_t *residual, const float *gamma,  \
        float *grad_x, uint16_t *grad_residual, float *grad_gamma, float *grad_beta, long long rows, int cols,        \
        float eps, void *stream) {                                                                                   \
        return add_layernorm_mixed_backward<V>(grad_y, reinterpret_cast<const V *>(grad_y16), x,                     \
                                               reinterpret_cast<const V *>(residual), gamma, grad_x,                 \
                                               reinterpret_cast<V *>(grad_residual), grad_gamma, grad_beta, rows,    \
                                               cols, eps, nullptr, stream, false);                                   \
    }                                                                                                                \
    int msda_b200_add_layernorm_mixed_backward_deterministic_##SUFFIX(                                               \
        const float *grad_y, const uint16_t *grad_y16, const float *x, const uint16_t *residual, const float *gamma,  \
        float *grad_x, uint16_t *grad_residual, float *grad_gamma, float *grad_beta, long long rows, int cols,        \
        float eps, void *workspace, void *stream) {                                                                  \
        return add_layernorm_mixed_backward<V>(grad_y, reinterpret_cast<const V *>(grad_y16), x,                     \
                                               reinterpret_cast<const V *>(residual), gamma, grad_x,                 \
                                               reinterpret_cast<V *>(grad_residual), grad_gamma, grad_beta, rows,    \
                                               cols, eps, workspace, stream, true);                                  \
    }                                                                                                                \
    int msda_b200_group_norm_nchw_mixed_##SUFFIX(                                                                    \
        const uint16_t *x, const float *channel_bias, const float *gamma, const float *beta, float *y, uint16_t *y16,\
        int batch, int channels, int height, int width, int groups, float eps, int relu, const float *up, int up_h,  \
        int up_w, void *workspace, void *stream) {                                                                   \
        return group_norm_nchw<V>(reinterpret_cast<const V *>(x), channel_bias, gamma, beta, y, reinterpret_cast<V *>(y16),\
                                  nullptr, batch, channels, height, width, groups, eps, relu, up, up_h, up_w, workspace,\
                                  stream, false);                                                                    \
    }                                                                                                                \
    int msda_b200_group_norm_nchw_mixed_train_##SUFFIX(                                                              \
        const uint16_t *x, const float *channel_bias, const float *gamma, const float *beta, float *y, uint16_t *y16,\
        float *mean_rstd, int batch, int channels, int height, int width, int groups, float eps, int relu,           \
        const float *up, int up_h, int up_w, void *workspace, void *stream) {                                        \
        return group_norm_nchw<V>(reinterpret_cast<const V *>(x), channel_bias, gamma, beta, y, reinterpret_cast<V *>(y16),\
                                  mean_rstd, batch, channels, height, width, groups, eps, relu, up, up_h, up_w, workspace,\
                                  stream, true);                                                                     \
    }                                                                                                                \
    int msda_b200_group_norm_nchw_to_rows_mixed_##SUFFIX(                                                            \
        const uint16_t *x, const float *channel_bias, const float *gamma, const float *beta, float *y_rows,          \
        long long row_stride, long long image_stride, int batch, int channels, long long plane, int groups, float eps,\
        int relu, void *workspace, void *stream) {                                                                   \
        return group_norm_nchw_to_rows<V>(reinterpret_cast<const V *>(x), channel_bias, gamma, beta, y_rows, nullptr,\
                                          row_stride, image_stride, batch, channels, plane, groups, eps, relu, workspace,\
                                          stream, false);                                                            \
    }                                                                                                                \
    int msda_b200_group_norm_nchw_to_rows_mixed_train_##SUFFIX(                                                      \
        const uint16_t *x, const float *channel_bias, const float *gamma, const float *beta, float *y_rows,          \
        float *mean_rstd, long long row_stride, long long image_stride, int batch, int channels, long long plane,    \
        int groups, float eps, int relu, void *workspace, void *stream) {                                            \
        return group_norm_nchw_to_rows<V>(reinterpret_cast<const V *>(x), channel_bias, gamma, beta, y_rows, mean_rstd,\
                                          row_stride, image_stride, batch, channels, plane, groups, eps, relu, workspace,\
                                          stream, true);                                                             \
    }                                                                                                                \
    int msda_b200_group_norm_backward_nchw_mixed_##SUFFIX(                                                           \
        const float *grad_y, const uint16_t *grad_y16, const uint16_t *x, const float *channel_bias, const float *gamma,\
        const float *beta, const float *mean_rstd, uint16_t *grad_x, float *grad_gamma, float *grad_beta,            \
        float *grad_channel_bias, float *grad_up, int batch, int channels, int height, int width, int groups, int relu,\
        int up_h, int up_w, void *workspace, void *stream) {                                                         \
        return group_norm_backward_nchw<V>(grad_y, reinterpret_cast<const V *>(grad_y16), reinterpret_cast<const V *>(x),\
                                           channel_bias, gamma, beta, mean_rstd, reinterpret_cast<V *>(grad_x),      \
                                           grad_gamma, grad_beta, grad_channel_bias, grad_up, batch, channels, height,\
                                           width, groups, relu, up_h, up_w, workspace, stream);                      \
    }                                                                                                                \
    int msda_b200_group_norm_rows_backward_mixed_##SUFFIX(                                                           \
        const float *grad_y_rows, long long row_stride, long long image_stride, const uint16_t *x,                   \
        const float *channel_bias, const float *gamma, const float *beta, const float *mean_rstd, uint16_t *grad_x,  \
        float *grad_gamma, float *grad_beta, float *grad_channel_bias, int batch, int channels, long long plane,     \
        int groups, int relu, void *workspace, void *stream) {                                                       \
        return group_norm_rows_backward<V>(grad_y_rows, row_stride, image_stride, reinterpret_cast<const V *>(x),    \
                                           channel_bias, gamma, beta, mean_rstd, reinterpret_cast<V *>(grad_x), grad_gamma,\
                                           grad_beta, grad_channel_bias, batch, channels, plane, groups, relu, workspace,\
                                           stream);                                                                  \
    }                                                                                                                \
    int msda_b200_add_channel_bias_nchw_##SUFFIX(uint16_t *x, const float *bias, int batch, int channels,            \
                                                 long long plane, void *stream) {                                    \
        return add_channel_bias_nchw<V>(reinterpret_cast<V *>(x), bias, batch, channels, plane, stream);             \
    }
MSDA_MIXED_ENTRIES(bf16, __nv_bfloat16)
MSDA_MIXED_ENTRIES(f16, __half)
#undef MSDA_MIXED_ENTRIES

// ---- 16-bit Linear under torch.autocast: bf16 / fp16 operands, fp32 bias, accumulation and weight gradient ----
#define MSDA_LINEAR_MIXED_ENTRIES(SUFFIX, T)                                                                         \
    int msda_b200_linear_mixed_##SUFFIX(const uint16_t *x, const uint16_t *weight16, const float *bias, uint16_t *y, \
                                        int rows, int out_features, int in_features, int relu, void *stream) {      \
        return linear_mixed<T>(reinterpret_cast<const T *>(x), reinterpret_cast<const T *>(weight16), bias,          \
                               reinterpret_cast<T *>(y), rows, out_features, in_features, relu, stream);             \
    }                                                                                                                \
    int msda_b200_linear_mixed_wgrad_##SUFFIX(const uint16_t *grad_y, const uint16_t *x, float *grad_weight,         \
                                              float *grad_bias, long long rows, int out_features, int in_features,   \
                                              void *workspace, void *stream) {                                       \
        return linear_mixed_wgrad<T>(reinterpret_cast<const T *>(grad_y), reinterpret_cast<const T *>(x),            \
                                     grad_weight, grad_bias, rows, out_features, in_features, workspace, stream);    \
    }
MSDA_LINEAR_MIXED_ENTRIES(bf16, __nv_bfloat16)
MSDA_LINEAR_MIXED_ENTRIES(f16, __half)
#undef MSDA_LINEAR_MIXED_ENTRIES

long long msda_b200_linear_mixed_wgrad_workspace_bytes(long long rows, int out_features, int in_features) {
    if (rows <= 0 || out_features <= 0 || in_features <= 0) return 0;
    return linear_mixed_wgrad_workspace_floats(rows, out_features, in_features) * (long long)sizeof(float);
}

int msda_b200_linear_f32(const float *x, const float *weight, const float *bias, float *y, int rows,
                         int out_features, int in_features, int relu, float *workspace, void *stream) {
    return linear(x, weight, bias, y, rows, out_features, in_features, relu, workspace, stream, false);
}

int msda_b200_linear_deterministic_f32(const float *x, const float *weight, const float *bias, float *y, int rows,
                                       int out_features, int in_features, int relu, float *workspace, void *stream) {
    return linear(x, weight, bias, y, rows, out_features, in_features, relu, workspace, stream, true);
}

int msda_b200_split_weight_f32(const float *weight, float *split_weight, int out_features, int in_features,
                               void *stream) {
    if (!weight || !split_weight) return MSDA_ERR_NULL_POINTER;
    if (out_features <= 0 || in_features <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_split_weight(weight, split_weight, out_features, in_features, (cudaStream_t)stream,
                                              &handled);
    return launch_rc(e, handled);
}

int msda_b200_linear_presplit_f32(const float *x, const float *split_weight, const float *bias, float *y, int rows,
                                  int out_features, int in_features, int relu, void *stream) {
    return linear_presplit(x, split_weight, bias, y, rows, out_features, in_features, relu, stream, false);
}

int msda_b200_linear_presplit_deterministic_f32(const float *x, const float *split_weight, const float *bias, float *y,
                                                int rows, int out_features, int in_features, int relu, void *stream) {
    return linear_presplit(x, split_weight, bias, y, rows, out_features, in_features, relu, stream, true);
}

int msda_b200_add_layernorm_f32(const float *x, const float *residual, const float *gamma, const float *beta,
                                float *y, long long rows, int cols, float eps, void *stream) {
    if (!x || !gamma || !beta || !y) return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || cols <= 0) return MSDA_ERR_BAD_SHAPE;
    bool handled = false;
    const cudaError_t e = launch_add_layernorm(x, residual, gamma, beta, y, rows, cols, eps, (cudaStream_t)stream,
                                               &handled);
    return launch_rc(e, handled);
}

int msda_b200_add_layernorm_backward_f32(const float *grad_y, const float *x, const float *residual,
                                         const float *gamma, float *grad_v, float *grad_gamma, float *grad_beta,
                                         long long rows, int cols, float eps, void *stream) {
    return add_layernorm_backward(grad_y, x, residual, gamma, grad_v, grad_gamma, grad_beta, rows, cols, eps, nullptr,
                                  stream, false);
}

int msda_b200_add_layernorm_backward_deterministic_f32(const float *grad_y, const float *x, const float *residual,
                                                       const float *gamma, float *grad_v, float *grad_gamma,
                                                       float *grad_beta, long long rows, int cols, float eps,
                                                       void *workspace, void *stream) {
    return add_layernorm_backward(grad_y, x, residual, gamma, grad_v, grad_gamma, grad_beta, rows, cols, eps,
                                  workspace, stream, true);
}

long long msda_b200_add_layernorm_backward_deterministic_workspace_bytes(long long rows, int cols) {
    if (rows <= 0 || cols <= 0) return 0;
    return add_layernorm_bwd_partials(rows, cols) * (long long)sizeof(float);
}

int msda_b200_linear_wgrad_f32(const float *grad_y, const float *x, float *grad_weight, float *grad_bias,
                               long long rows, int out_features, int in_features, void *stream) {
    return linear_wgrad(grad_y, x, grad_weight, grad_bias, rows, out_features, in_features, nullptr, stream, false);
}

int msda_b200_linear_wgrad_deterministic_f32(const float *grad_y, const float *x, float *grad_weight, float *grad_bias,
                                             long long rows, int out_features, int in_features, void *workspace,
                                             void *stream) {
    return linear_wgrad(grad_y, x, grad_weight, grad_bias, rows, out_features, in_features, workspace, stream, true);
}

long long msda_b200_linear_wgrad_deterministic_workspace_bytes(long long rows, int out_features, int in_features) {
    if (rows <= 0 || out_features <= 0 || in_features <= 0) return 0;
    return linear_wgrad_partials(rows, out_features, in_features) * (long long)sizeof(float);
}

int msda_b200_group_norm_nchw_f32(const float *x, const float *channel_bias, const float *gamma, const float *beta,
                                  float *y, int batch, int channels, int height, int width, int groups, float eps,
                                  int relu, const float *up, int up_h, int up_w, void *workspace, void *stream) {
    if (!y) return MSDA_ERR_NULL_POINTER;
    return group_norm_nchw<float>(x, channel_bias, gamma, beta, y, nullptr, nullptr, batch, channels, height, width,
                                  groups, eps, relu, up, up_h, up_w, workspace, stream, false);
}

int msda_b200_group_norm_nchw_to_rows_f32(const float *x, const float *channel_bias, const float *gamma,
                                          const float *beta, float *y_rows, long long row_stride,
                                          long long image_stride, int batch, int channels, long long plane,
                                          int groups, float eps, int relu, void *workspace, void *stream) {
    return group_norm_nchw_to_rows<float>(x, channel_bias, gamma, beta, y_rows, nullptr, row_stride, image_stride,
                                          batch, channels, plane, groups, eps, relu, workspace, stream, false);
}

int msda_b200_group_norm_nchw_train_f32(const float *x, const float *channel_bias, const float *gamma,
                                        const float *beta, float *y, float *mean_rstd, int batch, int channels,
                                        int height, int width, int groups, float eps, int relu, const float *up,
                                        int up_h, int up_w, void *workspace, void *stream) {
    if (!y) return MSDA_ERR_NULL_POINTER;
    return group_norm_nchw<float>(x, channel_bias, gamma, beta, y, nullptr, mean_rstd, batch, channels, height, width,
                                  groups, eps, relu, up, up_h, up_w, workspace, stream, true);
}

int msda_b200_group_norm_nchw_to_rows_train_f32(const float *x, const float *channel_bias, const float *gamma,
                                                const float *beta, float *y_rows, float *mean_rstd,
                                                long long row_stride, long long image_stride, int batch,
                                                int channels, long long plane, int groups, float eps, int relu,
                                                void *workspace, void *stream) {
    return group_norm_nchw_to_rows<float>(x, channel_bias, gamma, beta, y_rows, mean_rstd, row_stride, image_stride,
                                          batch, channels, plane, groups, eps, relu, workspace, stream, true);
}

int msda_b200_group_norm_backward_nchw_f32(const float *grad_y, const float *x, const float *channel_bias,
                                           const float *gamma, const float *beta, const float *mean_rstd,
                                           float *grad_x, float *grad_gamma, float *grad_beta,
                                           float *grad_channel_bias, float *grad_up, int batch, int channels,
                                           int height, int width, int groups, int relu, int up_h, int up_w,
                                           void *workspace, void *stream) {
    return group_norm_backward_nchw<float>(grad_y, nullptr, x, channel_bias, gamma, beta, mean_rstd, grad_x,
                                           grad_gamma, grad_beta, grad_channel_bias, grad_up, batch, channels, height,
                                           width, groups, relu, up_h, up_w, workspace, stream);
}

int msda_b200_group_norm_rows_backward_f32(const float *grad_y_rows, long long row_stride, long long image_stride,
                                           const float *x, const float *channel_bias, const float *gamma,
                                           const float *beta, const float *mean_rstd, float *grad_x,
                                           float *grad_gamma, float *grad_beta, float *grad_channel_bias, int batch,
                                           int channels, long long plane, int groups, int relu, void *workspace,
                                           void *stream) {
    return group_norm_rows_backward<float>(grad_y_rows, row_stride, image_stride, x, channel_bias, gamma, beta,
                                           mean_rstd, grad_x, grad_gamma, grad_beta, grad_channel_bias, batch,
                                           channels, plane, groups, relu, workspace, stream);
}

int msda_b200_add_channel_bias_nchw_f32(float *x, const float *bias, int batch, int channels, long long plane,
                                        void *stream) {
    return add_channel_bias_nchw<float>(x, bias, batch, channels, plane, stream);
}

long long msda_b200_group_norm_workspace_bytes(int batch, int groups) {
    if (batch <= 0 || groups <= 0) return 0;
    return (long long)group_norm_workspace_doubles(batch, groups) * (long long)sizeof(double);
}

long long msda_b200_group_norm_backward_workspace_bytes(int batch, int channels) {
    if (batch <= 0 || channels <= 0) return 0;
    return group_norm_bwd_workspace_doubles(batch, channels) * (long long)sizeof(double);
}

int msda_b200_transpose_f32(const float *x, float *y, long long rows, int cols, void *stream) {
    if (!x || !y) return MSDA_ERR_NULL_POINTER;
    if (rows <= 0 || cols <= 0 || (cols + 31) / 32 > 65535) return MSDA_ERR_BAD_SHAPE;
    return (int)launch_transpose(x, y, rows, cols, (cudaStream_t)stream);
}

int msda_b200_debug_indices_f32(const int64_t *spatial_shapes, const int64_t *level_start,
                                const float *sampling_loc, int batch, int spatial_size,
                                int num_heads, int channels, int num_levels, int num_query,
                                int num_point, int32_t *idx, int64_t *off, void *stream) {
    if (!spatial_shapes || !level_start || !sampling_loc || !idx || !off) return MSDA_ERR_NULL_POINTER;
    const Dims d{batch, spatial_size, num_heads, channels, num_levels, num_query, num_point};
    if (int rc = check_dims(d)) return rc;
    return (int)launch_debug_indices(spatial_shapes, level_start, sampling_loc, d, idx, off,
                                     (cudaStream_t)stream);
}

}  // extern "C"
