// msda_generic.cu -- shape-generic MSDA kernels (any channels-per-head, level and
// point count; fp32, fp64, and bf16 / fp16 value rows with fp32 locations, weights and sums)
// and the integer known-answer kernel.
//
// The 32-channel fp32 kernels in msda_fwd.cu / msda_bwd.cu are the hot path; these
// cover the rest of the reference op's domain (AT_DISPATCH_FLOATING_TYPES at
// ms_deform_attn_cuda.cu:69,139 instantiates float and double, and the col2im
// launcher accepts any channel count, ms_deform_im2col_cuda.cuh:980-1323).
//
// One warp per (image, query, head) row; lanes stride over channels, so a corner
// row is read as one coalesced segment.  grad_sampling_loc / grad_attn_weight are
// warp-shuffle sums (no shared memory, no barrier); grad_value uses scalar atomics, or, in the
// deterministic mode (RECORDS, msda_det.cu), is left alone while lanes 0-3 write the four corner records
// of every point.
#include "msda_common.cuh"

namespace msda {

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    return v;
}

// V: element type of value / out (grad_output); T: of the locations, weights and every sum (float for 16-bit V)
template <typename V, typename T>
__global__ void __launch_bounds__(256)
msda_fwd_generic_kernel(const V *__restrict__ value, const int64_t *__restrict__ shapes,
                        const int64_t *__restrict__ lstart, const T *__restrict__ loc,
                        const T *__restrict__ attw, const Dims d, V *__restrict__ out) {
    __shared__ LevelTable lt;
    fill_level_table(lt, shapes, lstart, d.L, d.P, d.S, d.Lq, 8, 1, 8, 0);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    const long long rows = (long long)d.N * d.Lq * d.M;
    const long long pix = (long long)d.M * d.D;
    for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows;
         row += warps) {
        const int m = (int)(row % d.M);
        const long long n = row / ((long long)d.Lq * d.M);
        const V *vb = value + n * (long long)d.S * pix + (long long)m * d.D;
        for (int c0 = 0; c0 < d.D; c0 += 32) {
            const int c = c0 + lane;
            T acc = 0;
            for (int l = 0; l < d.L; ++l) {
                const int H = lt.H[l], W = lt.W[l];
                const V *lb = vb + (long long)lt.start[l] * pix;
                for (int p = 0; p < d.P; ++p) {
                    const long long s = (row * d.L + l) * d.P + p;
                    const Geom<T> g = decompose(loc[2 * s], loc[2 * s + 1], H, W);
                    if (g.valid && c < d.D) {
                        const T hh = 1 - g.lh, hw = 1 - g.lw;
                        const V *p0 = lb + ((long long)g.h_low * W + g.w_low) * pix + c;
#ifdef MSDA_CHECK_BOUNDS
                        {
                            const V *lo = value + n * (long long)d.S * pix, *hi = lo + (long long)d.S * pix;
                            assert(!(g.cmask & 1) || (p0 >= lo && p0 < hi));
                            assert(!(g.cmask & 8) || (p0 + (long long)W * pix + pix >= lo && p0 + (long long)W * pix + pix < hi));
                        }
#endif
                        const T v1 = (g.cmask & 1) ? widen<T>(p0[0]) : (T)0;
                        const T v2 = (g.cmask & 2) ? widen<T>(p0[pix]) : (T)0;
                        const T v3 = (g.cmask & 4) ? widen<T>(p0[(long long)W * pix]) : (T)0;
                        const T v4 = (g.cmask & 8) ? widen<T>(p0[(long long)W * pix + pix]) : (T)0;
                        const T val = (hh * hw) * v1 + (hh * g.lw) * v2 + (g.lh * hw) * v3 + (g.lh * g.lw) * v4;
                        acc += val * attw[s];
                    }
                }
            }
            if (c < d.D) out[row * d.D + c] = narrow<V>(acc);
        }
    }
}

// 16-bit V: grad_value is the fp32 accumulation buffer (T = float)
template <typename V, typename T, bool RECORDS>
__global__ void __launch_bounds__(256)
msda_bwd_generic_kernel(const V *__restrict__ grad_out, const V *__restrict__ value,
                        const int64_t *__restrict__ shapes, const int64_t *__restrict__ lstart,
                        const T *__restrict__ loc, const T *__restrict__ attw, const Dims d,
                        T *__restrict__ grad_value, T *__restrict__ grad_loc,
                        T *__restrict__ grad_attw, const DetRecords det) {
    __shared__ LevelTable lt;
    fill_level_table(lt, shapes, lstart, d.L, d.P, d.S, d.Lq, 8, 1, 8, 0);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    const long long rows = (long long)d.N * d.Lq * d.M;
    const long long pix = (long long)d.M * d.D;
    for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows;
         row += warps) {
        const int m = (int)(row % d.M);
        const long long n = row / ((long long)d.Lq * d.M);
        const long long img = n * (long long)d.S * pix + (long long)m * d.D;
        for (int l = 0; l < d.L; ++l) {
            const int H = lt.H[l], W = lt.W[l];
            const long long lvl = img + (long long)lt.start[l] * pix;
            for (int p = 0; p < d.P; ++p) {
                const long long s = (row * d.L + l) * d.P + p;
                const Geom<T> g = decompose(loc[2 * s], loc[2 * s + 1], H, W);
                T gx = 0, gy = 0, ga = 0;
                if (RECORDS && lane < 4) {          // lane k: corner k (also of an invalid point: cmask == 0)
                    const int k = lane;
                    const bool live = g.cmask >> k & 1;
                    const T hh = 1 - g.lh, hw = 1 - g.lw;
                    const T cw = k == 0 ? hh * hw : k == 1 ? hh * g.lw : k == 2 ? g.lh * hw : g.lh * g.lw;
                    // element offset / D = destination row (n*S + pixel)*M + m
                    const long long o = lvl + (((long long)g.h_low + (k >> 1)) * W + g.w_low + (k & 1)) * pix;
                    const uint32_t slot = (uint32_t)(4 * s + k);
                    det.key[slot] = live ? (uint32_t)(o / d.D) : det.sentinel;
                    det.slot_id[slot] = slot;
                    static_cast<T *>(det.w)[slot] = live ? cw * attw[s] : (T)0;
                }
                if (g.valid) {
                    const T a = attw[s];
                    const T hh = 1 - g.lh, hw = 1 - g.lw;
                    const T cw[4] = {hh * hw, hh * g.lw, g.lh * hw, g.lh * g.lw};
                    const T dh[4] = {-hw, -g.lw, hw, g.lw};     // d val / d h per corner
                    const T dw[4] = {-hh, hh, -g.lh, g.lh};     // d val / d w per corner
                    const long long p0 = lvl + ((long long)g.h_low * W + g.w_low) * pix;
                    const long long co[4] = {0, pix, (long long)W * pix, (long long)W * pix + pix};
                    for (int c = lane; c < d.D; c += 32) {
                        const T tg = widen<T>(grad_out[row * d.D + c]);
                        const T tgv = tg * a;
                        T val = 0, sh = 0, sw = 0;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if (g.cmask >> k & 1) {
                                const long long o = p0 + co[k] + c;
#ifdef MSDA_CHECK_BOUNDS
                                assert(o >= n * (long long)d.S * pix && o < (n + 1) * (long long)d.S * pix);
#endif
                                const T v = widen<T>(value[o]);
                                sh += dh[k] * v;
                                sw += dw[k] * v;
                                val += cw[k] * v;
                                if (!RECORDS) atomicAdd(grad_value + o, cw[k] * tgv);
                            }
                        }
                        ga += tg * val;
                        gx += (T)W * sw * tgv;
                        gy += (T)H * sh * tgv;
                    }
                }
                gx = warp_sum(gx);
                gy = warp_sum(gy);
                ga = warp_sum(ga);
                if (lane == 0) {
                    grad_loc[2 * s] = gx;
                    grad_loc[2 * s + 1] = gy;
                    grad_attw[s] = ga;
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256)
msda_debug_indices_kernel(const int64_t *__restrict__ shapes, const int64_t *__restrict__ lstart,
                          const float *__restrict__ loc, const Dims d, int32_t *__restrict__ idx,
                          int64_t *__restrict__ off) {
    __shared__ LevelTable lt;
    fill_level_table(lt, shapes, lstart, d.L, d.P, d.S, d.Lq, 8, 1, 8, 0);
    __syncthreads();
    const long long total = (long long)d.N * d.Lq * d.M * d.L * d.P;
    const long long pix = (long long)d.M * d.D;
    for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < total;
         s += (long long)gridDim.x * blockDim.x) {
        const int l = (int)((s / d.P) % d.L);
        const long long row = s / ((long long)d.L * d.P);
        const int m = (int)(row % d.M);
        const long long n = row / ((long long)d.Lq * d.M);
        const int H = lt.H[l], W = lt.W[l];
        const Geom<float> g = decompose(loc[2 * s], loc[2 * s + 1], H, W);
        idx[4 * s + 0] = g.valid;
        idx[4 * s + 1] = g.h_low;
        idx[4 * s + 2] = g.w_low;
        idx[4 * s + 3] = g.cmask;
        const long long p0 = n * (long long)d.S * pix + (long long)m * d.D +
                             ((long long)lt.start[l] + (long long)g.h_low * W + g.w_low) * pix;
        off[4 * s + 0] = (g.cmask & 1) ? p0 : -1;
        off[4 * s + 1] = (g.cmask & 2) ? p0 + pix : -1;
        off[4 * s + 2] = (g.cmask & 4) ? p0 + (long long)W * pix : -1;
        off[4 * s + 3] = (g.cmask & 8) ? p0 + (long long)W * pix + pix : -1;
    }
}

static unsigned grid_for(long long work_items, int per_block) {
    long long b = (work_items + per_block - 1) / per_block;
    const long long cap = (long long)sm_count() * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (unsigned)b;
}

template <typename V, typename T>
cudaError_t launch_fwd_generic(const V *value, const int64_t *shapes, const int64_t *lstart,
                               const T *loc, const T *attw, const Dims &d, V *out,
                               cudaStream_t stream) {
    const long long rows = (long long)d.N * d.Lq * d.M;
    msda_fwd_generic_kernel<V, T><<<grid_for(rows, 8), 256, 0, stream>>>(value, shapes, lstart, loc,
                                                                       attw, d, out);
    note_launch();
    return cudaGetLastError();
}

template <typename V, typename T>
cudaError_t launch_bwd_generic(const V *grad_out, const V *value, const int64_t *shapes,
                               const int64_t *lstart, const T *loc, const T *attw, const Dims &d,
                               T *gv, T *gl, T *gw, cudaStream_t stream) {
    const long long rows = (long long)d.N * d.Lq * d.M;
    msda_bwd_generic_kernel<V, T, false><<<grid_for(rows, 8), 256, 0, stream>>>(
        grad_out, value, shapes, lstart, loc, attw, d, gv, gl, gw, DetRecords{nullptr, nullptr, nullptr, 0});
    note_launch();
    return cudaGetLastError();
}

// deterministic mode: grad_loc / grad_attw as above, the corner records into `det` (grad_value untouched)
template <typename V, typename T>
cudaError_t launch_bwd_generic_records(const V *grad_out, const V *value, const int64_t *shapes,
                                       const int64_t *lstart, const T *loc, const T *attw, const Dims &d,
                                       T *gl, T *gw, const DetRecords &det, cudaStream_t stream) {
    const long long rows = (long long)d.N * d.Lq * d.M;
    msda_bwd_generic_kernel<V, T, true><<<grid_for(rows, 8), 256, 0, stream>>>(grad_out, value, shapes, lstart,
                                                                             loc, attw, d, nullptr, gl, gw, det);
    note_launch();
    return cudaGetLastError();
}

cudaError_t launch_debug_indices(const int64_t *shapes, const int64_t *lstart, const float *loc,
                                 const Dims &d, int32_t *idx, int64_t *off, cudaStream_t stream) {
    const long long total = (long long)d.N * d.Lq * d.M * d.L * d.P;
    msda_debug_indices_kernel<<<grid_for(total, 256), 256, 0, stream>>>(shapes, lstart, loc, d, idx, off);
    note_launch();
    return cudaGetLastError();
}

// 16-bit grad_value: the fp32 accumulation buffer -> V, eight elements per thread with 128-bit accesses
// (two float4 loads, one 16-byte store); `vec` = 0 when a pointer is not 16-byte aligned (scalar loop)
template <typename V>
__global__ void __launch_bounds__(256)
msda_narrow_kernel(const float *__restrict__ acc, V *__restrict__ out, long long n, int vec) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n8 = vec ? n / 8 : 0;
    for (long long i = i0; i < n8; i += stride) {
        const float4 a = ldg_stream_f4(reinterpret_cast<const float4 *>(acc) + 2 * i);
        const float4 b = ldg_stream_f4(reinterpret_cast<const float4 *>(acc) + 2 * i + 1);
        const float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint4 u;
        uint32_t w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const V lo = narrow<V>(f[2 * k]), hi = narrow<V>(f[2 * k + 1]);
            unsigned short l16, h16;
            memcpy(&l16, &lo, 2);
            memcpy(&h16, &hi, 2);
            w[k] = (uint32_t)l16 | ((uint32_t)h16 << 16);
        }
        u = make_uint4(w[0], w[1], w[2], w[3]);
        asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
                     ::"l"(reinterpret_cast<uint4 *>(out) + i), "r"(u.x), "r"(u.y), "r"(u.z), "r"(u.w) : "memory");
    }
    for (long long i = n8 * 8 + i0; i < n; i += stride) out[i] = narrow<V>(acc[i]);
}

template <typename V>
cudaError_t launch_narrow(const float *acc, V *out, long long n, cudaStream_t stream) {
    const int vec = ((reinterpret_cast<uintptr_t>(acc) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0;
    msda_narrow_kernel<V><<<grid_for((n + 7) / 8, 256), 256, 0, stream>>>(acc, out, n, vec);
    note_launch();
    return cudaGetLastError();
}

#define MSDA_GENERIC(V, T)                                                                                          \
    template cudaError_t launch_fwd_generic<V, T>(const V *, const int64_t *, const int64_t *, const T *, const T *, \
                                                  const Dims &, V *, cudaStream_t);                                 \
    template cudaError_t launch_bwd_generic<V, T>(const V *, const V *, const int64_t *, const int64_t *, const T *, \
                                                  const T *, const Dims &, T *, T *, T *, cudaStream_t);            \
    template cudaError_t launch_bwd_generic_records<V, T>(const V *, const V *, const int64_t *, const int64_t *,   \
                                                          const T *, const T *, const Dims &, T *, T *,            \
                                                          const DetRecords &, cudaStream_t);
MSDA_GENERIC(float, float)
MSDA_GENERIC(double, double)
MSDA_GENERIC(__nv_bfloat16, float)
MSDA_GENERIC(__half, float)
#undef MSDA_GENERIC
template cudaError_t launch_narrow<__nv_bfloat16>(const float *, __nv_bfloat16 *, long long, cudaStream_t);
template cudaError_t launch_narrow<__half>(const float *, __half *, long long, cudaStream_t);

}  // namespace msda
