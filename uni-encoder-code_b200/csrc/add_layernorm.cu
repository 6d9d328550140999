// add_layernorm.cu -- y = LayerNorm(x + residual) * gamma + beta over the last dimension, fp32.
//
// SURVEY.md 8f.3: the two post-norm steps of every encoder layer, `norm1(src + dropout1(attn))` and
// `norm2(src + dropout3(ffn))` (msdeformattn.py:126-142).  The reference (torch eager) runs an add
// kernel and a LayerNorm kernel: 5 passes over [rows, 256] where 3 suffice.  HBM-bound: one warp per
// row, the row lives in registers between the statistics and the normalisation.
//   mean = sum(v) / C;  var = sum((v - mean)^2) / C  (two-pass, in registers);  rstd = rsqrt(var + eps)
//   y = (v - mean) * rstd * gamma + beta             (torch.nn.functional.layer_norm semantics)
// Mixed precision (torch.autocast, DESIGN.md 11.2): the same kernels with a bf16 / fp16 residual widened on load, and
// y also written rounded to the 16-bit type for the next GEMMs; the fp32 arithmetic is the fp32 kernels'.
#include <cuda_runtime.h>
#include <cstdint>

#include "msda_common.cuh"

namespace msda {

namespace {

// V = float4 chunks per lane: C = 128 * V columns.  R: element type of `res` -- float, or (the mixed-precision
// entries) bf16 / fp16, widened on load; then `y16` (may be null) also receives y rounded to R.  The fp32
// arithmetic does not depend on R.
template <int V, typename R>
__device__ __forceinline__ void add_layernorm_rows(const float4 *__restrict__ x, const R *__restrict__ res,
                                                   const float4 *__restrict__ gamma, const float4 *__restrict__ beta,
                                                   float4 *__restrict__ y, R *__restrict__ y16, long long rows,
                                                   float eps) {
    constexpr int C4 = 32 * V;                      // float4 per row
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    float4 g[V], b[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
        g[i] = gamma[i * 32 + lane];
        b[i] = beta[i * 32 + lane];
    }
    for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows; row += warps) {
        float4 v[V];
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            const float4 a = ldg_stream_f4(x + row * C4 + i * 32 + lane);
            v[i] = a;
            if (res != nullptr) {
                const float4 r = ldg_stream_v4<R>(res + (row * C4 + i * 32 + lane) * 4);
                v[i].x += r.x; v[i].y += r.y; v[i].z += r.z; v[i].w += r.w;
            }
            sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(kFullMask, sum, o);
        const float mean = sum * (1.f / (4 * C4));
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
            sq += (dx * dx + dy * dy) + (dz * dz + dw * dw);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(kFullMask, sq, o);
        const float rstd = rsqrtf(sq * (1.f / (4 * C4)) + eps);
#pragma unroll
        for (int i = 0; i < V; ++i) {
            float4 o;
            o.x = (v[i].x - mean) * rstd * g[i].x + b[i].x;
            o.y = (v[i].y - mean) * rstd * g[i].y + b[i].y;
            o.z = (v[i].z - mean) * rstd * g[i].z + b[i].z;
            o.w = (v[i].w - mean) * rstd * g[i].w + b[i].w;
            y[row * C4 + i * 32 + lane] = o;
            if constexpr (is16<R>) {
                if (y16 != nullptr) st_round4(y16 + (row * C4 + i * 32 + lane) * 4, o);
            }
        }
    }
}

template <int V>
__global__ void __launch_bounds__(256)
add_layernorm_kernel(const float4 *__restrict__ x, const float4 *__restrict__ res,
                     const float4 *__restrict__ gamma, const float4 *__restrict__ beta,
                     float4 *__restrict__ y, long long rows, float eps) {
    add_layernorm_rows<V, float>(x, reinterpret_cast<const float *>(res), gamma, beta, y, nullptr, rows, eps);
}

// mixed precision: fp32 x, 16-bit residual, fp32 y and its 16-bit copy y16
template <int V, typename R>
__global__ void __launch_bounds__(256)
add_layernorm_mixed_kernel(const float4 *__restrict__ x, const R *__restrict__ res,
                           const float4 *__restrict__ gamma, const float4 *__restrict__ beta,
                           float4 *__restrict__ y, R *__restrict__ y16, long long rows, float eps) {
    add_layernorm_rows<V, R>(x, res, gamma, beta, y, y16, rows, eps);
}

template <int V>
cudaError_t launch(const float *x, const float *res, const float *gamma, const float *beta, float *y,
                   long long rows, float eps, cudaStream_t stream) {
    long long blocks = (rows + 7) / 8;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    add_layernorm_kernel<V><<<(unsigned)blocks, 256, 0, stream>>>(
        reinterpret_cast<const float4 *>(x), reinterpret_cast<const float4 *>(res),
        reinterpret_cast<const float4 *>(gamma), reinterpret_cast<const float4 *>(beta),
        reinterpret_cast<float4 *>(y), rows, eps);
    note_launch();
    return cudaGetLastError();
}

template <int V, typename R>
cudaError_t launch_mixed(const float *x, const R *res, const float *gamma, const float *beta, float *y, R *y16,
                         long long rows, float eps, cudaStream_t stream) {
    long long blocks = (rows + 7) / 8;
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    add_layernorm_mixed_kernel<V, R><<<(unsigned)blocks, 256, 0, stream>>>(
        reinterpret_cast<const float4 *>(x), res, reinterpret_cast<const float4 *>(gamma),
        reinterpret_cast<const float4 *>(beta), reinterpret_cast<float4 *>(y), y16, rows, eps);
    note_launch();
    return cudaGetLastError();
}

}  // namespace

// cols in {128, 256, 384, 512}; 16-byte aligned pointers; residual may be null (plain LayerNorm)
cudaError_t launch_add_layernorm(const float *x, const float *res, const float *gamma, const float *beta, float *y,
                                 long long rows, int cols, float eps, cudaStream_t stream, bool *handled) {
    *handled = true;
    const uintptr_t bits = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(res) |
                           reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta) |
                           reinterpret_cast<uintptr_t>(y);
    if (bits % 16 != 0) {
        *handled = false;
        return cudaSuccess;
    }
    switch (cols) {
        case 128: return launch<1>(x, res, gamma, beta, y, rows, eps, stream);
        case 256: return launch<2>(x, res, gamma, beta, y, rows, eps, stream);
        case 384: return launch<3>(x, res, gamma, beta, y, rows, eps, stream);
        case 512: return launch<4>(x, res, gamma, beta, y, rows, eps, stream);
        default: *handled = false; return cudaSuccess;
    }
}

// mixed precision: 16-bit residual and y16 (may be null) 8-byte aligned, the fp32 tensors 16-byte aligned
template <typename R>
cudaError_t launch_add_layernorm_mixed(const float *x, const R *res, const float *gamma, const float *beta, float *y,
                                       R *y16, long long rows, int cols, float eps, cudaStream_t stream,
                                       bool *handled) {
    *handled = true;
    const uintptr_t bits = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(gamma) |
                           reinterpret_cast<uintptr_t>(beta) | reinterpret_cast<uintptr_t>(y);
    const uintptr_t bits16 = reinterpret_cast<uintptr_t>(res) | reinterpret_cast<uintptr_t>(y16);
    if (bits % 16 != 0 || bits16 % 8 != 0) {
        *handled = false;
        return cudaSuccess;
    }
    switch (cols) {
        case 128: return launch_mixed<1, R>(x, res, gamma, beta, y, y16, rows, eps, stream);
        case 256: return launch_mixed<2, R>(x, res, gamma, beta, y, y16, rows, eps, stream);
        case 384: return launch_mixed<3, R>(x, res, gamma, beta, y, y16, rows, eps, stream);
        case 512: return launch_mixed<4, R>(x, res, gamma, beta, y, y16, rows, eps, stream);
        default: *handled = false; return cudaSuccess;
    }
}
template cudaError_t launch_add_layernorm_mixed<__nv_bfloat16>(const float *, const __nv_bfloat16 *, const float *,
                                                               const float *, float *, __nv_bfloat16 *, long long,
                                                               int, float, cudaStream_t, bool *);
template cudaError_t launch_add_layernorm_mixed<__half>(const float *, const __half *, const float *, const float *,
                                                        float *, __half *, long long, int, float, cudaStream_t, bool *);

}  // namespace msda

// ---------------------------------------------------------------------------
// Backward of y = LayerNorm(x + residual) * gamma + beta (training): with v = x + residual,
// xhat = (v - mean) * rstd and g = grad_y * gamma,
//     grad_v = rstd * (g - mean_c(g) - xhat * mean_c(g * xhat))         (= grad_x = grad_residual)
//     grad_gamma = sum_rows grad_y * xhat,   grad_beta = sum_rows grad_y
// v, mean and rstd are recomputed from x and residual (one extra read of residual instead of a stored copy
// of v).  One warp per row as in the forward; each warp keeps its partial grad_gamma / grad_beta in
// registers over all its rows and adds them to the zero-filled outputs once at the end -- or, in the
// deterministic entry, stores the CTA's partials in a workspace that a second launch sums in CTA order (the
// grid is a fixed function of rows and SM count).
// ---------------------------------------------------------------------------
namespace msda {
namespace {

template <int V>
__global__ void __launch_bounds__(256)
add_layernorm_bwd_kernel(const float4 *__restrict__ gy, const float4 *__restrict__ x, const float4 *__restrict__ res,
                         const float4 *__restrict__ gamma, float4 *__restrict__ gv, float *__restrict__ ggamma,
                         float *__restrict__ gbeta, long long rows, float eps, float *__restrict__ partials) {
    constexpr int C4 = 32 * V;
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    float4 gm[V], dg[V], db[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
        gm[i] = gamma[i * 32 + lane];
        dg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        db[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows; row += warps) {
        float4 v[V], g[V];
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            v[i] = ldg_stream_f4(x + row * C4 + i * 32 + lane);
            if (res != nullptr) {
                const float4 r = ldg_stream_f4(res + row * C4 + i * 32 + lane);
                v[i].x += r.x; v[i].y += r.y; v[i].z += r.z; v[i].w += r.w;
            }
            g[i] = ldg_stream_f4(gy + row * C4 + i * 32 + lane);
            sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(kFullMask, sum, o);
        const float mean = sum * (1.f / (4 * C4));
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
            sq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(kFullMask, sq, o);
        const float rstd = rsqrtf(sq * (1.f / (4 * C4)) + eps);
        float s1 = 0.f, s2 = 0.f;                     // sum_c g,  sum_c g * xhat   (g = grad_y * gamma)
#pragma unroll
        for (int i = 0; i < V; ++i) {
            v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd;      // xhat
            dg[i].x += g[i].x * v[i].x; dg[i].y += g[i].y * v[i].y; dg[i].z += g[i].z * v[i].z; dg[i].w += g[i].w * v[i].w;
            db[i].x += g[i].x; db[i].y += g[i].y; db[i].z += g[i].z; db[i].w += g[i].w;
            g[i].x *= gm[i].x; g[i].y *= gm[i].y; g[i].z *= gm[i].z; g[i].w *= gm[i].w;
            s1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
            s2 += (g[i].x * v[i].x + g[i].y * v[i].y) + (g[i].z * v[i].z + g[i].w * v[i].w);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_xor_sync(kFullMask, s1, o);
            s2 += __shfl_xor_sync(kFullMask, s2, o);
        }
        s1 *= (1.f / (4 * C4));
        s2 *= (1.f / (4 * C4));
#pragma unroll
        for (int i = 0; i < V; ++i) {
            float4 o;
            o.x = rstd * (g[i].x - s1 - v[i].x * s2);
            o.y = rstd * (g[i].y - s1 - v[i].y * s2);
            o.z = rstd * (g[i].z - s1 - v[i].z * s2);
            o.w = rstd * (g[i].w - s1 - v[i].w * s2);
            gv[row * C4 + i * 32 + lane] = o;
        }
    }
    // per-CTA reduction of the 8 warps' partials in shared memory, then one reduction per column per CTA
    __shared__ float part[2][8][128 * V];
    const int w = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < V; ++i) {
        float *pg = &part[0][w][(i * 32 + lane) * 4], *pb = &part[1][w][(i * 32 + lane) * 4];
        pg[0] = dg[i].x; pg[1] = dg[i].y; pg[2] = dg[i].z; pg[3] = dg[i].w;
        pb[0] = db[i].x; pb[1] = db[i].y; pb[2] = db[i].z; pb[3] = db[i].w;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 128 * V; c += 256) {
        float a = 0.f, b = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            a += part[0][k][c];
            b += part[1][k][c];
        }
        if (partials != nullptr) {        // [2][gridDim.x][C]
            partials[(long long)blockIdx.x * (128 * V) + c] = a;
            partials[((long long)gridDim.x + blockIdx.x) * (128 * V) + c] = b;
        } else {
            asm volatile("red.global.add.f32 [%0], %1;" ::"l"(ggamma + c), "f"(a) : "memory");
            asm volatile("red.global.add.f32 [%0], %1;" ::"l"(gbeta + c), "f"(b) : "memory");
        }
    }
}

// Mixed precision (16-bit R = bf16 / fp16): fp32 x, 16-bit residual (widened on load); the incoming gradient is
// g = gy + widen(gy16), one fp32 add; G says which of the two is given (kGradY, kGradY16 or both), so that the loads
// carry no branch and are issued together as in the fp32 kernel; gv16 receives grad_v rounded to R.  After the
// loads, the fp32 kernel's arithmetic, reduction structure and epilogue, line for line.
enum { kGradY = 1, kGradY16 = 2 };
template <int V, typename R, int G>
__global__ void __launch_bounds__(256, 4)
add_layernorm_mixed_bwd_kernel(const float4 *__restrict__ gy, const R *__restrict__ gy16, const float4 *__restrict__ x,
                               const R *__restrict__ res, const float4 *__restrict__ gamma, float4 *__restrict__ gv,
                               R *__restrict__ gv16, float *__restrict__ ggamma, float *__restrict__ gbeta,
                               long long rows, float eps, float *__restrict__ partials) {
    constexpr int C4 = 32 * V;
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    float4 gm[V], dg[V], db[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
        gm[i] = gamma[i * 32 + lane];
        dg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        db[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows; row += warps) {
        float4 v[V], g[V];
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            v[i] = ldg_stream_f4(x + row * C4 + i * 32 + lane);
            {
                const float4 r = ldg_stream_v4<R>(res + (row * C4 + i * 32 + lane) * 4);
                v[i].x += r.x; v[i].y += r.y; v[i].z += r.z; v[i].w += r.w;
            }
            if constexpr (G == kGradY) {
                g[i] = ldg_stream_f4(gy + row * C4 + i * 32 + lane);
            } else {
                g[i] = ldg_stream_v4<R>(gy16 + (row * C4 + i * 32 + lane) * 4);
                if constexpr ((G & kGradY) != 0) {
                    const float4 a = ldg_stream_f4(gy + row * C4 + i * 32 + lane);
                    g[i].x = a.x + g[i].x; g[i].y = a.y + g[i].y; g[i].z = a.z + g[i].z; g[i].w = a.w + g[i].w;
                }
            }
            sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(kFullMask, sum, o);
        const float mean = sum * (1.f / (4 * C4));
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
            sq += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(kFullMask, sq, o);
        const float rstd = rsqrtf(sq * (1.f / (4 * C4)) + eps);
        float s1 = 0.f, s2 = 0.f;                     // sum_c g,  sum_c g * xhat   (g = grad_y * gamma)
#pragma unroll
        for (int i = 0; i < V; ++i) {
            v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd;      // xhat
            dg[i].x += g[i].x * v[i].x; dg[i].y += g[i].y * v[i].y; dg[i].z += g[i].z * v[i].z; dg[i].w += g[i].w * v[i].w;
            db[i].x += g[i].x; db[i].y += g[i].y; db[i].z += g[i].z; db[i].w += g[i].w;
            g[i].x *= gm[i].x; g[i].y *= gm[i].y; g[i].z *= gm[i].z; g[i].w *= gm[i].w;
            s1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
            s2 += (g[i].x * v[i].x + g[i].y * v[i].y) + (g[i].z * v[i].z + g[i].w * v[i].w);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_xor_sync(kFullMask, s1, o);
            s2 += __shfl_xor_sync(kFullMask, s2, o);
        }
        s1 *= (1.f / (4 * C4));
        s2 *= (1.f / (4 * C4));
#pragma unroll
        for (int i = 0; i < V; ++i) {
            float4 o;
            o.x = rstd * (g[i].x - s1 - v[i].x * s2);
            o.y = rstd * (g[i].y - s1 - v[i].y * s2);
            o.z = rstd * (g[i].z - s1 - v[i].z * s2);
            o.w = rstd * (g[i].w - s1 - v[i].w * s2);
            gv[row * C4 + i * 32 + lane] = o;
            st_round4(gv16 + (row * C4 + i * 32 + lane) * 4, o);
        }
    }
    // per-CTA reduction of the 8 warps' partials in shared memory, then one reduction per column per CTA
    __shared__ float part[2][8][128 * V];
    const int w = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < V; ++i) {
        float *pg = &part[0][w][(i * 32 + lane) * 4], *pb = &part[1][w][(i * 32 + lane) * 4];
        pg[0] = dg[i].x; pg[1] = dg[i].y; pg[2] = dg[i].z; pg[3] = dg[i].w;
        pb[0] = db[i].x; pb[1] = db[i].y; pb[2] = db[i].z; pb[3] = db[i].w;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 128 * V; c += 256) {
        float a = 0.f, b = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            a += part[0][k][c];
            b += part[1][k][c];
        }
        if (partials != nullptr) {        // [2][gridDim.x][C]
            partials[(long long)blockIdx.x * (128 * V) + c] = a;
            partials[((long long)gridDim.x + blockIdx.x) * (128 * V) + c] = b;
        } else {
            asm volatile("red.global.add.f32 [%0], %1;" ::"l"(ggamma + c), "f"(a) : "memory");
            asm volatile("red.global.add.f32 [%0], %1;" ::"l"(gbeta + c), "f"(b) : "memory");
        }
    }
}

// deterministic entry: grad_gamma / grad_beta = the CTAs' partials summed in CTA order
__global__ void __launch_bounds__(256)
add_layernorm_bwd_sum_kernel(const float *__restrict__ partials, float *__restrict__ ggamma, float *__restrict__ gbeta,
                             int ctas, int cols) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * cols) return;
    const int which = i / cols, c = i - which * cols;
    const float *p = partials + (long long)which * ctas * cols + c;
    float s = 0.f;
    for (int k = 0; k < ctas; ++k) s += p[(long long)k * cols];
    (which == 0 ? ggamma : gbeta)[c] = s;
}

long long bwd_ctas(long long rows) {
    long long blocks = (rows + 7) / 8;
    const long long cap = (long long)sm_count() * 4;      // few CTAs: each ends with 2 x C reductions
    return blocks > cap ? cap : blocks;
}

// R = float: the fp32 kernel (gy16 / gv16 unused); 16-bit R: the mixed-precision kernel
template <int V, typename R>
cudaError_t launch_bwd(const float *gy, const R *gy16, const float *x, const R *res, const float *gamma, float *gv,
                       R *gv16, float *ggamma, float *gbeta, long long rows, float eps, cudaStream_t stream,
                       float *partials) {
    if (partials == nullptr) {
        cudaError_t e = cudaMemsetAsync(ggamma, 0, 128 * V * sizeof(float), stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(gbeta, 0, 128 * V * sizeof(float), stream);
        if (e != cudaSuccess) return e;
    }
    const long long blocks = bwd_ctas(rows);
    if constexpr (is16<R>) {
        const int which = (gy != nullptr ? kGradY : 0) | (gy16 != nullptr ? kGradY16 : 0);
        const auto kern = which == kGradY ? add_layernorm_mixed_bwd_kernel<V, R, kGradY>
                          : which == kGradY16 ? add_layernorm_mixed_bwd_kernel<V, R, kGradY16>
                                              : add_layernorm_mixed_bwd_kernel<V, R, kGradY | kGradY16>;
        kern<<<(unsigned)blocks, 256, 0, stream>>>(
            reinterpret_cast<const float4 *>(gy), gy16, reinterpret_cast<const float4 *>(x), res,
            reinterpret_cast<const float4 *>(gamma), reinterpret_cast<float4 *>(gv), gv16, ggamma, gbeta, rows, eps,
            partials);
    } else {
        add_layernorm_bwd_kernel<V><<<(unsigned)blocks, 256, 0, stream>>>(
            reinterpret_cast<const float4 *>(gy), reinterpret_cast<const float4 *>(x),
            reinterpret_cast<const float4 *>(res), reinterpret_cast<const float4 *>(gamma),
            reinterpret_cast<float4 *>(gv), ggamma, gbeta, rows, eps, partials);
    }
    note_launch();
    if (partials == nullptr) return cudaGetLastError();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    add_layernorm_bwd_sum_kernel<<<(2 * 128 * V + 255) / 256, 256, 0, stream>>>(partials, ggamma, gbeta, (int)blocks,
                                                                              128 * V);
    note_launch();
    return cudaGetLastError();
}

}  // namespace

// floats of the deterministic entry's workspace: grad_gamma and grad_beta partials of every CTA
long long add_layernorm_bwd_partials(long long rows, int cols) { return 2 * bwd_ctas(rows) * cols; }

cudaError_t launch_add_layernorm_bwd(const float *gy, const float *x, const float *res, const float *gamma, float *gv,
                                     float *ggamma, float *gbeta, long long rows, int cols, float eps,
                                     cudaStream_t stream, bool *handled, float *partials) {
    *handled = true;
    const uintptr_t bits = reinterpret_cast<uintptr_t>(gy) | reinterpret_cast<uintptr_t>(x) |
                           reinterpret_cast<uintptr_t>(res) | reinterpret_cast<uintptr_t>(gamma) |
                           reinterpret_cast<uintptr_t>(gv);
    if (bits % 16 != 0) {
        *handled = false;
        return cudaSuccess;
    }
    switch (cols) {
        case 128: return launch_bwd<1, float>(gy, nullptr, x, res, gamma, gv, nullptr, ggamma, gbeta, rows, eps, stream,
                                              partials);
        case 256: return launch_bwd<2, float>(gy, nullptr, x, res, gamma, gv, nullptr, ggamma, gbeta, rows, eps, stream,
                                              partials);
        default: *handled = false; return cudaSuccess;
    }
}

// mixed precision: gy (fp32) and / or gy16 (16-bit), fp32 x, 16-bit residual; gv fp32 and gv16 16-bit.  The 16-bit
// tensors 8-byte aligned, the fp32 ones 16-byte aligned
template <typename R>
cudaError_t launch_add_layernorm_mixed_bwd(const float *gy, const R *gy16, const float *x, const R *res,
                                           const float *gamma, float *gv, R *gv16, float *ggamma, float *gbeta,
                                           long long rows, int cols, float eps, cudaStream_t stream, bool *handled,
                                           float *partials) {
    *handled = true;
    const uintptr_t bits = reinterpret_cast<uintptr_t>(gy) | reinterpret_cast<uintptr_t>(x) |
                           reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(gv);
    const uintptr_t bits16 = reinterpret_cast<uintptr_t>(gy16) | reinterpret_cast<uintptr_t>(res) |
                             reinterpret_cast<uintptr_t>(gv16);
    if (bits % 16 != 0 || bits16 % 8 != 0) {
        *handled = false;
        return cudaSuccess;
    }
    switch (cols) {
        case 128: return launch_bwd<1, R>(gy, gy16, x, res, gamma, gv, gv16, ggamma, gbeta, rows, eps, stream, partials);
        case 256: return launch_bwd<2, R>(gy, gy16, x, res, gamma, gv, gv16, ggamma, gbeta, rows, eps, stream, partials);
        default: *handled = false; return cudaSuccess;
    }
}
#define MSDA_LN_MIXED_BWD(R)                                                                                       \
    template cudaError_t launch_add_layernorm_mixed_bwd<R>(const float *, const R *, const float *, const R *,     \
                                                           const float *, float *, R *, float *, float *, long long, \
                                                           int, float, cudaStream_t, bool *, float *);
MSDA_LN_MIXED_BWD(__nv_bfloat16)
MSDA_LN_MIXED_BWD(__half)
#undef MSDA_LN_MIXED_BWD

}  // namespace msda
